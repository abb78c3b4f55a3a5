#!/usr/bin/env python
"""Headline benchmark: tokens/sec of the sharded-DP training step, Llama-3-8B config, bf16, seq 4096, synthetic tokens.

  python bench.py --gpus N --steps K --warmup W            our sm_100a path (torchrun launches N ranks for N>1)
  python bench.py --impl reference --gpus N ...            reference arm: the UNMODIFIED reference recipe (baseline/_ref install) on
                                                           the host cores, CPU/gloo, bounded sample (falls back to the numpy
                                                           restatement in oracle/ when the install is absent)
  python bench.py --steps K --dump-outputs DIR             also write what the last timed step computed to DIR/<name>.npy, to
                                                           compare two builds output for output (inputs and init are seeded)

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for what each field means.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# one hardware launch queue per stream (default 8 queues shared by every stream of the process): kernels that wait for a peer GPU
# (the in-kernel barriers of the NVLink collectives, NCCL's) must never sit in front of unrelated work in a shared queue
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

LLAMA3_8B = {"vocab_size": 128256, "hidden_size": 4096, "intermediate_size": 14336, "num_hidden_layers": 32, "num_attention_heads": 32,
             "num_key_value_heads": 8, "max_position_embeddings": 8192, "rms_norm_eps": 1e-5, "rope_theta": 500000.0,
             "rope_scaling": {"rope_type": "llama3", "factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                              "original_max_position_embeddings": 8192}}
SEQ = 4096
METRIC = "tokens/sec Llama-3-8B bf16 SFT seq4096"


def flops_per_token(cfg, S):
    """The reference's own formula (nemo_automodel/components/utils/flops_utils.py:51-78): fwd+bwd, causal attention 1/2."""
    L, h = cfg["num_hidden_layers"], cfg["hidden_size"]
    kv, heads, ffn, V = cfg["num_key_value_heads"], cfg["num_attention_heads"], cfg["intermediate_size"], cfg["vocab_size"]
    return L * h * h * (12 + 12 * kv / heads + 18 * ffn / h + 6 * S / h + 6 * V / (L * h))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


DUMP_SAMPLE = 16384     # elements kept per parameter tensor: the 291 tensors of Llama-3-8B come to 16 MB of float32


def dump_outputs(out_dir, loss, grad_norm, params):
    """What one training step hands its caller, as float32 .npy files in out_dir: loss.npy, grad_norm.npy and one file per updated
    parameter (HF name).  A parameter of more than DUMP_SAMPLE elements is sampled at fixed, distinct indices seeded by its name, so that two
    builds run with the same arguments can be compared file by file.  Compare with a tolerance: the attention backward adds dQ tiles
    in whatever order its CTAs finish, and at these shapes dQ differs in its last bits from launch to launch (50 of 50 launches on a
    B200 at 1000 W), so two runs of one build agree to rounding, not bit for bit."""
    import zlib
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([float(loss)], dtype=np.float32))
    np.save(os.path.join(out_dir, "grad_norm.npy"), np.array([float(grad_norm)], dtype=np.float32))
    for name, p in params.items():
        flat = p.reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(flat.numel(), DUMP_SAMPLE, replace=False))
            flat = flat.index_select(0, torch.from_numpy(idx).to(flat.device))
        np.save(os.path.join(out_dir, name + ".npy"), flat.float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def _host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count()


def run_cpu_reference(steps, warmup, budget_s=150.0):
    """The reference's own CPU implementation of the path, timed on the host cores on a bounded sample of the workload.

    kind "reference" (baseline/_ref present): the UNMODIFIED `TrainFinetuneRecipeForNextTokenPrediction` over CPU/gloo, world size 1, in a
    subprocess (baseline/run_ref_cpu.py): Llama-3-8B layer dimensions, ONE decoder layer, vocab 2048, seq 512, b=1, fp32, full optimizer
    steps, every host thread torch uses.  kind "port" (no install): the numpy restatement oracle/llama_step.py on the same sample.
    Either way tokens/s is converted to the full workload by the reference's FLOPs formula (components/utils/flops_utils.py:51-78):
        tokens/s(8B, S=4096) = achieved CPU FLOP/s / 4.825e10."""
    f_full = flops_per_token(LLAMA3_8B, SEQ)
    runner = os.path.join(ROOT, "baseline", "run_ref_cpu.py")
    if os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "nemo_automodel")):
        try:
            r = subprocess.run([sys.executable, runner, str(steps), str(warmup), str(budget_s)], capture_output=True, text=True,
                               timeout=budget_s + 300, cwd=ROOT)
            lines = [l for l in r.stdout.splitlines() if l.startswith("REF_CPU_RESULT ")]
            if r.returncode == 0 and lines:
                d = json.loads(lines[-1][len("REF_CPU_RESULT "):])
                cpu_flops = d["flops_per_step"] / d["mean_step_s"]
                return {"value": cpu_flops / f_full, "unit": "tokens/s", "cores": d["cores"], "threads": d["threads"], "kind": "reference",
                        "sample": f"unmodified reference recipe ({d['model_class']} + torch.optim.{d['optimizer_class']} + MaskedCrossEntropy, CPU/gloo, fp32) on 1 decoder "
                                  f"layer of Llama-3-8B dims, vocab {d['vocab']}, seq {d['seq']}, b=1: {d['mean_step_s'] * 1e3:.0f} ms/step over {d['steps_timed']} steps "
                                  f"= {cpu_flops / 1e9:.1f} GFLOP/s; scaled to 8B/seq4096 by the reference FLOPs formula",
                        "ms_per_sample_step": d["mean_step_s"] * 1e3, "steps_timed": d["steps_timed"], "cpu_gflops": cpu_flops / 1e9}
            sys.stderr.write("reference CPU run failed, falling back to the numpy port:\n" + r.stderr[-2000:] + "\n")
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"reference CPU run failed ({e}); falling back to the numpy port\n")
    import numpy as np
    from oracle import llama_step as O
    from oracle.portable_init import llama_param_shapes
    S = 512
    cfg = dict(LLAMA3_8B, num_hidden_layers=1, vocab_size=2048, max_position_embeddings=S)
    rng = np.random.default_rng(0)
    params = {k: (rng.standard_normal(shp, dtype=np.float32) * 0.02 if len(shp) > 1 else np.ones(shp, np.float32))
              for k, shp in llama_param_shapes(cfg).items()}
    opt = O.AdamW(lr=1e-5, prec="fp32")
    ids = rng.integers(0, cfg["vocab_size"], (1, S))
    mb = [{"input_ids": ids, "labels": O.mock_labels(ids)}]
    f_tok = flops_per_token(cfg, S)
    times = []
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.train_step(params, opt, cfg, mb, prec="fp32", max_grad_norm=1.0, timing=True)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s and times:
            break
    mean = sum(times) / len(times)
    cpu_flops = f_tok * S / mean
    return {"value": cpu_flops / f_full, "unit": "tokens/s", "cores": _host_cores(), "kind": "port",
            "sample": f"oracle (numpy fp32) full train step on 1 decoder layer of Llama-3-8B dims, vocab 2048, seq {S}, b=1: "
                      f"{mean * 1e3:.0f} ms/step over {len(times)} steps = {cpu_flops / 1e9:.1f} GFLOP/s; scaled to 8B/seq4096 by the reference FLOPs formula",
            "ms_per_sample_step": mean * 1e3, "steps_timed": len(times), "cpu_gflops": cpu_flops / 1e9}


# ------------------------------------------------------------------------------------------------ our arm (GPU)
def _claim_stdout():
    """The driver parses ONE JSON line from stdout; libraries (NCCL prints its version banner there) must not interleave.
    fd 1 is pointed at stderr for the whole run and the JSON line is written to the saved descriptor at the end."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit(saved_fd, line):
    os.write(saved_fd, (json.dumps(line) + "\n").encode())


def main():
    # watchdog: a wedged collective must not hold a multi-GPU box until the driver's own limit.  faulthandler's timer thread works even
    # while the main thread is blocked inside a CUDA / NCCL call: it writes every thread's Python stack to stderr (which rank, which
    # call) and then terminates the process, so the peers' NCCL / in-kernel barriers time out instead of spinning silently.
    import faulthandler
    wd = int(os.environ.get("B200_BENCH_WATCHDOG_S", "900"))
    sys.stderr.write(f"[bench rank {os.environ.get('RANK', '0')}] watchdog armed: {wd} s\n")
    faulthandler.dump_traceback_later(wd, exit=True)
    saved_stdout = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--layers", type=int, default=None, help="debug only: fewer layers (result is then NOT the headline metric)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-api", default="facade", choices=["engine", "facade"],
                    help="public call timed by the e2e leg: the reference-facing facade (default: B200CausalLM -> B200MaskedCrossEntropy -> backward "
                         "-> clip -> B200FusedAdamW.step, the call sequence of the reference recipe) or ShardedLlamaEngine.train_step")
    ap.add_argument("--no-parity", action="store_true", help="N > 1 only: skip the correctness block that precedes the timed region")
    ap.add_argument("--profile", action="store_true", help="for ncu runs only: 1 warm-up step, no e2e leg, no CPU baseline (numbers printed are NOT bench values)")
    ap.add_argument("--adam-mode", type=int, default=1, help="1 = torch.optim.AdamW bf16 op sequence (reference default optimizer), 0 = fp32 math")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's loss, grad norm and (sampled) updated parameters to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; the reference arm has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        cb = run_cpu_reference(args.steps, args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "tokens/s", "n_gpus": args.gpus, "steps": cb["steps_timed"],
                "warmup": args.warmup, "ms_per_step": cb["ms_per_sample_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": "llama3_8b_sft_seq4096_b1_per_gpu", "note": "CPU reference arm runs a bounded sample, see cpu_baseline.sample"},
                "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        _emit(saved_stdout, line)
        return 0

    import torch
    import torch.distributed as dist
    from automodel_b200 import ops
    from automodel_b200.engine import ShardedLlamaEngine

    assert torch.cuda.is_available(), "bench.py needs a GPU (the product path has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ops.device_check()
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    cfg = dict(LLAMA3_8B)
    if args.layers:
        cfg["num_hidden_layers"] = args.layers
    eng = ShardedLlamaEngine(cfg, dev, process_group=pg, max_tokens=SEQ, lr=1e-5, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1,
                             adam_mode=args.adam_mode, max_positions=SEQ)
    # ---- N > 1: correctness of the multi-GPU path, in the driver-visible record (the GPU test box has one GPU).  (1) the production
    # collectives on one full-size decoder-layer unit of THIS engine vs fp32 NCCL references; (2) 10 optimizer steps of a small Llama
    # sharded over the N ranks vs one rank accumulating the same sequences.  Out of tolerance = the run fails (rc 3), no number printed.
    parity = None
    if world > 1 and not args.no_parity and not args.profile:
        from automodel_b200 import diagnostics
        col = diagnostics.check_collectives(eng, unit_index=1)
        par = diagnostics.check_sharded_step_parity(pg, dev, steps=10)
        ok = (col["ag_bit_exact"] and col["rs_norm_sq_rel_err"] < 1e-5 and par["ranks_agree"] and par["max_abs_dloss"] <= 1e-3
              and par["max_rel_dgnorm"] <= 2e-2 and (col["reduce_dtype"] != "float32" or col["rs_err_over_fp32_accumulate_bound"] <= 1.25))
        parity = dict(par, collectives=col, ok=bool(ok), tolerance={"max_abs_dloss": 1e-3, "max_rel_dgnorm": 2e-2,
                                                          "rs": "|got - fp32 sum| <= 1.25 x (2^-8 |sum| + 2^-21 sum|addends|): fp32 accumulation in any order + one rounding (measured 0.996; the NVSwitch reducer 1.99, a bf16 ring >> 10)"})
        if not ok:
            sys.stderr.write(f"[bench rank {rank}] N={world} parity block FAILED: {json.dumps(parity)}\n")
            if rank == 0:
                _emit(saved_stdout, {"metric": METRIC, "n_gpus": world, "parity": parity, "error": "multi-GPU parity block out of tolerance; no throughput reported"})
            dist.destroy_process_group()
            return 3
    eng.init_random_(seed=1234)

    # synthetic tokens, MockIterableDataset semantics (components/datasets/llm/mock_iterable_dataset.py:41-59); every rank draws its own
    g = torch.Generator().manual_seed(1234 + rank)
    nbatch = 4
    host = []
    for _ in range(nbatch):
        ids = torch.randint(0, cfg["vocab_size"], (1, SEQ), generator=g, dtype=torch.int64).pin_memory()
        lab = torch.full((1, SEQ), -100, dtype=torch.int64); lab[:, :-1] = ids[:, 1:]
        host.append({"input_ids": ids, "labels": lab.pin_memory()})
    n_label = (SEQ - 1) * world
    tokens_per_step = SEQ * world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------ leg 1: device-resident inputs (`value`)
    staged = [eng.stage(host[0]["input_ids"], host[0]["labels"])]
    n_warm = 1 if args.profile else max(args.warmup, 3)
    for _ in range(n_warm):
        eng.train_step(None, 1.0, num_label_tokens=n_label, staged=staged)
    gemm_events = []

    @contextlib.contextmanager
    def gemm_timer(kind, M, N, K):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        yield
        e1.record()
        gemm_events.append((e0, e1, 2.0 * M * N * K))

    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    if args.profile:
        torch.cuda.profiler.start()     # ncu --profile-from-start off: capture exactly the timed region
    l0 = ops.LAUNCHES
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    h0 = time.perf_counter()
    for _ in range(args.steps):
        loss, gn = eng.train_step(None, 1.0, num_label_tokens=n_label, staged=staged)
    host_issue_ms = (time.perf_counter() - h0) * 1e3 / args.steps   # CPU time to enqueue one step (back-pressured by the launch queue)
    eng.sync_params()   # the last step's optimizer sweep / all-gather run on side streams: they belong to the timed region
    t1.record()
    barrier()
    if args.profile:
        torch.cuda.profiler.stop()
    launches = ops.LAUNCHES - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, gn, eng.state_dict())
    # pure host cost of enqueueing one step: start from an idle GPU so the launch queue never back-pressures
    torch.cuda.synchronize()
    h0 = time.perf_counter()
    eng.train_step(None, 1.0, num_label_tokens=n_label, staged=staged)
    host_only_ms = (time.perf_counter() - h0) * 1e3
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms = t0.elapsed_time(t1)
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_step = float(tms.item()) / args.steps
    value = tokens_per_step / (ms_step / 1e3)
    # ---- roofline pass: the same step with stream overlap off (weight-gradient GEMMs and the optimizer sweep back to back on the compute
    # stream), so the CUDA events around each GEMM launch bracket that kernel alone; in the timed region above GEMMs of two streams
    # time-slice the SMs and an event pair would also count the other stream's CTAs.
    roof_steps = 0 if args.profile else min(args.steps, 4)
    if roof_steps:
        eng.set_stream_overlap(False)
        eng.train_step(None, 1.0, num_label_tokens=n_label, staged=staged)
        barrier()
        ops.GEMM_TIMER = gemm_timer
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(roof_steps):
            eng.train_step(None, 1.0, num_label_tokens=n_label, staged=staged)
        eng.sync_params()
        r1.record()
        barrier()
        ops.GEMM_TIMER = None
        roof_ms_step = r0.elapsed_time(r1) / roof_steps
        eng.set_stream_overlap(True)
    else:
        roof_ms_step = float("nan")
    gemm_ms = sum(a.elapsed_time(b) for a, b, _ in gemm_events)
    gemm_flops = sum(f for _, _, f in gemm_events)
    n_gemm = len(gemm_events)
    final_loss, final_gnorm = float(loss), float(gn)

    # ------------------------------------------------ leg 2: end to end through the public API (`e2e`): pinned host inputs copied
    # every step inside the timed region + device->host read of the step's loss and grad norm
    if args.e2e_api == "facade":
        from automodel_b200.recipe import B200CausalLM, B200MaskedCrossEntropy, B200FusedAdamW
        fac = B200CausalLM(cfg, eng)
        fac_loss = B200MaskedCrossEntropy()
        fac_opt = B200FusedAdamW(fac.parameters(), lr=1e-5, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1)

        def e2e_step(mb):
            # the recipe's sequence (train_ft.py:1436-1473, 1536-1558): model(**batch) without labels, loss_fn(logits, labels,
            # num_label_tokens), (loss * dp).backward(), clip utility, optimizer.step(), zero_grad()
            fac.set_requires_gradient_sync(True)
            out = fac(input_ids=mb["input_ids"])
            loss = fac_loss(logits=out.logits, labels=mb["labels"], num_label_tokens=n_label)
            (loss * world).backward()
            gn_ = fac.b200_clip_grad_norm(1.0)
            fac_opt.step()
            fac_opt.zero_grad()
            tot = loss.detach().clone()
            if world > 1:
                dist.all_reduce(tot)
            return tot, gn_
    else:
        def e2e_step(mb):
            return eng.train_step([mb], 1.0)

    eng.h2d_bytes = 0
    for i in range(0 if args.profile else 2):
        l, g_ = e2e_step(host[i % nbatch])
        float(l)
    barrier()
    eng.h2d_bytes = 0
    w0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_steps = 1 if args.profile else args.steps
    e0.record()
    for i in range(e2e_steps):
        l, g_ = e2e_step(host[i % nbatch])
        lv, gv = float(l), float(g_)         # D2H read of the step result (host sync, as the reference recipe does every step)
    eng.sync_params()
    e1.record()
    barrier()
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_ms_step = float(e2e_ms.item()) / e2e_steps
    h2d = eng.h2d_bytes // e2e_steps
    e2e = {"value": tokens_per_step / (e2e_ms_step / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 8,
           "ms_per_step": e2e_ms_step, "host_threads": 1, "api": "ShardedLlamaEngine.train_step" if args.e2e_api == "engine" else "B200CausalLM facade (recipe call sequence)"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks = measured_peaks()
    f_tok = flops_per_token(cfg, SEQ)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")   # from one ncu capture of the same command (tools/summarize_ncu.py traffic)
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath))["traffic_bytes_per_launch"]
        except Exception:
            traffic = None
    achieved_tf = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
    roofline = {"bound": "tensor", "kernel": "pair::gemm_pair_kernel (CTA-pair tcgen05 GEMM: every nn.Linear fwd / dgrad / wgrad of the step)", "achieved": achieved_tf, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                "frac": (achieved_tf / peaks["tflops_sustained"]) if achieved_tf else None, "traffic": traffic,
                "traffic_unit": "DRAM bytes per GEMM launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, average over the step's GEMM launches)",
                "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_timed": n_gemm, "gemm_share_of_step": gemm_ms / (roof_ms_step * roof_steps) if roof_steps else None,
                "measured_in": f"{roof_steps} extra steps with stream overlap off (GEMMs serialised on one stream; {roof_ms_step:.2f} ms/step incl. event overhead)",
                "algorithmic_flops_per_step": gemm_flops / roof_steps if roof_steps else None,
                "step_model_tflops_per_gpu": f_tok * SEQ / (ms_step / 1e3) / 1e12,
                "step_frac_of_peak": f_tok * SEQ / (ms_step / 1e3) / 1e12 / peaks["tflops_sustained"]}
    line = {"metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": n_warm,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "llama3_8b_sft_seq4096_b1_per_gpu", "layers": cfg["num_hidden_layers"], "global_batch": world, "seq_len": SEQ,
                       "parallelism": f"sharded-dp{world}", "collectives": eng.comm_kind,
                       "grad_reduce": ("fp32 accumulate, one rounding" if eng.reduce_dtype == "float32" else "bf16") if world > 1 else "none", "grad_accum": 1, "optimizer": "AdamW(bf16 states)" if args.adam_mode == 1 else "AdamW(fp32 math)",
                       "clip_grad_norm": 1.0, "l2": "working set (16 GB params + 16 GB grads + activations) >> 126 MB L2; no flush needed",
                       "tokens_per_step": tokens_per_step},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "final_loss": final_loss, "final_grad_norm": final_gnorm,
            "flops_per_token": f_tok, "host_issue_ms_per_step": host_issue_ms, "host_enqueue_ms_idle_gpu": host_only_ms}
    if parity is not None:
        line["parity"] = parity
    if args.profile:
        line["profile_mode"] = True
    if not args.no_cpu_baseline and not args.profile and world == 1:
        line["cpu_baseline"] = run_cpu_reference(steps=3, warmup=1, budget_s=40.0)
    _emit(saved_stdout, line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
