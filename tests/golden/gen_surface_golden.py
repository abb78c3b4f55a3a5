#!/usr/bin/env python
"""Golden data for tests/test_recipe_surface.py from the UNMODIFIED reference: the field names of its FSDP2Config
(components/distributed/config.py) and the losses its MaskedCrossEntropy (components/loss/masked_ce.py) returns on seeded logits /
labels in fp32 and bf16.  Test infrastructure; needs the reference checkout (B200_REFERENCE_PATH).  Writes
tests/golden/surface_golden.npz (read by tests/test_recipe_surface.py on any host)."""
import dataclasses
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _ref_env  # noqa: F401,E402
import numpy as np  # noqa: E402
import torch  # noqa: E402
from nemo_automodel.components.distributed.config import FSDP2Config  # noqa: E402
from nemo_automodel.components.loss.masked_ce import MaskedCrossEntropy  # noqa: E402

out = {"fsdp2_config_fields": np.array(sorted(f.name for f in dataclasses.fields(FSDP2Config)))}
g = torch.Generator().manual_seed(0)
logits = torch.randn(2, 48, 96, generator=g) * 3
labels = torch.randint(0, 96, (2, 48), generator=g)
labels[torch.rand(2, 48, generator=g) < 0.25] = -100
n = int((labels != -100).sum())
out["ce/logits"], out["ce/labels"], out["ce/num_label_tokens"] = logits.numpy(), labels.numpy(), np.array(n)
ce = MaskedCrossEntropy()
for dt in ("float32", "bfloat16"):
    x = logits.to(getattr(torch, dt))
    out[f"ce/loss_{dt}"] = np.array(float(ce(x, labels, num_label_tokens=n)), dtype=np.float64)
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "surface_golden.npz"), **out)
print({k: (v.shape, v.dtype) for k, v in out.items()})
