#!/usr/bin/env python3
"""Per-conv-layer TFLOP/s of one network pass (tcs_score_profiled)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vae-diffusion-toy-crystals_b200"))
import bench  # noqa: E402
from toycrystals_b200.models import sde_score_model as shim  # noqa: E402

torch.manual_seed(1)
m = shim.CondUNetTiny(4, 4, 96, 128, 8, 8, precision="bf16").cuda().eval()
n = int(sys.argv[1]) if len(sys.argv) > 1 else 128   # samples per pass (images = 2n); bench.py uses 128
k = bench.profile_kernels(m, shim.VPSDE(0.1, 30.0), torch.device("cuda", 0), n)
print(round(k["conv_tflops"], 1), round(k["conv_ms"], 3), round(k["conv_share"], 3),
      json.dumps(k["per_layer"]))
