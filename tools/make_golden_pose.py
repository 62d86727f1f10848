#!/usr/bin/env python
"""Generate tests/golden/g6_pose_matches.npz: the matches of the LIVE, UNMODIFIED reference (modules.xfeat.XFeat.match_xfeat,
top_k=2048, on the CPU) for the four synthetic pose samples of tests/test_gpu_geometry.py::plane_pose_samples.

The reference is imported through oracle/build_ref.py, so its sources must be where that module looks for them
(XFEAT_REFERENCE_ROOT):

    python tools/make_golden_pose.py
"""
import os
import sys

os.environ["CUDA_VISIBLE_DEVICES"] = ""            # the reference picks CUDA when it sees one (modules/xfeat.py:25)
import numpy as np  # noqa: E402
import torch  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from accelerated_features_b200 import weights as _w  # noqa: E402
from oracle import build_ref  # noqa: E402
from oracle import xfeat_oracle as orc  # noqa: E402
from tests.conftest import load_golden  # noqa: E402
from tests.test_gpu_geometry import plane_pose_samples  # noqa: E402

if build_ref.build_ref() is None:
    raise SystemExit(f"reference sources not found at {build_ref.REF_ROOT} (set XFEAT_REFERENCE_ROOT)")
sd = {k: torch.as_tensor(v) for k, v in _w.load_state_dict(_w.DEFAULT_WEIGHTS).items()}
ref_xf = build_ref.import_reference()(weights=sd, top_k=2048)
g = load_golden("inputs_assets_vga.npz")
samples = plane_pose_samples(g["ref"], g["tgt"])
state = orc.load_state()
out = {}
with torch.inference_mode():
    for i, s in enumerate(samples):
        m0, m1 = ref_xf.match_xfeat(s["image0"], s["image1"], top_k=2048)
        out[f"mkpts0_{i}"], out[f"mkpts1_{i}"] = np.asarray(m0, np.float32), np.asarray(m1, np.float32)
        p0, p1 = orc.match_xfeat(state, s["image0"], s["image1"], 2048)
        a = {tuple(r) for r in np.concatenate([m0, m1], 1).tolist()}
        b = {tuple(r) for r in np.concatenate([np.asarray(p0), np.asarray(p1)], 1).tolist()}
        print(f"sample {i}: {s['image0'].shape[:2]}, {len(m0)} reference matches, {len(a ^ b)} differ from the oracle port")
path = os.path.join(ROOT, "tests", "golden", "g6_pose_matches.npz")
np.savez_compressed(path, **out)
print(f"{path}: {os.path.getsize(path) / 1e6:.2f} MB")
