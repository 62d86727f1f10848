#!/usr/bin/env python
"""A/B of the block1 tail (block1.2 -> block1.3 + skip1) at 128 x VGA, the batch xfeat_net runs for bench.py's sparse config.

    python tools/block1_ab.py [--iters 60] [--prof-iters 10] [--out DIR]

1. CUDA events around each xfeat_net launch, fused and two-kernel tail alternating in one process (the rest of the network is
   the same in both): median ms per launch of each variant and their difference.
2. A separate torch.profiler run of --prof-iters launches per variant: the block1 kernels' names and mean us per launch, and
   the fused kernel's achieved GB/s against its HBM floor (read a2 and xn, write s4a).
Prints one JSON line; with --out, also writes it and the profiler kernel table there."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch  # noqa: E402

from accelerated_features_b200 import XFeat, _lib  # noqa: E402

B, H, W = 128, 480, 640
# bytes the fused kernel must move: a2 split (32 B per half-res px), xn (4 B per px), s4a split (128 B per quarter-res px)
FLOOR_BYTES = B * (H // 2) * (W // 2) * 32 + B * H * W * 4 + B * (H // 4) * (W // 4) * 128
BLOCK1_KERNELS = ("block1_tc_kernel", "conv_tc_halo_kernel<8, 8>", "conv_tc_kernel<3, 8, 32>")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=60)
    ap.add_argument("--prof-iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    xf = XFeat()
    lib = xf._lib
    g = torch.Generator().manual_seed(0)
    xn = torch.randn(B, H, W, generator=g).cuda()
    feats = torch.empty(B, H // 8, W // 8, 64, device="cuda")
    heat = torch.empty(B, H, W, device="cuda")
    rel = torch.empty(B, H // 8, W // 8, device="cuda")
    nbytes = lib.xfeat_net_workspace_bytes(B, H, W)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def net():
        _lib.check(lib.xfeat_net(xf._ctx, xn.data_ptr(), B, H, W, feats.data_ptr(), heat.data_ptr(), rel.data_ptr(), None,
                                 ws.data_ptr(), ws.numel(), stream), "xfeat_net")

    variants = {"fused": 1, "unfused": 0}
    outs = {}
    for name, on in variants.items():            # warm-up, and the outputs of both paths for an equality check
        lib.xfeat_set_block1_fused(on)
        assert lib.xfeat_get_block1_fused() == on, "XFEAT_BLOCK1_UNFUSED is set"
        for _ in range(3):
            net()
        torch.cuda.synchronize()
        outs[name] = (feats.clone(), heat.clone(), rel.clone())
    same = all(torch.equal(x, y) for x, y in zip(outs["fused"], outs["unfused"]))

    times = {k: [] for k in variants}
    for _ in range(a.iters):
        for name, on in variants.items():
            lib.xfeat_set_block1_fused(on)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            net()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1))

    kern = {}
    rows = []
    from torch.profiler import ProfilerActivity, profile
    for name, on in variants.items():
        lib.xfeat_set_block1_fused(on)
        net()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.prof_iters):
                net()
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if ev.device_type.name != "CUDA" or ev.count == 0:
                continue
            us = ev.device_time_total / a.prof_iters
            rows.append((name, ev.key, ev.count // a.prof_iters, us))
            if any(k in ev.key for k in BLOCK1_KERNELS):
                kern.setdefault(name, {})[ev.key] = round(us, 1)
    lib.xfeat_set_block1_fused(1)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    med = {k: statistics.median(v) for k, v in times.items()}
    fused_us = sum(kern.get("fused", {}).values())
    res = {
        "gpu": smi, "B": B, "H": H, "W": W, "iters": a.iters, "prof_iters": a.prof_iters,
        "net_ms_median": {k: round(v, 4) for k, v in med.items()},
        "net_ms_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()},
        "net_saving_us": round((med["unfused"] - med["fused"]) * 1000, 1),
        "block1_kernels_us": kern,
        "block1_us": {k: round(sum(v.values()), 1) for k, v in kern.items()},
        "fused_floor_MB": round(FLOOR_BYTES / 1e6, 1),
        "fused_GBps_vs_floor": round(FLOOR_BYTES / (fused_us * 1e-6) / 1e9, 1) if fused_us else None,
        "outputs_equal": same,
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "block1_ab.json"), "w") as f:
            f.write(line + "\n")
        with open(os.path.join(a.out, "block1_ab_kernels.md"), "w") as f:
            f.write(f"# xfeat_net kernels at {B} x {H}x{W}, torch.profiler, mean per launch over {a.prof_iters} launches ({smi})\n\n")
            f.write("| variant | kernel | calls | us |\n|---|---|---|---|\n")
            for name, key, cnt, us in sorted(rows, key=lambda r: (r[0], -r[3])):
                f.write(f"| {name} | `{key[:90]}` | {cnt} | {us:.1f} |\n")


if __name__ == "__main__":
    main()
