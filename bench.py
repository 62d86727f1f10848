#!/usr/bin/env python
"""bench.py -- image-pairs/sec (extract + match) on synthetic batches (BASELINE.json configs 2 and 3).

    python bench.py --gpus N --steps K --warmup W                  # this repo's CUDA path, config 2 (one process per GPU)
    python bench.py --config star --steps K --warmup W             # config 3: 64 x 1280x960 semi-dense match_xfeat_star
    python bench.py --impl reference --steps K --warmup W          # the UNMODIFIED reference on the host CPU (oracle/_ref)
    python bench.py --steps K --warmup W --dump-outputs DIR        # also write the last timed step's results as DIR/*.npy

A "step" is one pass of the hot path over one batch of 64 synthetic image pairs per GPU:
  sparse: detectAndCompute on both image sets (backbone, NMS/top-k 4096, bicubic descriptors) + per-pair MNN match;
  star  : detectAndComputeDense (dual scale) on both sets + batch_match + refine_matches.
`value`   : pairs/s with the inputs already resident in HBM (CUDA events around K steps, max over ranks).
`e2e`     : pairs/s through the PUBLIC API (XFeat.match_xfeat_stream / XFeat.match_xfeat_star) with HOST (pinned) inputs: H2D of
            both image sets and D2H of the results inside the timed region.
`roofline`: the dominant kernel: algorithmic FLOPs / its CUDA-event time inside the timed steps, against MEASURED_PEAKS.json.
`cpu_baseline` / `--impl reference`: the reference's own modules/xfeat.py (byte-compiled into oracle/_ref by
            oracle/build_ref.py), CUDA hidden, all host threads, same workload shape; falls back to the oracle PORT only if
            oracle/_ref is missing, and says so in `kind`.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOPK, BATCH = 4096, 64
CONFIGS = {
    "sparse": {"H": 480, "W": 640, "metric": "image-pairs/sec (extract+match) VGA batch=64",
               "workload": "batch=64 synthetic VGA (640x480) sparse match_xfeat top_k=4096", "cpu_pairs": 64},
    "star": {"H": 960, "W": 1280, "metric": "image-pairs/sec (semi-dense match_xfeat_star) 1280x960 batch=64",
             "workload": "batch=64 synthetic 1280x960 semi-dense match_xfeat_star top_k=4096", "cpu_pairs": 4},
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm_sorted = sorted(sm)   # median over the upper half = samples taken under load
        return {"sm_mhz": statistics.median(sm_sorted[len(sm_sorted) // 2:]), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference (oracle/_ref), CUDA hidden.  Runs in its own process (CUDA_VISIBLE_DEVICES='' must be
# exported before torch is imported: the reference picks CUDA when it sees a device, modules/xfeat.py:25).
# ---------------------------------------------------------------------------------------------------------------------
def cpu_arm(config: str, n_pairs: int, repeats: int, warmup: int, seed: int = 0, budget_s: float = 270.0):
    import torch
    assert not torch.cuda.is_available(), "the CPU arm must not see a GPU"
    cfg = CONFIGS[config]
    H, W = cfg["H"], cfg["W"]
    want = max(1, (os.cpu_count() or 2) // 2)      # physical cores; torchrun exports OMP_NUM_THREADS=1, undo that here
    if torch.get_num_threads() < want:
        torch.set_num_threads(want)
    from accelerated_features_b200 import weights as _w
    sd = {k: torch.as_tensor(v) for k, v in _w.load_state_dict(_w.DEFAULT_WEIGHTS).items()}
    from oracle import build_ref
    kind = "reference"
    if build_ref.available():
        xf = build_ref.import_reference()(weights=sd, top_k=TOPK)
        detect, match, star = xf.detectAndCompute, xf.match, xf.match_xfeat_star
    else:   # labelled fallback: the oracle's restatement of the same algorithm
        kind = "port"
        from oracle import xfeat_oracle as orc
        state = orc.load_state()
        detect = lambda x, top_k: orc.detect_and_compute(state, x, top_k)          # noqa: E731
        match = lambda a, b, min_cossim: orc.mnn_match(a, b, min_cossim)          # noqa: E731
        star = lambda a, b, top_k: orc.match_xfeat_star(state, a, b, top_k)       # noqa: E731
    g = torch.Generator().manual_seed(seed)
    x1 = torch.randn(n_pairs, 3, H, W, generator=g)
    x2 = torch.randn(n_pairs, 3, H, W, generator=g)

    def step():
        with torch.inference_mode():
            if config == "star":
                return sum(len(m) for m in star(x1, x2, top_k=TOPK)) if n_pairs > 1 else len(star(x1, x2, top_k=TOPK)[0])
            o1 = detect(x1, top_k=TOPK)            # BASELINE.md section 3: 2 x detectAndCompute(B) + B x match(-1)
            o2 = detect(x2, top_k=TOPK)
            n = 0
            for a, b in zip(o1, o2):
                i0, _ = match(a["descriptors"], b["descriptors"], min_cossim=-1)
                n += len(i0)
            return n

    # honour (warmup, repeats) as long as the whole run stays inside `budget_s`; the first step is timed to project it
    t0 = time.perf_counter()
    step()
    t_first = time.perf_counter() - t0
    fit = max(2, int(budget_s / max(t_first, 1e-3)))
    if warmup + repeats > fit:
        warmup = max(1, min(warmup, fit // 5))
        repeats = max(1, fit - warmup)
    for _ in range(max(0, warmup - 1)):                # (the timed first step was the first warm-up step)
        step()
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    return {"pairs_per_s": n_pairs / statistics.median(times), "seconds": sum(times), "threads": torch.get_num_threads(),
            "kind": kind, "n_pairs": n_pairs, "repeats": repeats, "warmup": max(1, warmup), "torch": torch.__version__}


def cpu_arm_subprocess(config: str, n_pairs: int, repeats: int, warmup: int):
    env = dict(os.environ)
    env["CUDA_VISIBLE_DEVICES"] = ""
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-arm-worker", config, str(n_pairs), str(repeats), str(warmup)],
                       capture_output=True, text=True, env=env, timeout=1500)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("cpu arm failed: " + r.stderr[-2000:])


def cpu_sample_text(c, config):
    cfg = CONFIGS[config]
    what = "modules.xfeat.XFeat (unmodified reference, oracle/_ref)" if c["kind"] == "reference" else "oracle port (oracle/_ref missing)"
    call = "match_xfeat_star" if config == "star" else "2 x detectAndCompute + B x match(-1)"
    return (f"{c['repeats']} x {c['n_pairs']} {cfg['W']}x{cfg['H']} pairs, {what}: {call}, torch {c['torch']} CPU, "
            f"{c['threads']} threads of {os.cpu_count()} logical cores, {c['seconds']:.1f} s")


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = CONFIGS[args.config]
    n_pairs = int(os.environ.get("XFEAT_BENCH_CPU_PAIRS", cfg["cpu_pairs"]))     # (tests shrink the batch; the line then says "scaled")
    # a step = the full batch (B = 64 VGA pairs: ~10 s on the host, 25 steps ~ 4 min).  --steps / --warmup are honoured unless
    # the projected run exceeds 270 s, in which case the worker shortens it and the line reports what was actually run.
    c = cpu_arm_subprocess(args.config, n_pairs, max(1, args.steps), max(1, args.warmup))
    v = c["pairs_per_s"]
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": c["repeats"],
        "warmup": c["warmup"], "steps_requested": args.steps, "warmup_requested": args.warmup, "ms_per_step": 1e3 * n_pairs / v,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic randn",
        "config": {"workload": cfg["workload"], "pairs_per_gpu": n_pairs, "top_k": TOPK,
                   "note": "CPU arm: one host, no GPU" + ("" if n_pairs == BATCH else f"; {n_pairs} pairs per step instead of {BATCH} (scaled)")},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": c["threads"], "kind": c["kind"], "sample": cpu_sample_text(c, args.config)},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def load_ncu(name):
    for rnd in ("r02", "r01"):
        try:
            with open(os.path.join(ROOT, "profiles", rnd, name)) as f:
                d = json.load(f)
            d["profile"] = f"profiles/{rnd}/{name}"
            return d
        except Exception:
            pass
    return None


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from accelerated_features_b200 import XFeat, _lib
    from accelerated_features_b200 import weights as _w

    cfg = CONFIGS[args.config]
    H, W = cfg["H"], cfg["W"]
    star = args.config == "star"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the XFeat hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    xf = XFeat(weights=_w.load_state_dict(_w.DEFAULT_WEIGHTS), top_k=TOPK, device=local)   # dict: no 'loading weights' print on stdout
    lib = _lib.load()

    # synthetic data: the reference's own style (minimal_example.py: torch.randn), one distinct shard per rank
    g = torch.Generator().manual_seed(1000 + rank)
    h1 = torch.randn(BATCH, 3, H, W, generator=g).pin_memory()
    h2 = torch.randn(BATCH, 3, H, W, generator=g).pin_memory()
    d1, d2 = h1.to(dev), h2.to(dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dom_events = []

    def step_resident(record=False):
        if star:
            if record:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            o1 = xf._dense_device(d1, TOPK, True)
            o2 = xf._dense_device(d2, TOPK, True)
            if record:
                e1.record()
                dom_events.append((e0, e1))
            K = o1["descriptors"].shape[1]
            idx0, idx1, cnt = xf._mnn_device(o1["descriptors"], None, K, K * 64, o2["descriptors"], None, K, K * 64, BATCH, -1)
            m, n_ref = xf._refine_device(o1, o2, idx0, idx1, cnt)
            return m, n_ref, cnt
        presplit = lib.xfeat_get_mnn_impl() in (1, 3)       # the same kernel sequence as XFeat._match_sparse_batch_device
        o = xf._detect_sparse_device([d1, d2], TOPK, xf.detection_threshold, want_split=presplit, want_desc=not presplit)
        k1, k2 = o["keypoints"][:BATCH], o["keypoints"][BATCH:]
        n1, n2 = o["n_valid"][:BATCH], o["n_valid"][BATCH:]
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if presplit:
            sp = o["desc_split"]
            idx0, idx1, cnt = xf._mnn_presplit_device(sp[:BATCH], n1, sp[BATCH:], n2, TOPK, sp.shape[1], BATCH, -1)
        else:
            f1, f2 = o["descriptors"][:BATCH], o["descriptors"][BATCH:]
            idx0, idx1, cnt = xf._mnn_device(f1, n1, TOPK, TOPK * 64, f2, n2, TOPK, TOPK * 64, BATCH, -1, abs_bound=1.0)
        if record:
            e1.record()
            dom_events.append((e0, e1))
        mk0, mk1, cnt = xf._gather_matches(k1, k2, idx0, idx1, cnt, BATCH, TOPK)
        return mk0, mk1, cnt, n1, n2

    warm = max(args.warmup, 3)
    for _ in range(warm):
        out = step_resident()
    barrier()
    launches0 = lib.xfeat_launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        out = step_resident(record=True)
    t1.record()
    barrier()
    launches = lib.xfeat_launch_count() - launches0
    ms_total = t0.elapsed_time(t1)
    dump = last_step_outputs(out, star) if args.dump_outputs and rank == 0 else None
    dom_ms = statistics.mean(a.elapsed_time(b) for a, b in dom_events)

    # ---- sustained self-check: the same resident step back to back for >= 2 s (clocks settle under the power cap) ----
    n_sus = max(args.steps, int(2200.0 / max(ms_total / args.steps, 1e-3)) + 1)
    u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u0.record()
    for _ in range(n_sus):
        step_resident()
    u1.record()
    barrier()
    sus_ms = u0.elapsed_time(u1)

    # ---- end to end through the public API: pinned host inputs -> H2D -> kernels -> D2H of the results ----
    def e2e_public(n, a, b):
        if star:
            tot = 0
            for _ in range(n):
                res = xf.match_xfeat_star(a, b, top_k=TOPK)               # H2D inside; list of (n,4) device tensors
                tot += sum(int(r.shape[0]) for r in res)                  # (the counts are the D2H read of the result)
            return tot
        tot = 0
        stamps = [time.perf_counter()]
        for res in xf.match_xfeat_stream(((a, b) for _ in range(n)), top_k=TOPK):
            tot += len(res)
            stamps.append(time.perf_counter())
        if os.environ.get("XFEAT_BENCH_DEBUG"):
            print("e2e batch intervals (ms):", [round(1e3 * (y - x), 2) for x, y in zip(stamps, stamps[1:])], file=sys.stderr)
        return tot

    e2e_public(max(3, args.warmup), h1, h2)
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    e2e_public(args.steps, h1, h2)
    s1.record()
    barrier()
    e2e_ms = s0.elapsed_time(s1)
    e2e_u8_ms, hu_bytes = None, 0
    if not star:
        # uint8 HWC images (what cv2 / camera callers hand to match_xfeat): 4x fewer bytes over PCIe, "/255" on the device
        hu1 = xf.pinned_like((BATCH, H, W, 3)); hu2 = xf.pinned_like((BATCH, H, W, 3))
        hu1.copy_((torch.rand(BATCH, H, W, 3, generator=g) * 255).to(torch.uint8))
        hu2.copy_((torch.rand(BATCH, H, W, 3, generator=g) * 255).to(torch.uint8))
        n1u, n2u = hu1.numpy(), hu2.numpy()                                # numpy views of pinned memory
        e2e_public(max(3, args.warmup), n1u, n2u)
        barrier()
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        e2e_public(args.steps, n1u, n2u)
        v1.record()
        barrier()
        e2e_u8_ms = v0.elapsed_time(v1)
        hu_bytes = int(2 * hu1.numel())
    # host link alone: the same fp32 upload with no kernels behind it
    tmp1, tmp2 = torch.empty_like(d1), torch.empty_like(d2)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(3):
        tmp1.copy_(h1, non_blocking=True)
        tmp2.copy_(h2, non_blocking=True)
    c1.record()
    barrier()
    h2d_gbs = 3 * 2 * h1.numel() * 4 / (c0.elapsed_time(c1) / 1e3) / 1e9
    clocks = sampler.stop() if sampler else None

    t = torch.tensor([ms_total, e2e_ms, dom_ms, e2e_u8_ms or 0.0, sus_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, dom_ms, e2e_u8_ms, sus_ms = t.tolist()

    if rank == 0:
        pk, pk_kind = peaks()
        pairs = BATCH * world * args.steps
        value = pairs / (ms_total / 1e3)
        peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        if star:
            # dominant stage: dual-scale dense extraction = 2 x xfeat_net at 0.6x and 1.3x (SURVEY 8d: 21.5 GFLOP per 1280x960 image)
            flops = 2.0 * BATCH * 21.50e9
            kname = ("dense extraction of both image sets (resize + xfeat_net at 768x576 and 1664x1248 + top-k/gather): tcgen05 split-fp16 "
                     "implicit-GEMM convolutions dominate")
            cfg_extra = {"mean_coarse_matches": float(out[2].float().mean()), "mean_refined": float(out[1].float().mean())}
            d2h = int(BATCH * 4)
            ncu, note = None, "algorithmic conv FLOPs (each MAC once) of both image sets / event time of the extraction stage"
        else:
            flops = 2.0 * 64.0 * float((out[3].double() * out[4].double()).sum())
            impl = lib.xfeat_get_mnn_impl()
            kname = (f"xfeat_mnn_match_presplit (impl {impl}): mnn_tc_persist_kernel, fused D1.D2^T (3-term split fp16) + row arg-max, both "
                     "directions, tcgen05; timed call also contains the finalize kernel")
            cfg_extra = {"mean_keypoints": [float(out[3].float().mean()), float(out[4].float().mean())],
                         "mean_matches_per_pair": float(out[2].float().mean())}
            d2h = int(2 * BATCH * TOPK * 2 * 4 + BATCH * 4)
            ncu = load_ncu("ncu_mnn.json")
            note = "achieved counts each MAC of ONE similarity matrix once (SURVEY 8d); both scan directions and precision passes are overhead"
        achieved = flops / (dom_ms / 1e3) / 1e12
        line = {
            "metric": cfg["metric"], "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic randn (reference minimal_example.py style), pretrained XFeat weights",
            "config": {"workload": cfg["workload"], "pairs_per_gpu": BATCH, "top_k": TOPK,
                       "l2": f"inputs {2 * h1.numel() * 4 // 1000000} MB/step > 126 MB L2", "parallelism": f"pair-sharded x{world}",
                       **cfg_extra},
            "e2e": {"value": pairs / (e2e_ms / 1e3), "unit": "pairs/s", "h2d_bytes_per_step": int(2 * h1.numel() * 4),
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps, "h2d_only_gbs": h2d_gbs,
                    "api": "XFeat.match_xfeat_star(host tensors)" if star else "XFeat.match_xfeat_stream(pinned host batches)",
                    "note": "fp32 images (the reference's synthetic input style): bound by the host link, see h2d_only_gbs"},
            "sustained": {"value": BATCH * world * n_sus / (sus_ms / 1e3), "unit": "pairs/s", "steps": n_sus, "seconds": sus_ms / 1e3},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": kname, "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "peak_kind": f"{pk_kind} bf16 dense, sustained", "ms_per_launch": dom_ms,
                         "note": note,
                         "traffic": (ncu["dram_bytes_read"] + ncu["dram_bytes_write"]) if ncu else None, "ncu": ncu},
        }
        if e2e_u8_ms:
            line["e2e_u8"] = {"value": pairs / (e2e_u8_ms / 1e3), "unit": "pairs/s", "h2d_bytes_per_step": hu_bytes,
                              "ms_per_step": e2e_u8_ms / args.steps, "api": "XFeat.match_xfeat_stream(pinned uint8 HWC numpy batches)",
                              "input": "uint8 HWC images, /255 on device (camera / cv2 callers)"}
        if world == 1 and not args.no_cpu:
            try:
                c = cpu_arm_subprocess(args.config, cfg["cpu_pairs"], 2, 1)
                line["cpu_baseline"] = {"value": c["pairs_per_s"], "unit": "pairs/s", "cores": c["threads"], "kind": c["kind"],
                                        "sample": cpu_sample_text(c, args.config)}
            except Exception as e:   # reported, never silently dropped
                line["cpu_baseline"] = {"value": None, "unit": "pairs/s", "cores": 0, "kind": "failed", "sample": str(e)[-300:]}
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def last_step_outputs(out, star: bool):
    """The arrays the timed step returns, as float32 / float64 host arrays.  Rows past a pair's count hold no result and are
    zeroed, so two runs of the same build give identical files."""
    import numpy as np

    def valid_rows(x, n):
        x = x.float().cpu().numpy()
        x[np.arange(x.shape[1])[None, :] >= np.maximum(n, 0)[:, None]] = 0
        return x

    if star:
        m, n_ref, cnt = out
        n_ref = n_ref.cpu().numpy()
        return {"matches": valid_rows(m, n_ref), "n_matches": n_ref.astype(np.float64),
                "n_coarse_matches": cnt.cpu().numpy().astype(np.float64)}
    mk0, mk1, cnt, n1, n2 = out
    cnt = cnt.cpu().numpy()
    return {"mkpts0": valid_rows(mk0, cnt), "mkpts1": valid_rows(mk1, cnt), "n_matches": cnt.astype(np.float64),
            "n_keypoints0": n1.cpu().numpy().astype(np.float64), "n_keypoints1": n2.cpu().numpy().astype(np.float64)}


def write_outputs(path: str, arrays: dict):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    if len(sys.argv) >= 6 and sys.argv[1] == "--cpu-arm-worker":
        print(json.dumps(cpu_arm(sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]))))
        return
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="sparse", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's batch) to DIR/<name>.npy; the inputs are seeded, "
                         "so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
