"""SURVEY 8f-2 / 8f-3: the batched evaluation-harness callers and the GPU geometric verification.

RANSAC is stochastic in the reference too (README.md:163), and its estimators live in un-vendored packages (OpenCV, poselib):
the checks are agreement with OpenCV on the same correspondences (inlier sets, model error), exact equality of the batched
matcher adapter with per-pair calls, and equality of the resulting AUC with the reference pipeline run pair by pair."""
import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xf():
    from accelerated_features_b200 import XFeat
    return XFeat()


def synth_correspondences(rng, n, inlier_frac, noise, w=640, h=480):
    """n correspondences under a random mild homography; outliers uniform in the image."""
    ang = rng.uniform(-0.3, 0.3)
    s = rng.uniform(0.8, 1.2)
    H = np.array([[s * np.cos(ang), -s * np.sin(ang), rng.uniform(-40, 40)],
                  [s * np.sin(ang), s * np.cos(ang), rng.uniform(-30, 30)],
                  [rng.uniform(-2e-4, 2e-4), rng.uniform(-2e-4, 2e-4), 1.0]])
    p0 = np.stack([rng.uniform(0, w, n), rng.uniform(0, h, n)], 1)
    q = (H @ np.concatenate([p0, np.ones((n, 1))], 1).T).T
    p1 = q[:, :2] / q[:, 2:]
    inl = rng.uniform(size=n) < inlier_frac
    p1 = p1 + rng.normal(0, noise, p1.shape)
    p1[~inl] = np.stack([rng.uniform(0, w, (~inl).sum()), rng.uniform(0, h, (~inl).sum())], 1)
    return p0.astype(np.float32), p1.astype(np.float32), inl, H


def transfer_err(H, p0, p1):
    q = (H @ np.concatenate([p0, np.ones((len(p0), 1))], 1).T).T
    return np.linalg.norm(q[:, :2] / q[:, 2:] - p1, axis=1)


def test_ransac_homography_vs_opencv_synthetic():
    from accelerated_features_b200.geometry import find_homography_batch
    rng = np.random.default_rng(0)
    B, nmax, thr = 8, 3000, 3.0
    sets = [synth_correspondences(rng, n, f, 0.7) for n, f in
            [(3000, 0.6), (2000, 0.5), (1500, 0.35), (800, 0.7), (300, 0.5), (64, 0.8), (3, 1.0), (2500, 0.25)]]
    p0 = np.zeros((B, nmax, 2), np.float32); p1 = np.zeros((B, nmax, 2), np.float32)
    cnt = np.array([len(s[0]) for s in sets], np.int32)
    for b, s in enumerate(sets):
        p0[b, :cnt[b]] = s[0]; p1[b, :cnt[b]] = s[1]
    H, mask, n_inl = find_homography_batch(torch.from_numpy(p0).cuda(), torch.from_numpy(p1).cuda(), torch.from_numpy(cnt).cuda(),
                                           thr=thr, iters=1024, seed=1)
    H, mask, n_inl = H.cpu().numpy().astype(np.float64), mask.cpu().numpy(), n_inl.cpu().numpy()
    for b, (a, c, inl, Hgt) in enumerate(sets):
        n = cnt[b]
        if n < 4:
            assert n_inl[b] == 0 and not mask[b].any()
            continue
        assert not mask[b, n:].any() and mask[b, :n].sum() == n_inl[b]
        Hcv, mcv = cv2.findHomography(a, c, cv2.USAC_MAGSAC, thr, maxIters=2000, confidence=0.9999)
        mcv = mcv.ravel() > 0
        agree = (mask[b, :n] == mcv).mean()
        e_gpu = transfer_err(H[b], a[inl], c[inl]).mean()
        e_cv = transfer_err(Hcv, a[inl], c[inl]).mean()
        print(f"pair {b}: n={n} inliers gpu {n_inl[b]} cv {mcv.sum()} true {inl.sum()} agree {agree:.3f} err gpu {e_gpu:.3f} cv {e_cv:.3f}")
        assert agree >= 0.97                                  # same classification of almost every correspondence
        assert abs(int(n_inl[b]) - int(mcv.sum())) <= max(3, 0.03 * n)
        assert e_gpu <= e_cv + 0.15                           # the model explains the true inliers as well as OpenCV's (px)
        assert mask[b, :n][inl].mean() > 0.93                 # recall of the true inliers (noise 0.7 px, threshold 3 px)
    # deterministic for a given seed
    H2, mask2, _ = find_homography_batch(torch.from_numpy(p0).cuda(), torch.from_numpy(p1).cuda(), torch.from_numpy(cnt).cuda(),
                                         thr=thr, iters=1024, seed=1)
    assert np.array_equal(mask2.cpu().numpy(), mask) and np.allclose(H2.cpu().numpy(), H)


def test_verified_batch_on_assets(xf, assets_vga):
    """The notebook / demo flow: match_xfeat then findHomography, here in one batched device call."""
    from accelerated_features_b200.geometry import find_homography
    ref, tgt = assets_vga
    out = xf.match_xfeat_verified_batch(np.stack([ref, tgt]), np.stack([tgt, ref]), top_k=4096, ransac_thr=3.5, iters=2048)
    mk0, mk1 = xf.match_xfeat(ref, tgt, top_k=4096)
    assert np.array_equal(out[0]["mkpts0"], mk0) and np.array_equal(out[0]["mkpts1"], mk1)
    Hcv, mcv = cv2.findHomography(mk0, mk1, cv2.USAC_MAGSAC, 3.5, maxIters=2000, confidence=0.9999)
    mcv = mcv.ravel() > 0
    inl = out[0]["inliers"]
    print(f"asset pair: {len(mk0)} matches, inliers gpu {inl.sum()} cv {mcv.sum()}, agreement {(inl == mcv).mean():.3f}")
    # the scene is not one plane: the dominant-plane inlier sets of two robust estimators overlap largely, not exactly
    assert inl.sum() >= 0.85 * mcv.sum() and (inl & mcv).sum() >= 0.8 * min(inl.sum(), mcv.sum())
    # the reverse pair's homography is (close to) the inverse
    P = out[0]["H"].astype(np.float64) @ out[1]["H"].astype(np.float64)
    P /= P[2, 2]
    c = np.array([[320, 240, 1.0]]).T
    assert np.linalg.norm((P @ c)[:2, 0] / (P @ c)[2, 0] - c[:2, 0]) < 6.0
    H1, m1 = find_homography(mk0, mk1, thr=3.5, iters=2048)
    assert H1.shape == (3, 3) and m1.shape == (len(mk0), 1) and m1.dtype == np.uint8


def make_plane_pair(img, K, rvec, t, out_hw=None):
    """Second view of a fronto-parallel plane at depth 1 (n = (0,0,1), d = 1): x1 ~ K (R + t n^T) K^-1 x0, X1 = R X0 + t."""
    R, _ = cv2.Rodrigues(np.asarray(rvec, np.float64))
    Hm = K @ (R + np.outer(t, [0, 0, 1.0])) @ np.linalg.inv(K)
    h, w = img.shape[:2] if out_hw is None else out_hw
    warped = cv2.warpPerspective(img, Hm, (w, h), flags=cv2.INTER_LINEAR)
    T = np.eye(4); T[:3, :3] = R; T[:3, 3] = t
    return warped, T


def plane_pose_samples(ref_img, tgt_img):
    """Four synthetic two-view samples of the asset images (two image shapes) in run_pose_benchmark's format."""
    K = np.array([[520.0, 0, 320], [0, 520.0, 240], [0, 0, 1]])
    samples = []
    poses = [((0.02, -0.05, 0.03), (0.10, 0.02, 0.05)), ((-0.04, 0.06, -0.05), (-0.08, 0.05, 0.10)),
             ((0.05, 0.03, 0.08), (0.05, -0.09, -0.06)), ((0.0, 0.08, -0.02), (0.12, 0.0, 0.02))]
    for i, (rv, t) in enumerate(poses):
        base = ref_img if i % 2 == 0 else tgt_img
        if i >= 2:   # a second image shape in the same list: the adapter must bucket by shape
            base = np.ascontiguousarray(base[32:416, 64:576])
            Kc = K.copy(); Kc[0, 2] -= 64; Kc[1, 2] -= 32
        else:
            Kc = K
        warped, T = make_plane_pair(base, Kc, rv, np.asarray(t))
        samples.append({"image0": base, "image1": warped, "scale0": np.ones(2, np.float32), "scale1": np.ones(2, np.float32),
                        "K0": Kc, "K1": Kc, "T_0to1": T})
    return samples


def test_batched_harness_equals_per_pair_and_reference_auc(xf, golden, assets_vga):
    from accelerated_features_b200.evalharness import batched_matcher, run_pose_benchmark
    samples = plane_pose_samples(*assets_vga)
    match_pairs = batched_matcher(xf, "sparse", top_k=2048, batch_size=3)
    pairs = [(s["image0"], s["image1"]) for s in samples]
    got = match_pairs(pairs)
    for (a, b), (g0, g1) in zip(pairs, got):                       # the adapter == per-pair public calls, bit for bit
        s0, s1 = xf.match_xfeat(a, b, top_k=2048)
        assert np.array_equal(g0, s0) and np.array_equal(g1, s1)

    # the reference pipeline: the unmodified modules.xfeat.XFeat's match_xfeat on the CPU, one pair at a time, stored by
    # tools/make_golden_pose.py
    g = golden("g6_pose_matches.npz")
    want = [(g[f"mkpts0_{i}"], g[f"mkpts1_{i}"]) for i in range(len(samples))]
    for (g0, g1), (w0, w1) in zip(got, want):
        gs = {tuple(map(float, np.concatenate([a, b]))) for a, b in zip(g0, g1)}
        ws = {tuple(map(float, np.concatenate([a, b]))) for a, b in zip(w0, w1)}
        assert len(gs ^ ws) <= 4, len(gs ^ ws)                     # near-tie matches only (tests/test_gpu_e2e.py protocol)

    def pose_fn(*a, **k):
        from accelerated_features_b200.evalharness import estimate_pose_opencv
        cv2.setRNGSeed(7)
        return estimate_pose_opencv(*a, **k)

    mine = run_pose_benchmark(match_pairs, samples, ransac_thr=2.5, batch_size=3, pose_fn=pose_fn)
    theirs = run_pose_benchmark(lambda ps: want, samples, ransac_thr=2.5, batch_size=len(samples), pose_fn=pose_fn)
    print("AUC batched B200:", {k: round(v, 4) for k, v in mine.items() if k != "pairs"})
    print("AUC reference   :", {k: round(v, 4) for k, v in theirs.items() if k != "pairs"})
    from tests.parity_util import record
    record("eval_harness_auc", b200={k: v for k, v in mine.items() if k != "pairs"},
           reference={k: v for k, v in theirs.items() if k != "pairs"})
    for k in ("auc@5", "auc@10", "auc@20", "mAcc@5", "mAcc@10", "mAcc@20"):
        assert abs(mine[k] - theirs[k]) <= 0.02, k
    assert mine["mAcc@20"] >= 0.5                                   # the synthetic poses are recoverable at all


def test_star_adapter(xf, assets_vga):
    from accelerated_features_b200.evalharness import batched_matcher
    ref, tgt = assets_vga
    small = np.ascontiguousarray(ref[:320, :448])
    pairs = [(ref, tgt), (tgt, ref), (small, small)]
    got = batched_matcher(xf, "star", top_k=2048, batch_size=2)(pairs)
    for (a, b), (g0, g1) in zip(pairs, got):
        s0, s1 = xf.match_xfeat_star(a, b, top_k=2048)
        assert g0.shape == s0.shape and np.allclose(g0, s0, atol=1e-4) and np.array_equal(g1, s1)


def synth_two_view(rng, n, inlier_frac, noise_px, f=600.0):
    """Random 3-D points seen by two calibrated cameras (X1 = R X0 + t), pixel noise, outliers."""
    rv = rng.uniform(-0.25, 0.25, 3)
    R, _ = cv2.Rodrigues(rv)
    t = rng.uniform(-1, 1, 3); t /= np.linalg.norm(t)
    X0 = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(3, 9, n)], 1)
    X1 = (R @ X0.T).T + t
    K = np.array([[f, 0, 320], [0, f, 240], [0, 0, 1.0]])
    p0 = (K @ (X0 / X0[:, 2:]).T).T[:, :2] + rng.normal(0, noise_px, (n, 2))
    p1 = (K @ (X1 / X1[:, 2:]).T).T[:, :2] + rng.normal(0, noise_px, (n, 2))
    inl = rng.uniform(size=n) < inlier_frac
    p1[~inl] = np.stack([rng.uniform(0, 640, (~inl).sum()), rng.uniform(0, 480, (~inl).sum())], 1)
    T = np.eye(4); T[:3, :3] = R; T[:3, 3] = t
    return p0.astype(np.float32), p1.astype(np.float32), inl, K, T


def test_ransac_essential_pose_vs_opencv():
    """Relative pose from the GPU essential-matrix RANSAC on non-planar synthetic scenes: pose error against ground truth no worse
    than OpenCV's 5-point RANSAC + recoverPose on the same correspondences (+1 degree), inliers recalled."""
    from accelerated_features_b200.evalharness import estimate_pose_gpu, estimate_pose_opencv, relative_pose_error
    rng = np.random.default_rng(3)
    worst = 0.0
    for n, frac in [(2000, 0.6), (1200, 0.45), (600, 0.7), (300, 0.5)]:
        p0, p1, inl, K, T = synth_two_view(rng, n, frac, 0.5)
        got = estimate_pose_gpu(p0, p1, K, K, 1.5, iters=16384, seed=5)   # 8-point samples: 0.45^8 = 0.17 % all-inlier
        cv2.setRNGSeed(1)
        ref = estimate_pose_opencv(p0, p1, K, K, 1.5)
        assert got is not None and ref is not None
        te, re_ = relative_pose_error(T, got[0], got[1])
        te_cv, re_cv = relative_pose_error(T, ref[0], ref[1])
        rec = got[2][inl].mean()
        print(f"n={n} inl={frac}: gpu err (t {te:.2f}, R {re_:.2f}) deg, cv (t {te_cv:.2f}, R {re_cv:.2f}); inlier recall {rec:.3f}, false {got[2][~inl].mean():.3f}")
        assert max(te, re_) <= max(te_cv, re_cv) + 1.0 and max(te, re_) < 3.0
        assert rec > 0.9 and got[2][~inl].mean() < 0.1
        worst = max(worst, te, re_)
    from tests.parity_util import record
    record("ransac_essential_synthetic", worst_pose_error_deg=worst)
