"""Small, bounded inputs for `compute-sanitizer --tool racecheck` on the thread-block-cluster solvers (local_ba2_kernel in its
lane / warp / CTA-block / scalar solver variants, local_ba_kernel, pose_only_kernel).  The parity suite is too slow
under racecheck (the cluster kernels run ~1000x slower), so this drives the same entry points through the C ABI with a few
LM iterations on small scenes and prints one line per case:

    compute-sanitizer --tool racecheck --print-limit 20 python tools/racecheck_clusters.py

No oracle here: the results are only checked for being finite and for a cost that does not increase."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from ygz_slam_b200 import Context, se3, synth  # noqa: E402


def g2o(v):
    v = np.asarray(v)
    return np.concatenate([v[..., 3:], v[..., :3]], -1)


def t_aa(v):
    out = []
    for x in np.atleast_2d(v):
        T = se3.se3_exp(x)
        out.append(np.r_[T[:, 3], se3.so3_log(T[:, :3])])
    return np.array(out)


def pose_only_case(ctx, t0):
    # pose-only refinement: 3 frames (3 clusters), one with outliers
    rng = np.random.default_rng(7)
    sc = synth.ba_scene(n_kf=5, n_pt=300, target_obs=1200, seed=62)
    offs, pws, pxs, Ts = [0], [], [], []
    for k in range(3):
        sel = sc["kf_idx"] == (k + 1)
        pw = sc["pts_true"][sc["pt_idx"][sel]]
        px = sc["px"][sel].copy()
        if k == 1:
            px[::7] += 25
        offs.append(offs[-1] + len(pw))
        pws.append(pw); pxs.append(px)
        Ts.append(se3.se3_exp(sc["poses_true"][k + 1] + rng.normal(0, 0.003, 6)).reshape(-1))
    T, inl, depth, cnt = ctx.pose_only(offs, np.concatenate(pws), np.concatenate(pxs), np.stack(Ts))
    assert np.isfinite(T).all() and (cnt > 0).all()
    print(f"pose_only 3 frames x ~{offs[1]} points inliers={list(map(int, cnt))} ok t={time.time() - t0:.1f}s", flush=True)


def main():
    iters = int(os.environ.get("RACECHECK_ITERS", "3"))
    ctx = Context(0)
    t0 = time.time()
    # (key-frames, YGZB_BA_SOLVER): 2 / 3 key-frames -> one lane, 4 -> one warp, 8 -> CTA 6x6 blocks, 14 -> scalar CTA; "1" = scalar everywhere
    cases = ((3, "0"), (4, "0"), (8, "0"), (2, "0"), (14, "0"), (4, "1"))
    pose_only_case(ctx, t0)          # the two kernels of the C5 loop first: pose-only, then the 3-key-frame BA
    for n_kf, solver in cases:
        os.environ["YGZB_BA_SOLVER"] = solver
        sc = synth.ba_scene(n_kf=n_kf, n_pt=96, target_obs=96 * min(n_kf, 4), seed=40 + n_kf)
        fixed = np.zeros(n_kf, np.uint8)
        fixed[0] = 1
        n_obs = len(sc["kf_idx"])
        P, X, out, st = ctx.local_ba([0, n_kf], [0, 96], [0, n_obs], g2o(sc["poses_noisy"]), fixed, sc["pts_noisy"], sc["kf_idx"],
                                     sc["pt_idx"], sc["px"], max_iters=iters)
        ok = np.isfinite(P).all() and np.isfinite(X).all() and st[0]["chi2_final"] <= st[0]["chi2_initial"]
        print(f"local_ba  n_kf={n_kf:2d} solver={solver} obs={n_obs} chi2 {st[0]['chi2_initial']:.1f} -> {st[0]['chi2_final']:.3f} "
              f"ok={bool(ok)} t={time.time() - t0:.1f}s", flush=True)
        assert ok
    os.environ.pop("YGZB_BA_SOLVER", None)

    # two problems in one launch (two clusters), the second with a fixed observer
    a = synth.ba_scene(n_kf=3, n_pt=96, target_obs=288, seed=51)
    b = synth.ba_scene(n_kf=5, n_pt=64, target_obs=256, seed=52)
    fa = np.zeros(3, np.uint8); fa[0] = 1
    fb = np.zeros(5, np.uint8); fb[[0, 3]] = 1
    na, nb = len(a["kf_idx"]), len(b["kf_idx"])
    P, X, out, st = ctx.local_ba([0, 3, 8], [0, 96, 160], [0, na, na + nb], np.concatenate([g2o(a["poses_noisy"]), g2o(b["poses_noisy"])]),
                                 np.concatenate([fa, fb]), np.concatenate([a["pts_noisy"], b["pts_noisy"]]),
                                 np.concatenate([a["kf_idx"], b["kf_idx"]]), np.concatenate([a["pt_idx"], b["pt_idx"]]),
                                 np.concatenate([a["px"], b["px"]]), max_iters=iters)
    assert np.isfinite(P).all() and np.isfinite(X).all()
    print(f"local_ba  batched 2 problems ok t={time.time() - t0:.1f}s", flush=True)

    # Ceres flavour (ba.cu cluster kernel)
    sc = synth.ba_scene(n_kf=4, n_pt=96, target_obs=384, seed=61)
    fixed = np.zeros(4, np.uint8); fixed[0] = 1
    n_obs = len(sc["kf_idx"])
    res = ctx.local_ba_ceres([0, 4], [0, 96], [0, n_obs], t_aa(sc["poses_noisy"]), fixed, sc["pts_noisy"], sc["kf_idx"], sc["pt_idx"], sc["px"],
                             max_iters=iters)
    assert np.isfinite(res[0]).all() and np.isfinite(res[1]).all()
    print(f"local_ba_ceres ok t={time.time() - t0:.1f}s", flush=True)

    ctx.close()
    print("racecheck_clusters: done")


if __name__ == "__main__":
    main()
