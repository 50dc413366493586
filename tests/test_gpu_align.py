"""GPU parity suite for the photometric alignment path (BASELINE config C3): Align2D / FindDirectProjection
are bit-exact against the oracle (one thread per patch, reference summation order); SparseImgAlign poses
agree within ||log(T_gpu^-1 T_ref)|| < 1e-4 (block-parallel reduction of the normal equations)."""
import numpy as np
import pytest

from ygz_slam_b200 import se3, synth

pytestmark = pytest.mark.gpu


def _scene(oracle, k0=1, k1=4, levels=3):
    g1, d1, T1 = synth.stream_frame(k0)
    g2, _, T2 = synth.stream_frame(k1)
    p1, p2 = oracle.build_pyramid(g1, levels), oracle.build_pyramid(g2, levels)
    f = oracle.detect(p1, n_levels=levels)
    px = np.stack([f["px"], f["py"]], 1)
    depth = d1[f["py"].astype(int), f["px"].astype(int)]
    Trel = se3.mul(T2, se3.inv(T1))
    Xc = np.stack([(px[:, 0] - synth.CX) * depth / synth.FX, (px[:, 1] - synth.CY) * depth / synth.FY, depth], 1)
    Xc2 = (Trel[:, :3] @ Xc.T).T + Trel[:, 3]
    gt = np.stack([synth.FX * Xc2[:, 0] / Xc2[:, 2] + synth.CX, synth.FY * Xc2[:, 1] / Xc2[:, 2] + synth.CY], 1)
    return dict(g1=g1, g2=g2, p1=p1, p2=p2, f=f, px=px, depth=depth, T1=T1, T2=T2, Trel=Trel, gt=gt)


def test_align2d_bit_exact(ctx3, oracle):
    s = _scene(oracle)
    fr = ctx3.frames(2)
    fr.upload(np.stack([s["g1"], s["g2"]]))
    rng = np.random.default_rng(3)
    n = 2000
    # templates cut from frame 1 around random points on random levels, searched in frame 2 from a perturbed guess;
    # some guesses are placed at the border so that the "window leaves the image" break is exercised
    level = rng.integers(0, 3, n).astype(np.uint8)
    ref_border = np.empty((n, 100), np.uint8)
    uv = np.empty((n, 2))
    for i in range(n):
        L = int(level[i])
        img = oracle.level_view(s["p1"], 640, 480, 3, L)
        h, w = img.shape
        x, y = int(rng.integers(6, w - 6)), int(rng.integers(6, h - 6))
        ref_border[i] = img[y - 5:y + 5, x - 5:x + 5].reshape(-1)
        uv[i] = (x + rng.uniform(-2.5, 2.5), y + rng.uniform(-2.5, 2.5))
    uv[:50, 0] = rng.uniform(0, 6, 50)
    slot = np.ones(n, np.int32)
    got_uv, got_ok = fr.align2d(slot, level, ref_border, None, uv, 10)
    conv = 0
    for i in range(n):
        img = oracle.level_view(s["p2"], 640, 480, 3, int(level[i]))
        rb = ref_border[i].reshape(10, 10)
        ok, u, v = oracle.align2d(img, rb, rb[1:9, 1:9], uv[i, 0], uv[i, 1], 10)
        assert ok == got_ok[i], i
        assert u == got_uv[i, 0] and v == got_uv[i, 1], (i, u, v, got_uv[i])
        conv += ok
    assert conv > 400  # small camera motion: a good part of the random patches really converges
    fr.close()


@pytest.mark.parametrize("identity_ref", [True, False])
def test_find_direct_projection_bit_exact(ctx3, oracle, identity_ref):
    s = _scene(oracle)
    fr = ctx3.frames(2)
    fr.upload(np.stack([s["g1"], s["g2"]]))
    rng = np.random.default_rng(7)
    n = len(s["depth"])
    init = s["gt"] + rng.uniform(-2, 2, s["gt"].shape)
    depth = s["depth"].copy()
    depth[::97] = -1.0  # invalid depth -> false (Matcher.cpp:388-392)
    if identity_ref:
        Tr, Tc = np.eye(4)[:3], s["Trel"]
    else:
        Tr, Tc = s["T1"], s["T2"]  # exercises the world/ref-camera mix-up of GetWarpAffineMatrix
    want_px, want_lvl, want_ok = oracle.find_direct_projection(s["p1"], s["p2"], 640, 480, 3, Tr, Tc, s["px"], depth,
                                                               s["f"]["level"], init)
    poses = np.stack([Tr.reshape(-1), Tc.reshape(-1)])
    got_px, got_lvl, got_ok = fr.project_align(np.zeros(n, np.int32), np.ones(n, np.int32), poses, np.zeros(n, np.int32),
                                               np.ones(n, np.int32), s["px"], depth, s["f"]["level"].astype(np.uint8), init)
    assert np.array_equal(got_lvl, want_lvl)
    assert np.array_equal(got_ok, want_ok)
    assert np.array_equal(got_px, want_px)
    if identity_ref:
        assert got_ok.mean() > 0.85
        err = np.linalg.norm(got_px - s["gt"], axis=1)[got_ok]
        assert np.median(err) < 0.25
    fr.close()


def _pose_err(Ta, Tb):
    return float(np.linalg.norm(se3.se3_log(se3.mul(se3.inv(Ta), Tb))))


@pytest.mark.parametrize("levels,max_level", [(3, 2), (8, 3)])
def test_sparse_align_pose_tolerance(levels, max_level, ctx3, ctx8, oracle):
    ctx = ctx3 if levels == 3 else ctx8
    s = _scene(oracle, levels=levels)
    s2 = _scene(oracle, 2, 5, levels=levels)
    fr = ctx.frames(4)
    fr.upload(np.stack([s["g1"], s["g2"], s2["g1"], s2["g2"]]))
    n1, n2 = len(s["depth"]), len(s2["depth"])
    has1 = np.ones(n1, np.uint8)
    has1[::11] = 0
    has2 = np.ones(n2, np.uint8)
    px = np.concatenate([s["px"], s2["px"]])
    depth = np.concatenate([s["depth"], s2["depth"]])
    has = np.concatenate([has1, has2])
    T_ref = np.stack([s["T1"].reshape(-1), s2["T1"].reshape(-1)])
    T, n_meas, iters = fr.sparse_align([0, 2], [1, 3], [0, n1, n1 + n2], px, depth, has, T_ref, T_ref, max_level=max_level)
    for p, (sc, hm) in enumerate(((s, has1), (s2, has2))):
        wT, wn, wit = oracle.sparse_align(sc["p1"], sc["p2"], 640, 480, levels, sc["px"], sc["depth"], hm, sc["T1"], sc["T1"],
                                          max_level=max_level)
        assert _pose_err(T[p], wT) < 1e-4          # stated tolerance (SURVEY 8d)
        assert n_meas[p] == wn
        assert _pose_err(T[p], sc["T2"]) < 2e-3    # and it really aligned: close to the ground-truth pose
    # empty problem: pose untouched, zero measurements
    T0, nm0, _ = fr.sparse_align([0], [1], [0, 0], np.zeros((0, 2)), np.zeros(0), np.zeros(0, np.uint8), T_ref[:1], T_ref[:1])
    assert nm0[0] == 0 and np.allclose(T0[0].reshape(-1), T_ref[0])
    fr.close()


def test_sparse_align_global_staging(ctx3, oracle):
    """A problem whose cluster cannot stage its features in shared memory (more than 8 CTAs x (227 KB - 8 KB) / 360 B
    features) runs from the global staging buffer; the small problem before it checks that the buffer is indexed by the
    problem's CSR offset."""
    s = _scene(oracle)
    g1, d1, T1 = synth.stream_frame(2)
    g2, _, T2 = synth.stream_frame(5)
    p1, p2 = oracle.build_pyramid(g1, 3), oracle.build_pyramid(g2, 3)
    u, v = np.meshgrid(np.arange(4, 636, 5), np.arange(4, 476, 5))
    dense_px = np.stack([u.ravel() + 0.37, v.ravel() + 0.61], 1)
    dense_depth = d1[v.ravel(), u.ravel()]
    n1, n2 = len(s["depth"]), len(dense_depth)
    assert n2 > 8 * ((227 - 8) * 1024 // 360)
    has1 = np.ones(n1, np.uint8)
    has1[::11] = 0
    has2 = np.ones(n2, np.uint8)
    fr = ctx3.frames(4)
    fr.upload(np.stack([s["g1"], s["g2"], g1, g2]))
    T_ref = np.stack([s["T1"].reshape(-1), T1.reshape(-1)])
    T, n_meas, _ = fr.sparse_align([0, 2], [1, 3], [0, n1, n1 + n2], np.concatenate([s["px"], dense_px]),
                                   np.concatenate([s["depth"], dense_depth]), np.concatenate([has1, has2]), T_ref, T_ref)
    for p, (rp, cp, px, depth, hm, Tr, Tgt) in enumerate(((s["p1"], s["p2"], s["px"], s["depth"], has1, s["T1"], s["T2"]),
                                                        (p1, p2, dense_px, dense_depth, has2, T1, T2))):
        wT, wn, _ = oracle.sparse_align(rp, cp, 640, 480, 3, px, depth, hm, Tr, Tr)
        assert _pose_err(T[p], wT) < 1e-4
        assert n_meas[p] == wn
        assert _pose_err(T[p], Tgt) < 2e-3
    fr.close()


def test_align1d_bit_exact(ctx3, oracle):
    """cvutils::Align1D (epipolar 1-D search): u, v, converged flag and h_inv against the oracle."""
    s = _scene(oracle)
    fr = ctx3.frames(2)
    fr.upload(np.stack([s["g1"], s["g2"]]))
    rng = np.random.default_rng(13)
    n = 600
    level = rng.integers(0, 3, n).astype(np.uint8)
    ref_border = np.empty((n, 100), np.uint8)
    uv = np.empty((n, 2))
    ang = rng.uniform(0, 2 * np.pi, n)
    direction = np.stack([np.cos(ang), np.sin(ang)], 1).astype(np.float32)
    for i in range(n):
        img = oracle.level_view(s["p1"], 640, 480, 3, int(level[i]))
        h, w = img.shape
        x, y = int(rng.integers(6, w - 6)), int(rng.integers(6, h - 6))
        ref_border[i] = img[y - 5:y + 5, x - 5:x + 5].reshape(-1)
        t = rng.uniform(-2.5, 2.5)
        uv[i] = (x + t * direction[i, 0], y + t * direction[i, 1])
    got_uv, got_ok, got_h = fr.align1d(np.ones(n, np.int32), level, direction, ref_border, None, uv, 10)
    for i in range(n):
        img = oracle.level_view(s["p2"], 640, 480, 3, int(level[i]))
        rb = ref_border[i].reshape(10, 10)
        ok, u, v, hinv = oracle.align1d(img, float(direction[i, 0]), float(direction[i, 1]), rb, rb[1:9, 1:9], uv[i, 0], uv[i, 1], 10)
        assert ok == got_ok[i] and u == got_uv[i, 0] and v == got_uv[i, 1], i
        assert hinv == got_h[i] or (np.isinf(hinv) and np.isinf(got_h[i]))
    fr.close()


def test_alignment_and_klt_on_another_geometry(oracle):
    """752 x 480, 4 levels (not the 640 x 480 default): FindDirectProjection bit-exact, SparseImgAlign and KLT within
    their tolerances -- the level geometry (pitches, offsets, borders) is a run-time parameter everywhere."""
    from ygz_slam_b200 import Context
    w, h, levels = 752, 480, 4
    tex = synth.texture(0x59475A00, 2048)
    T1, T2 = synth.trajectory(1), synth.trajectory(4)
    g1, d1 = synth.render_plane(tex, T1, noise_sigma=2.0, seed=11, w=w, h=h)
    g2, _ = synth.render_plane(tex, T2, noise_sigma=2.0, seed=12, w=w, h=h)
    p1, p2 = oracle.build_pyramid(g1, levels), oracle.build_pyramid(g2, levels)
    f = oracle.detect(p1, w=w, h=h, n_levels=levels)
    px = np.stack([f["px"], f["py"]], 1)
    depth = d1[f["py"].astype(int), f["px"].astype(int)]
    n = len(depth)
    assert n > 500
    Trel = se3.mul(T2, se3.inv(T1))
    Xc = np.stack([(px[:, 0] - synth.CX) * depth / synth.FX, (px[:, 1] - synth.CY) * depth / synth.FY, depth], 1)
    Xc2 = (Trel[:, :3] @ Xc.T).T + Trel[:, 3]
    gt = np.stack([synth.FX * Xc2[:, 0] / Xc2[:, 2] + synth.CX, synth.FY * Xc2[:, 1] / Xc2[:, 2] + synth.CY], 1)
    init = gt + np.random.default_rng(5).uniform(-2, 2, gt.shape)
    ctx = Context(0, image_width=w, image_height=h, n_levels=levels)
    try:
        fr = ctx.frames(2)
        fr.upload(np.stack([g1, g2]))
        eye = np.eye(4)[:3]
        want_px, want_lvl, want_ok = oracle.find_direct_projection(p1, p2, w, h, levels, eye, Trel, px, depth, f["level"], init)
        z, o = np.zeros(n, np.int32), np.ones(n, np.int32)
        got_px, got_lvl, got_ok = fr.project_align(z, o, np.stack([eye.reshape(-1), Trel.reshape(-1)]), z, o, px, depth,
                                                   f["level"].astype(np.uint8), init)
        assert np.array_equal(got_ok, want_ok) and np.array_equal(got_lvl, want_lvl) and np.array_equal(got_px, want_px)
        assert got_ok.mean() > 0.8
        has = np.ones(n, np.uint8)
        wT, wn, _ = oracle.sparse_align(p1, p2, w, h, levels, px, depth, has, T1, T1, max_level=3)
        gT, gn, _ = fr.sparse_align([0], [1], [0, n], px, depth, has, T1.reshape(1, 12), T1.reshape(1, 12), max_level=3)
        assert gn[0] == wn
        assert np.linalg.norm(se3.se3_log(se3.mul(se3.inv(gT[0]), wT))) < 1e-4
        assert np.linalg.norm(se3.se3_log(se3.mul(se3.inv(gT[0]), T2))) < 5e-3
        ref = px.astype(np.float32)
        want, wst, werr = oracle.klt(g1, g2, ref, ref.copy())
        got, gst, gerr = fr.klt([0], [1], [0, n], ref, ref.copy())
        assert (gst != wst.astype(bool)).mean() < 0.005
        both = gst & wst.astype(bool)
        assert np.abs(got[both] - want[both]).max() < 1e-3 and both.mean() > 0.9
        fr.close()
    finally:
        ctx.close()
