"""The C++ shim (reference call surface over the C ABI) builds with g++ against libygz_b200.so (CPU suite) and
reproduces the oracle's numbers when driven like test/test_orb_match.cpp (GPU suite)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def shim_exe(tmp_path_factory):
    """The shim test binary, built in a temporary directory: the repository tree may be read-only."""
    from ygz_slam_b200 import capi
    capi.load_library()
    exe = tmp_path_factory.mktemp("cpp_shim") / "cpp_shim_test"
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-o", str(exe), str(ROOT / "tests" / "cpp_shim_test.cpp"),
           f"-L{ROOT / 'ygz_slam_b200'}", "-lygz_b200", f"-Wl,-rpath,{ROOT / 'ygz_slam_b200'}"]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


def test_shim_compiles_and_links_without_cuda_headers(shim_exe):
    """Host C++ only needs include/ygz_b200.h + the shim header: no CUDA toolkit on the include path."""
    assert shim_exe.exists()
    r = subprocess.run([str(shim_exe)], capture_output=True)
    assert r.returncode == 2  # usage error, i.e. the binary starts and the shared library resolves


@pytest.mark.gpu
def test_shim_reproduces_oracle(shim_exe, oracle, tmp_path):
    from ygz_slam_b200 import se3, synth
    g1, d1, T1 = synth.stream_frame(1)
    g2, _, T2 = synth.stream_frame(4)
    Trel = se3.mul(T2, se3.inv(T1))
    blob = tmp_path / "in.bin"
    with open(blob, "wb") as f:
        f.write(g1.tobytes()); f.write(g2.tobytes()); f.write(d1.astype(np.float32).tobytes()); f.write(Trel.astype(np.float64).tobytes())
    voc_file = tmp_path / "voc.bin"
    voc_data = synth.make_vocabulary(k=8, L=5, seed=21)
    voc_file.write_bytes(voc_data)
    g3, _, T3 = synth.stream_frame(16)
    T31 = se3.mul(T3, se3.inv(T1))
    blob3 = tmp_path / "third.bin"
    with open(blob3, "wb") as f:
        f.write(g3.tobytes()); f.write(T31.astype(np.float64).tobytes())
    r = subprocess.run([str(shim_exe), str(blob), str(voc_file), str(blob3)], capture_output=True, text=True, check=True)
    lines = r.stdout.strip().splitlines()
    f1 = oracle.detect(oracle.build_pyramid(g1, 3))
    f2 = oracle.detect(oracle.build_pyramid(g2, 3))
    idx, dist = oracle.match_bf(f1["desc"], f2["desc"], True)
    want = f"features {f1['n']} {f2['n']} matches {(idx >= 0).sum()} dist_sum {dist[idx >= 0].sum()}"
    assert lines[0] == want
    ok, err = lines[1].split()[2], float(lines[1].split()[-1])
    assert ok == "1" and err < 2e-3
    assert int(lines[2].split()[-1]) > 0.8 * len(range(0, f1["n"], 4))
    # Tracker (KLT) against the oracle: same survivors (status && InFrame(pt, 20)) and mean disparity
    ref = np.stack([f1["px"], f1["py"]], 1).astype(np.float32)
    cur, st, _ = oracle.klt(g1, g2, ref, ref.copy())
    inside = (cur[:, 0] >= 20) & (cur[:, 0] < 620) & (cur[:, 1] >= 20) & (cur[:, 1] < 460)
    keep = st.astype(bool) & inside
    parts = lines[3].split()
    assert parts[2] == "1" and abs(int(parts[4]) - keep.sum()) <= 3
    want_disp = np.linalg.norm(ref[keep] - cur[keep], axis=1).mean()
    assert abs(float(parts[6]) - want_disp) < 0.02
    # both bundle-adjustment flavours (ba::LocalBAG2O, ba::LocalBA) on the test_local_ba.cpp fixture: noise-free
    # observations, so the reprojection error must collapse; key-frame 0 keeps its pose
    for line, name in ((lines[4], "g2o"), (lines[7], "ceres")):
        parts = line.split()
        assert parts[1] == name and float(parts[3]) > 1.0 and float(parts[5]) < 1e-3 and parts[7] == "0"
    # ba::OptimizeCurrent (pose + points, Huber 0.1) and ba::OptimizeCurrentPointOnly after perturbing the converged map
    oc, op = lines[5].split(), lines[6].split()
    assert oc[0] == "optimize_current" and float(oc[2]) > 0.5 and float(oc[4]) < 1e-3 and oc[6] == "0"
    assert op[0] == "optimize_point_only" and float(op[2]) > 0.5 and float(op[4]) < 1e-3
    # slot ownership (a live key-frame keeps its pyramid; exhaustion is reported, not silently recycled) and the 8b helpers
    sl = lines[8].split()
    assert sl[0] == "slots" and sl[4] == "1" and sl[6] == "1" and sl[8] == "1" and sl[10] == "1"
    assert abs(float(sl[12]) - (-(1.0 + 0.1 * 0.1 / 4.0))) < 1e-9      # JacobXYZ2Cam(0.1, -0.2, 2)(0, 4) = -(1 + x^2/z^2)
    # DBoW3 front (ORBVocabulary::loadFromBinaryFile, Frame::ComputeBoW, Matcher::SearchByBoW with the shim's th_low = 65)
    v = oracle.vocab_load(voc_data)
    _, n1, _, bw1, bv1 = oracle.bow_transform(v, f1["desc"], 4)
    _, n2, _, _, _ = oracle.bow_transform(v, f2["desc"], 4)
    om, ocnt = oracle.search_by_bow(f1["desc"], n1, f1["angle"], f2["desc"], n2, f2["angle"], th_low=65, knn_ratio=0.9, check_orientation=False)
    h = 0
    for i in np.flatnonzero(om >= 0):
        h = (h * 31 + int(i) * 7 + int(om[i])) % 1000003
    bl = lines[9].split()
    assert bl[0] == "bow" and int(bl[2]) == oracle.vocab_info(v)["words"] and int(bl[4]) == len(bw1)
    assert int(bl[6]) == len(set(n1[n1 >= 0])) and int(bl[8]) == int((n1 >= 0).sum())
    assert abs(float(bl[10]) - bv1.sum()) < 1e-10 and int(bl[12]) == ocnt and int(bl[14]) == int((om >= 0).sum()) and int(bl[16]) == h
    oracle.vocab_free(v)
    # LocalMapping::CreateNewMapPoints: the same composition on the oracle's functions
    v2 = oracle.vocab_load(voc_data)
    cml = [l for l in lines if l.startswith("create_new_map_points")][0].split()
    f3 = oracle.detect(oracle.build_pyramid(g3, 3))
    _, n3, _, _, _ = oracle.bow_transform(v2, f3["desc"], 4)
    want_new, want_assoc, want_sum = _create_new_map_points_on_oracle(oracle, g1, g3, d1, T31, f1, f3, n1, n3)
    assert abs(int(cml[2]) - want_new) <= 2 and abs(int(cml[4]) - want_assoc) <= 2 and want_new >= 1 and want_assoc > 20
    if int(cml[2]) == want_new:
        assert np.allclose([float(cml[6]), float(cml[7]), float(cml[8])], want_sum, rtol=0, atol=1e-6)
    # Initializer::FindModels on the same matches: scores, inlier counts and F21(2,2) are the oracle's, bit for bit
    m1 = np.stack([f1["px"], f1["py"]], 1)[idx >= 0]
    m2 = np.stack([f2["px"], f2["py"]], 1)[idx[idx >= 0]]
    ro = oracle.initializer_ransac(m1, m2, oracle.initializer_sets(len(m1), 200))
    il = [l for l in lines if l.startswith("initializer")][0].split()
    assert il[0] == "initializer" and int(il[2]) == len(m1)
    assert il[6] == "%.3f" % ro["score_H"] and il[8] == "%.3f" % ro["score_F"]
    assert int(il[10]) == int(ro["inliers_H"].sum()) and int(il[12]) == int(ro["inliers_F"].sum())
    assert il[14] == "%.9e" % ro["F21"][2, 2]
    assert int(il[4]) == int(ro["score_H"] / (ro["score_H"] + ro["score_F"]) > 0.4)
    # Initializer::TryInitialize end to end (model choice + ReconstructF / ReconstructH)
    use_h = bool(ro["score_H"] / (ro["score_H"] + ro["score_F"]) > 0.4)
    rq = oracle.initializer_reconstruct(m1, m2, use_h, ro["H21"] if use_h else ro["F21"], ro["inliers_H"] if use_h else ro["inliers_F"])
    tl = [l for l in lines if l.startswith("try_initialize")][0].split()
    assert tl[0] == "try_initialize" and int(tl[2]) == int(rq["ok"])
    assert int(tl[4]) == (int(rq["triangulated"].sum()) if rq["ok"] else 0)
    if rq["ok"]:
        # quaternion round trip inside the shim's SE3: compare with a tolerance
        assert np.allclose([float(tl[6]), float(tl[7]), float(tl[8])], rq["t21"], atol=1e-9) and abs(float(tl[10]) - rq["R21"][0, 0]) < 1e-9


def _create_new_map_points_on_oracle(oracle, g1, g2, d1, Trel, f1, f2, node1, node2):
    """LocalMapping.cpp:375-571 with frame 2 as the new key-frame and frame 1 as its only neighbour, on the oracle's
    SearchForTriangulation / DepthFromTriangulation / FindDirectProjection (the twin of the shim's LocalMapping)."""
    from ygz_slam_b200 import se3, synth
    fx, fy, cx, cy = (float(np.float32(v)) for v in (synth.FX, synth.FY, synth.CX, synth.CY))
    p_cur, p_nb = oracle.build_pyramid(g2, 3), oracle.build_pyramid(g1, 3)
    I = np.eye(4)[:3]
    T_cur, T_nb = Trel, I
    T12 = se3.mul(T_cur, se3.inv(T_nb))
    t = T12[:, 3]
    hat = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    E12 = hat @ T12[:, :3]
    px_cur = np.stack([f2["px"], f2["py"]], 1).astype(np.float64)
    px_nb = np.stack([f1["px"], f1["py"]], 1).astype(np.float64)
    depth_nb = d1[px_nb[:, 1].astype(int), px_nb[:, 0].astype(int)].astype(np.float32).astype(np.float64)
    # neighbour map points on every second feature (camera 1 = world)
    mp_nb = {i: np.array([(px_nb[i, 0] - cx) * depth_nb[i] / fx, (px_nb[i, 1] - cy) * depth_nb[i] / fy, depth_nb[i]]) for i in range(0, len(px_nb), 2)}
    mp_cur = {}
    # baseline against the neighbour's mean map-point depth (LocalMapping.cpp:394-399)
    c_cur, c_nb = se3.inv(T_cur)[:, 3], se3.inv(T_nb)[:, 3]
    mean_depth = np.mean([(T_nb[:, :3] @ pw + T_nb[:, 3])[2] for pw in mp_nb.values()])
    if np.linalg.norm(c_cur - c_nb) / mean_depth < 0.01:
        return 0, 0, np.zeros(3)
    m = oracle.search_for_triangulation(f2["desc"], px_cur, node2, f1["desc"], px_nb, node1, E12, th_low=65, epipolar_dsqr=1e-4)
    T21 = se3.inv(T12)

    def p2c(px, depth=1.0):
        return np.array([(px[0] - cx) * depth / fx, (px[1] - cy) * depth / fy, depth])

    def c2p(p):
        return np.array([fx * p[0] / p[2] + cx, fy * p[1] / p[2] + cy])

    n_new = n_assoc = 0
    total = np.zeros(3)
    for i1 in range(len(px_cur)):
        i2 = int(m[i1])
        if i2 < 0:
            continue
        has1, has2 = i1 in mp_cur, i2 in mp_nb
        if not has1 and not has2:
            pt1, pt2 = p2c(px_cur[i1]), p2c(px_nb[i2])
            if pt1 @ pt2 / (np.linalg.norm(pt1) * np.linalg.norm(pt2)) >= 0.9998:
                continue
            d1_, d2_, ok = oracle.depth_from_triangulation(T21, pt1, pt2)
            if not ok[0] or d1_[0] < 0 or d2_[0] < 0:
                continue
            px, _, okp = oracle.find_direct_projection(p_cur, p_nb, 640, 480, 3, T_cur, T_nb, px_cur[i1:i1 + 1], np.array([d1_[0]]),
                                                       f2["level"][i1:i1 + 1], px_nb[i2:i2 + 1].copy())
            if not okp[0]:
                continue
            px_nb[i2] = px[0]
            pt2 = p2c(px_nb[i2])
            d1_, d2_, ok = oracle.depth_from_triangulation(T21, pt1, pt2)
            if not ok[0] or d1_[0] < 0 or d2_[0] < 0:
                continue
            tri = pt1 * d1_[0]
            if np.linalg.norm(c2p(T21[:, :3] @ tri + T21[:, 3]) - px_nb[i2]) > 5.991:
                continue
            Ti = se3.inv(T_cur)
            world = Ti[:, :3] @ tri + Ti[:, 3]
            mp_cur[i1] = world
            mp_nb[i2] = world
            total += world
            n_new += 1
        elif has2 and not has1:
            pw = mp_nb[i2]
            if np.linalg.norm(c2p(T_cur[:, :3] @ pw + T_cur[:, 3]) - px_cur[i1]) > 5.991:
                continue
            mp_cur[i1] = pw
            n_assoc += 1
        elif has1 and not has2:
            pw = mp_cur[i1]
            if np.linalg.norm(c2p(T_nb[:, :3] @ pw + T_nb[:, 3]) - px_nb[i2]) > 5.991:
                continue
            mp_nb[i2] = pw
            n_assoc += 1
    return n_new, n_assoc, total
