"""The Tanks and Temples registration (K9 registration, csrc/pointcloud.cu, mvs_b200/registration.py) on the GPU against the fp64
oracle (oracle/tnt_register.py): the index search against cKDTree with planted ties, the Umeyama sums against numpy and run to run,
the fp64 update bit for bit, one ICP run on a scene whose every decision has a clear margin, the three stages on noisy scenes, an
end-to-end run from fused depth maps, empty crops and refusals, and the command-line tool."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fusion as fusion_oracle
import tnt_eval
import tnt_register as oracle
import mvs_b200
from mvs_b200 import _lib, tanks

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytest.importorskip("scipy.spatial")
OTHER = dict(max_iteration=20, relative_rmse=1e-6)


def _g(a, dtype=np.float32):
    return torch.from_numpy(np.ascontiguousarray(a, dtype)).to(DEV)


def test_index_search_against_ckdtree_and_ties():
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(0)
    t = rng.uniform(-1, 1, (60000, 3)).astype(np.float32)
    t[:, 2] *= 0.1
    t[1000:1100] = t[50000:50100]                               # exact duplicates: the smaller row wins
    q = rng.uniform(-1.2, 1.2, (40000, 3)).astype(np.float32)
    q[:, 2] *= 0.1
    q[:100] = t[50000:50100]                                    # queries on the duplicates: distance 0, tied
    cap = 0.05
    d, i = mvs_b200.nearest_neighbour(_g(q), _g(t), cap)
    d, i = d.cpu().numpy(), i.cpu().numpy()
    assert i.dtype == np.int64
    dd, ii = cKDTree(t.astype(np.float64)).query(q.astype(np.float64), k=2)
    has = dd[:, 0] < cap
    sure = np.abs(dd[:, 0] - cap) > 1e-5 * cap
    assert np.array_equal(np.isfinite(d)[sure], has[sure]) and np.array_equal(i[sure] >= 0, has[sure])
    assert (i[~np.isfinite(d)] == -1).all()
    ok = has & np.isfinite(d)
    assert (np.abs(d[ok] - dd[ok, 0]) <= 1e-6 * dd[ok, 0]).all()
    gap = (dd[:, 1] - dd[:, 0]) / np.maximum(dd[:, 1], 1e-30)
    clear = ok & (gap >= 1e-4)
    print("queries with a clear nearest point", int(clear.sum()), "of", len(q))
    assert clear.sum() > 5000
    assert np.array_equal(i[clear], ii[clear, 0])
    assert np.array_equal(i[:100], np.arange(1000, 1100)) and (d[:100] == 0).all()
    d2, _ = mvs_b200.nearest_neighbour(_g(q), _g(t), cap)
    assert np.array_equal(mvs_b200.nearest_distance(_g(q), _g(t), cap).cpu().numpy(), d)      # same search, same distances
    assert np.array_equal(d2.cpu().numpy(), d)


def _sums_gpu(s, idx, t):
    n = s.shape[0]
    partial = torch.empty(_lib.PC_ICP_BLOCKS * 10, dtype=torch.float64, device=DEV)
    ticket = torch.zeros(2, dtype=torch.int32, device=DEV)
    out = torch.empty(_lib.PC_ICP_SUMS, dtype=torch.float64, device=DEV)
    _lib.call("mvsb200_pc_icp_sums", s.data_ptr(), idx.data_ptr(), n, t.data_ptr(), partial.data_ptr(), ticket.data_ptr(),
              out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert int(ticket.abs().sum()) == 0
    return out.cpu().numpy()


@pytest.mark.parametrize("n", [1, 1000, 400_000])
def test_icp_sums_against_numpy_and_deterministic(n):
    rng = np.random.default_rng(n)
    t = rng.normal(size=(max(n // 2, 1), 3)) * [5.0, 3.0, 1.0] + [100.0, -40.0, 7.0]
    s = rng.normal(size=(n, 3)) * [5.0, 3.0, 1.0] + [100.5, -40.0, 7.0]
    idx = rng.integers(0, len(t), n).astype(np.int32)
    idx[rng.random(n) < 0.3] = -1
    if n == 1:
        idx[0] = 0
    got = _sums_gpu(_g(s, np.float64), _g(idx, np.int32), _g(t, np.float64))
    sel = idx >= 0
    ss, tt = s[sel], t[idx[sel]]
    mu_s, mu_t = ss.mean(0), tt.mean(0)
    a, b = ss - mu_s, tt - mu_t
    want = np.concatenate([[sel.sum(), ((ss - tt) ** 2).sum()], ss.sum(0), tt.sum(0), (b.T @ a).reshape(9), [(a * a).sum()]])
    scale = np.maximum(np.abs(want), np.concatenate([[1, 1], np.abs(want[2:8]), [np.abs(want[8:17]).max()] * 9, [want[17]]]))
    assert (np.abs(got - want) <= 1e-12 * scale + 1e-300).all(), (got - want) / scale
    again = _sums_gpu(_g(s, np.float64), _g(idx, np.int32), _g(t, np.float64))
    assert got.tobytes() == again.tobytes()


def test_icp_sums_without_correspondences():
    got = _sums_gpu(_g(np.ones((500, 3)), np.float64), _g(np.full(500, -1), np.int32), _g(np.ones((3, 3)), np.float64))
    assert (got == 0).all()


def test_transform64_is_bit_exact():
    rng = np.random.default_rng(3)
    p = rng.normal(size=(100_000, 3)) * 50 + [1e3, -2e2, 3.0]
    U = oracle.similarity(oracle.rotation([0.1, 0.7, -0.2], 13.0), 1.013, [0.25, -3.5, 1e-3])
    x = _g(p, np.float64)
    x32 = torch.empty(x.shape, dtype=torch.float32, device=DEV)
    _lib.call("mvsb200_pc_transform64", x.data_ptr(), x.shape[0], np.ascontiguousarray(U[:3].reshape(12)).ctypes.data_as(_lib._c.c_void_p),
              x32.data_ptr(), torch.cuda.current_stream().cuda_stream)
    want = tnt_eval.transform(p, U)
    assert x.cpu().numpy().tobytes() == want.tobytes()
    assert x32.cpu().numpy().tobytes() == want.astype(np.float32).tobytes()


@pytest.mark.parametrize("criteria", [{}, OTHER])
def test_one_icp_run_equals_the_oracle(criteria):
    s, t = oracle.lattice_icp_scene()
    want = oracle.icp(s, t, 0.3, **criteria)
    assert want["min_margin"] >= 1e-4
    got = mvs_b200.icp_point_to_point(_g(s, np.float64), _g(t, np.float64), 0.3, return_history=True, **criteria)
    assert got["iterations"] == want["iterations"]
    assert [h["correspondences"] for h in got["history"]] == [h["correspondences"] for h in want["history"]]
    for k in ("fitness", "inlier_rmse"):
        assert abs(got[k] - want[k]) <= 1e-9 * abs(want[k]), k
    assert np.abs(got["transformation"] - want["transformation"]).max() <= 1e-9 * np.abs(want["transformation"]).max()


@pytest.fixture(scope="module")
def walls():
    return oracle.walls_scene()


@pytest.mark.parametrize("criteria", [{}, OTHER])
def test_three_stages_against_the_oracle(walls, criteria):
    x, g, crop, T_true, T0, tau = walls
    want = oracle.register(x, g, crop, T0, tau, **criteria)
    got = mvs_b200.register_tanks_and_temples(_g(x), _g(g), tanks._crop_volume(*crop), T0, tau, **criteria)
    extent = float(np.ptp(g, 0).max())
    dR = np.abs(got["transformation"][:3, :3] - want["transformation"][:3, :3]).max()
    dt = np.abs(got["transformation"][:3, 3] - want["transformation"][:3, 3]).max()
    counts = [(a["correspondences"], b["correspondences"]) for a, b in zip(got["stages"], want["stages"])]
    print(criteria, "dR", dR, "dt / extent", dt / extent, "counts", counts, "iterations",
          [(a["iterations"], b["iterations"]) for a, b in zip(got["stages"], want["stages"])], "oracle margin", want["min_margin"])
    for a, b in zip(got["stages"], want["stages"]):
        assert a["n_down"] == b["n_down"] and a["m_down"] == b["m_down"]
    assert all(abs(a - b) <= 1e-3 * b for a, b in counts)
    assert dR <= 1e-6 and dt <= 1e-6 * extent
    assert got["transformation"][3].tolist() == [0.0, 0.0, 0.0, 1.0]
    assert np.array_equal(got["init"], T0)


# three rigid placements X -> Q (X - centre) + o of one fused disk, on planes whose normals are 70-120 degrees apart: one plane
# leaves ICP free to slide, turn and scale in it, which moves the voxel-quantised F-score by about 0.01 either way; three pin all
# seven degrees of freedom, so the exact alignment is the registration's optimum
PLACEMENTS = (([1.0, 0.0, 0.0], 0.0, [0.0, 0.0, 0.0]), ([1.0, 0.2, 0.0], 80.0, [9.0, 1.0, 2.0]), ([0.1, 1.0, 0.3], -75.0, [2.0, 9.0, -1.5]))


def _place(x, centre):
    return np.concatenate([(x - centre) @ (oracle.rotation(ax, deg) if deg else np.eye(3)).T + np.asarray(o) for ax, deg, o in PLACEMENTS])


def test_end_to_end_fused_disks():
    s = fusion_oracle.analytic_scene(6, 48, 64, normal="sweep", seed=0)
    depth = torch.from_numpy(s["depth"].astype(np.float32))[:, None].to(DEV)
    src = [[j for j in range(6) if j != i] for i in range(6)]
    xyz, _, _ = mvs_b200.fuse_depth_maps(depth, torch.ones_like(depth), torch.rand(6, 3, 48, 64, device=DEV), s["K"], s["R"], s["T"],
                                         src, conf_min=0.0, reproj_px=1e3, rel_depth=1.0, min_views=1)
    r, n0, centre = s["radius"], s["n0"], s["centre"]
    a0 = np.cross(n0, [0.0, 1.0, 0.0])
    a0 /= np.linalg.norm(a0)
    b0 = np.cross(n0, a0)
    rec = _place(xyz.double().cpu().numpy(), centre).astype(np.float32)
    # the ground truth: the same disk on a lattice of 0.01 r in its plane, in the same three placements, mapped by A
    step = 0.01 * r
    k = np.arange(-int(r / step) - 1, int(r / step) + 2) * step
    u, v = (a.ravel() for a in np.meshgrid(k, k, indexing="ij"))
    on = u * u + v * v <= r * r
    A = oracle.similarity(oracle.rotation([0.3, 1.0, -0.5], 40.0), 1.7, [3.0, -1.0, 2.0])
    gt = tnt_eval.transform(_place(centre + u[on, None] * a0 + v[on, None] * b0, centre), A).astype(np.float32)
    lo, hi = gt.min(0) - 1, gt.max(0) + 1
    crop = tanks._crop_volume("y", lo[1], hi[1], [[lo[0], 0, lo[2]], [hi[0], 0, lo[2]], [hi[0], 0, hi[2]], [lo[0], 0, hi[2]]])
    tau = 0.05 * 1.7 * r / 4                               # 0.085: about 6 lattice steps of the GT
    # T0: the exact alignment perturbed about the reconstruction's centroid by 3 degrees, scale 1.02 and 3 tau
    c = tnt_eval.transform(rec.mean(0, dtype=np.float64)[None], A)[0]
    P = oracle.similarity(oracle.rotation(a0 + 0.3 * b0, 3.0), 1.02, np.zeros(3))
    P[:3, 3] = c - P[:3, :3] @ c + 3 * tau * (A[:3, :3] @ n0) / 1.7
    T0 = P @ A
    xg, gg = _g(rec), _g(gt)
    f_exact = mvs_b200.evaluate_tanks_and_temples(xg, gg, crop, A, tau)["fscore"]
    f_init = mvs_b200.evaluate_tanks_and_temples(xg, gg, crop, T0, tau)["fscore"]
    reg = mvs_b200.register_tanks_and_temples(xg, gg, crop, T0, tau)
    f_reg = mvs_b200.evaluate_tanks_and_temples(xg, gg, crop, reg["transformation"], tau)["fscore"]
    print("fscore exact", f_exact, "init", f_init, "registered", f_reg,
          [(st["iterations"], st["correspondences"], st["n_down"], st["m_down"]) for st in reg["stages"]])
    assert abs(f_reg - f_exact) <= 0.01 and f_reg > f_init + 0.1
    # from the exact alignment, registration moves the reconstruction by less than tau / 10
    still = mvs_b200.register_tanks_and_temples(xg, gg, crop, A, tau)
    p = rec.astype(np.float64)
    move = np.linalg.norm(tnt_eval.transform(p, still["transformation"]) - tnt_eval.transform(p, A), axis=1).max()
    print("move from the exact alignment", move, "tau", tau)
    assert move < tau / 10


def test_empty_crops_and_refusals():
    rng = np.random.default_rng(5)
    x = _g(rng.uniform(0, 1, (2000, 3)))
    far = tanks._crop_volume("z", -1.0, 1.0, [[10, 10, 0], [11, 10, 0], [11, 11, 0]])
    T0 = oracle.similarity(np.eye(3), 1.1, [0.1, 0.0, 0.0])
    r = mvs_b200.register_tanks_and_temples(x, x, far, T0, 0.05)
    assert np.array_equal(r["transformation"], T0)
    assert all(st["fitness"] == 0 and st["n_down"] == 0 and st["m_down"] == 0 and st["iterations"] == 1 for st in r["stages"])
    out = mvs_b200.icp_point_to_point(torch.empty((0, 3), dtype=torch.float64, device=DEV), x.double(), 0.1)
    assert out["fitness"] == 0 and out["inlier_rmse"] == 0 and np.array_equal(out["transformation"], np.eye(4))
    box = tanks._crop_volume("z", -1.0, 2.0, [[-1, -1, 0], [2, -1, 0], [2, 2, 0], [-1, 2, 0]])
    bad = np.eye(4)
    bad[3, 0] = 1e-9
    with pytest.raises(mvs_b200.MvsB200Error, match="affine"):
        mvs_b200.register_tanks_and_temples(x, x, box, bad, 0.05)
    for tau in (0.0, -1.0, float("nan")):
        with pytest.raises(mvs_b200.MvsB200Error, match="tau"):
            mvs_b200.register_tanks_and_temples(x, x, box, np.eye(4), tau)
    y = x.clone()
    y[3, 1] = float("inf")
    with pytest.raises(mvs_b200.MvsB200Error, match="finite"):
        mvs_b200.register_tanks_and_temples(y, x, box, np.eye(4), 0.05)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.register_tanks_and_temples(x.cpu(), x, box, np.eye(4), 0.05)
    with pytest.raises(mvs_b200.MvsB200Error, match="fp64"):
        mvs_b200.icp_point_to_point(x, x.double(), 0.1)
    u = mvs_b200.uniform_down_sample(x.double(), 3)
    assert torch.equal(u, x.double()[::3])


def test_eval_tnt_tool_register(tmp_path):
    x, g, crop, T_true, T0, tau = oracle.walls_scene(n_gt=20000, n_rec=12000)
    d = tmp_path / "Synth"
    d.mkdir()
    mvs_b200.write_ply(str(d / "Synth.ply"), g)
    axis, amin, amax, poly = crop
    with open(d / "Synth.json", "w") as f:
        json.dump({"class_name": "SelectionPolygonVolume", "orthogonal_axis": axis, "axis_min": amin, "axis_max": amax,
                   "bounding_polygon": poly.tolist(), "version_major": 1, "version_minor": 0}, f)
    np.savetxt(str(d / "Synth_trans.txt"), T0, fmt="%.17g")
    ply = str(tmp_path / "rec.ply")
    mvs_b200.write_ply(ply, x)
    out = str(tmp_path / "r.json")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "eval_tnt.py"), "--ply", ply, "--tnt", str(tmp_path), "--scene",
                        "Synth", "--tau", str(tau), "--register", "--out", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = json.load(open(out))
    reg = mvs_b200.register_tanks_and_temples(_g(x), _g(g), tanks._crop_volume(*crop), T0, tau)
    assert np.array_equal(np.array(got["registration"]["transformation"]), reg["transformation"])
    assert len(got["registration"]["stages"]) == 3
    want = mvs_b200.evaluate_tanks_and_temples(_g(x), _g(g), tanks._crop_volume(*crop), reg["transformation"], tau)
    assert got["fscore"] == want["fscore"]
    plain = mvs_b200.evaluate_tanks_and_temples(_g(x), _g(g), tanks._crop_volume(*crop), T0, tau)
    assert got["fscore"] > plain["fscore"]
