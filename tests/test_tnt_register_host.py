"""The Tanks and Temples registration without a GPU: the fp64 oracle (oracle/tnt_register.py) recovers planted similarities, each of
its mutation switches changes the outcome, the library's host-side Umeyama solve and uniform rate agree with it, and the C ABI and
the Python functions refuse what they should before touching a device."""
import ctypes
import math

import numpy as np
import pytest
import torch

import tnt_register as oracle
import mvs_b200
from mvs_b200 import _lib, registration

pytest.importorskip("scipy.spatial")
OTHER = dict(max_iteration=20, relative_rmse=1e-6)          # the other reading of ICPConvergenceCriteria(1e-6, 20)


def _sums(s, t):
    """pc_icp_sums' 18 values in numpy fp64."""
    mu_s, mu_t = s.mean(0), t.mean(0)
    a, b = s - mu_s, t - mu_t
    return np.concatenate([[len(s), ((s - t) ** 2).sum()], s.sum(0), t.sum(0), (b.T @ a).reshape(9), [(a * a).sum()]])


def test_umeyama_recovers_a_planted_similarity():
    rng = np.random.default_rng(0)
    s = rng.normal(size=(500, 3))
    A = oracle.similarity(oracle.rotation([0.3, -1.0, 0.4], 37.0), 1.7, [0.5, -2.0, 3.0])
    t = s @ A[:3, :3].T + A[:3, 3]
    for U in (oracle.umeyama(s, t), registration.umeyama(_sums(s, t))):
        assert np.abs(U - A).max() <= 1e-12 * np.abs(A).max()
    rigid = oracle.similarity(A[:3, :3] / 1.7, 1.0, A[:3, 3])
    t = s @ rigid[:3, :3].T + rigid[:3, 3]
    assert np.abs(oracle.umeyama(s, t, with_scaling=False) - rigid).max() <= 1e-12 * 3
    assert np.abs(registration.umeyama(_sums(s, t), with_scaling=False) - rigid).max() <= 1e-12 * 3


def test_umeyama_takes_the_reflection_branch():
    rng = np.random.default_rng(1)
    s = rng.normal(size=(300, 3)) * [3.0, 2.0, 0.5]
    t = s * [1.0, 1.0, -1.0]                                   # a mirror image: the best fit is a rotation, not the reflection
    sigma = (t - t.mean(0)).T @ (s - s.mean(0)) / len(s)
    U, _, Vt = np.linalg.svd(sigma)
    assert np.linalg.det(U) * np.linalg.det(Vt) < 0
    for M in (oracle.umeyama(s, t), registration.umeyama(_sums(s, t))):
        assert np.linalg.det(M[:3, :3]) > 0
        R = M[:3, :3] / np.cbrt(np.linalg.det(M[:3, :3]))
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-12)
    assert np.abs(oracle.umeyama(s, t) - registration.umeyama(_sums(s, t))).max() < 1e-12


def test_umeyama_degenerate_cases_are_the_identity():
    assert np.array_equal(registration.umeyama(np.zeros(18)), np.eye(4))
    assert np.array_equal(oracle.umeyama(np.zeros((0, 3)), np.zeros((0, 3))), np.eye(4))
    one = np.ones((4, 3))
    assert np.array_equal(oracle.umeyama(one, one + 1), np.eye(4))
    assert np.array_equal(registration.umeyama(_sums(one, one + 1)), np.eye(4))


@pytest.fixture(scope="module")
def walls():
    return oracle.walls_scene()


def _err(r, T_true):
    return oracle.similarity_error(r["transformation"], T_true)


def test_three_stages_recover_a_planted_perturbation(walls):
    x, g, crop, T_true, T0, tau = walls
    ang0, sc0, tr0 = oracle.similarity_error(T0, T_true)
    assert ang0 > 0.05 and abs(sc0 - 0.02) < 1e-12 and tr0 > 3 * tau
    # the toolbox's criteria: stages 1 and 2 keep every point within 80 tau and 20 tau, so |delta fitness| = 0 after one update and
    # each stops after one iteration; stage 3 stops once its correspondence count repeats.  Recovery is therefore partial.
    r = oracle.register(x, g, crop, T0, tau)
    ang, sc, tr = _err(r, T_true)
    print("toolbox reading", [(s["iterations"], s["correspondences"]) for s in r["stages"]], ang, sc, tr)
    assert [s["iterations"] for s in r["stages"][:2]] == [1, 1] and r["stages"][2]["iterations"] > 1
    assert ang < ang0 / 5 and sc < 0.6 * sc0 and tr < tr0 / 5
    # the other reading (20 iterations, relative_rmse 1e-6) runs each stage to convergence and meets the proposed bounds
    r = oracle.register(x, g, crop, T0, tau, **OTHER)
    ang, sc, tr = _err(r, T_true)
    print("other reading", [(s["iterations"], s["correspondences"]) for s in r["stages"]], ang, sc, tr)
    assert ang <= 1e-3 and sc <= 1e-3 and tr <= tau / 4


def test_mutations_change_the_outcome(walls):
    x, g, crop, T_true, T0, tau = walls
    base = oracle.register(x, g, crop, T0, tau, **OTHER)
    ang, sc, tr = _err(base, T_true)
    noscale = _err(oracle.register(x, g, crop, T0, tau, with_scaling=False, **OTHER), T_true)
    assert abs(noscale[1] - 0.02) < 1e-9                                   # a rigid update never touches the planted 2 %
    for kw in (dict(compose="init_first"), dict(transform_gt=True)):
        e = _err(oracle.register(x, g, crop, T0, tau, **kw, **OTHER), T_true)
        print(kw, e)
        assert e[0] > 1e-3 or e[1] > 1e-3 or e[2] > tau / 4, kw         # recovery fails
    toolbox = oracle.register(x, g, crop, T0, tau)
    assert [s["iterations"] for s in toolbox["stages"]] != [s["iterations"] for s in base["stages"]]


def test_criteria_readings_give_different_iteration_counts():
    s, t = oracle.lattice_icp_scene()
    a = oracle.icp(s, t, 0.3)
    b = oracle.icp(s, t, 0.3, relative_rmse=1e-6, max_iteration=20)
    assert a["iterations"] == 2 and b["iterations"] == 3


@pytest.mark.parametrize("rounding, n, k", [("half_up", 100, 3), ("ceil", 100, 3), ("floor", 140, 3)])
def test_uniform_rate_rounding(rounding, n, k):
    want = {100: 2, 140: 4}[n]                          # 2.5 -> 2 and 3.5 -> 4: Python's round, halves to even
    assert oracle.uniform_rate(n, 40) == registration.uniform_rate(n, 40) == want
    assert oracle.uniform_rate(n, 40, rounding) == k != want


def test_uniform_rate_matches_the_oracle():
    for n in [0, 1, 39, 40, 41, 59, 60, 61, 99, 100, 101, 139, 140, 141, 10 ** 6]:
        assert registration.uniform_rate(n, 40) == oracle.uniform_rate(n, 40)
    assert registration.uniform_rate(6_000_000) == 2 and registration.uniform_rate(10_000_000) == 2
    assert registration.uniform_rate(14_000_000) == 4


def test_c_abi_refusals():
    lib = mvs_b200.load_library()
    assert lib.mvsb200_pc_icp_sums(None, None, 1, None, None, None, None, None) == -1
    assert b"null pointer" in lib.mvsb200_last_error()
    a = (ctypes.c_double * 12)(*([1.0] * 11 + [math.nan]))
    buf = (ctypes.c_double * 3)()
    f32 = (ctypes.c_float * 3)()
    assert lib.mvsb200_pc_transform64(buf, 1, a, f32, None) == -1
    assert b"finite" in lib.mvsb200_last_error()
    assert lib.mvsb200_pc_nearest_index(None, 1, None, None, None, 0.0, 0.0, 0.0, 1.0, 1, 1, 1, 0.0, 1.0, None, None, None) == -1
    assert _lib.PC_ICP_SUMS == 18 and _lib.PC_ICP_BLOCKS == 1024


def test_cpu_tensors_are_refused():
    x = torch.rand(10, 3)
    crop = mvs_b200.CropVolume("Z", -1.0, 1.0, np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float64))
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.register_tanks_and_temples(x, x, crop, np.eye(4), 0.1)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.icp_point_to_point(x.double(), x.double(), 0.1)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.nearest_neighbour(x, x, 0.1)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.uniform_down_sample(x.double(), 2)
