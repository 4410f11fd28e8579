"""GPU parity of the tensor-core (tcgen05 / TMEM / TMA) hitting-time sweep behind the dense continuous diameter
(colosseum/hardness/measures/diameter.py:76-106; SURVEY App. B.5).  The oracle is the fp64 restatement of the
synchronous sweep  E'[k,s] = (s == target_k) ? 0 : min_a(1 + sum_j T[s,a,j] E[k,j])  (numpy here, oracle/ for the
fixed point).  Bar: 1e-4 relative in f32 mode (BASELINE.json north_star) -- the 3 x TF32 split lands near 1e-6."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def sweeps_f64(T, targets, n):
    S, A, _ = T.shape
    K = len(targets)
    Td = T.astype(np.float64).reshape(S * A, S)
    E = np.zeros((K, S))
    for _ in range(n):
        C_ = (Td @ E.T).reshape(S, A, K)  # [(s,a), k]
        En = (1.0 + C_).min(1).T          # [k, s]
        En[np.arange(K), targets] = 0.0
        E = En
    return E


def umma_sweeps(T, targets, n):
    import torch

    from colosseum_b200 import _cabi

    S, A, _ = T.shape
    K = len(targets)
    Td = torch.from_numpy(np.ascontiguousarray(T, np.float32)).cuda()
    tg = torch.from_numpy(np.ascontiguousarray(targets, np.int32)).cuda()
    E = torch.full((K, S), 7.0, dtype=torch.float32, device="cuda")  # zero_start must overwrite this
    W = torch.empty_like(E)
    rc = _cabi.lib().colo_hitting_umma_sweeps_f32(_cabi.ptr(Td), _cabi.ptr(tg), K, S, A, n, 1, _cabi.ptr(E), _cabi.ptr(W),
                                                  _cabi.current_stream())
    _cabi.check(rc, "colo_hitting_umma_sweeps_f32")
    torch.cuda.synchronize()
    return E.cpu().numpy()


def dirichlet_T(S, A, alpha, seed):
    rs = np.random.RandomState(seed)
    T = rs.dirichlet(np.ones(S) * alpha, size=(S, A)).astype(np.float32)
    return T


@pytest.mark.parametrize("S,A,K,n", [(256, 2, 256, 6), (300, 5, 200, 6), (129, 1, 64, 4), (640, 8, 333, 5),
                                     (512, 4, 512, 12)])
def test_umma_sweeps_match_fp64(S, A, K, n):
    """fixed numbers of synchronous sweeps, ragged S / K (padding rows and columns), BN = 128 (A <= 4) and 64 (A > 4)"""
    T = dirichlet_T(S, A, 0.3, S + A)
    targets = np.random.RandomState(1).permutation(S)[:K].astype(np.int32)
    ref = sweeps_f64(T, targets, n)
    got = umma_sweeps(T, targets, n)
    err = np.abs(got - ref).max() / np.abs(ref).max()
    assert err < 2e-6, err
    assert (got[np.arange(K), targets] == 0).all()


def test_umma_rooms_instance_948():
    """the largest benchmark instance (MiniGridRooms, S = 948, A = 3, all 948 targets): 12 sweeps vs fp64"""
    from colosseum_b200.suite import load_suite

    suite = load_suite(os.path.join(GOLDEN, "c3_suite.npz"))
    inst = max((i for i in suite if not i.episodic), key=lambda i: i.S)
    T = inst.tables.T
    S = inst.S
    assert S >= 900
    targets = np.arange(S, dtype=np.int32)
    ref = sweeps_f64(T, targets, 12)
    got = umma_sweeps(T, targets, 12)
    assert np.abs(got - ref).max() / np.abs(ref).max() < 2e-6


def test_umma_large_dense_2048():
    """S = 2,048, A = 8, K = 2,048 synthetic dense MDP: 3 sweeps vs fp64 (137 GFLOP per sweep)"""
    import torch

    S, A = 2048, 8
    T = dirichlet_T(S, A, 0.05, 5)
    targets = np.arange(S, dtype=np.int32)
    # the fp64 restatement of sweeps_f64, evaluated by cuBLAS DGEMM (137 GFLOP per sweep: minutes in numpy)
    Td = torch.from_numpy(T).cuda().double().reshape(S * A, S)
    E = torch.zeros((S, S), dtype=torch.float64, device="cuda")
    idx = torch.arange(S, device="cuda")
    for _ in range(3):
        E = (1.0 + (Td @ E.T).reshape(S, A, S)).min(1).values.T.contiguous()
        E[idx, idx] = 0.0
    ref = E.cpu().numpy()
    got = umma_sweeps(T, targets, 3)
    assert np.abs(got - ref).max() / np.abs(ref).max() < 2e-6


def test_diameter_dense_through_umma(monkeypatch):
    """get_diameter (f32 mode) on a dense synthetic MDP takes the tensor-core path, one hitting_umma launch per sweep
    and no other solver path, and meets the f32 bar against the fp64 fixed-point oracle.  (The forced SIMT GEMM is
    compared with this path in test_gpu_solver_paths.py: COLO_DIAM_PATH is read once per process.)"""
    import colosseum_b200.hardness as hd

    from colosseum_b200 import _cabi

    def paths():
        return np.array([_cabi.lib().colo_solver_path_launches(k) for k in range(len(_cabi.PATH_KINDS))], np.int64)

    T = dirichlet_T(384, 8, 0.02, 11)  # 4.7 MB: too large for the on-chip resident solver, dense rows
    # fp64 fixed point of the multi-target recurrence (SURVEY App. B.5), all targets side by side
    S, A = 384, 8
    Td, E, idx = T.astype(np.float64).reshape(S * A, S), np.zeros((S, S)), np.arange(S)
    for _ in range(20000):
        En = (1.0 + (Td @ E.T).reshape(S, A, S)).min(1).T
        En[idx, idx] = 0.0
        done = np.abs(En - E).max() < 1e-9
        E = En
        if done:
            break
    d_ref = float(E.max())
    assert abs(orc.diameter_continuous_f64(T, targets=np.arange(4, dtype=np.int32)) - E[:4].max()) < 1e-6  # same recurrence
    n0 = _cabi.lib().colo_launch_count()
    p0 = paths()
    d, sweeps = hd.get_diameter(T, False, precision="f32", epsilon=2e-5, return_sweeps=True)
    assert abs(d - d_ref) < 1e-4 * d_ref, (d, d_ref)
    assert sweeps > 3 and _cabi.lib().colo_launch_count() - n0 >= sweeps
    ran = {_cabi.PATH_KINDS[k]: int(v) for k, v in enumerate(paths() - p0) if v}
    assert ran == {"HIT_UMMA": sweeps}, ran


@pytest.mark.parametrize("cluster", ["0", "1"])
@pytest.mark.parametrize("bn", ["64", "128"])
def test_umma_cluster_multicast_is_identical(monkeypatch, cluster, bn):
    """2 x 2 thread-block clusters with multicast TMA (each CTA loads half of the T tile and half of the E tile for
    the pair that shares it) against one CTA per tile: the same sweeps bit for bit, on a grid with odd tile counts
    (padding to whole clusters) and both tile widths"""
    monkeypatch.setenv("COLO_UMMA_BN", bn)
    S, A, K = 400, 3, 330
    T = dirichlet_T(S, A, 0.2, 9)
    targets = np.random.RandomState(2).permutation(S)[:K].astype(np.int32)
    monkeypatch.setenv("COLO_UMMA_CLUSTER", "0")
    base = umma_sweeps(T, targets, 7)
    monkeypatch.setenv("COLO_UMMA_CLUSTER", cluster)
    got = umma_sweeps(T, targets, 7)
    assert np.array_equal(got, base)
    ref = sweeps_f64(T, targets, 7)
    assert np.abs(got - ref).max() / np.abs(ref).max() < 2e-6
