"""GPU parity of every Bellman-solver path against the fp64 oracle, at the shapes that select it.

The solvers behind VI / PE, the episodic backward induction, the diameter, the value norm and the in-place order each
pick one of several kernels from the tensor's shape and sparsity (DESIGN 4.8):

  discounted VI / PE   sparse_vi_kernel (compressed rows, S <= 2048) -> sparse_sweep_kernel -> resident_solve_kernel
                       -> backup_kernel, one warp per state or one CTA per state (B*S < 64*SMs and S*A >= 4096)
  episodic VI / PE     episodic_batched_kernel (B >= 16, no bound) -> resident (episodic_H) -> backup_kernel per layer
  continuous diameter  sparse_hitting_kernel<NT> -> resident (NV = 4) -> hitting_umma (f32) / hitting_gemm
                       (K*S >= 128^2) -> backup_kernel with pinned targets
  episodic diameter    sparse_episodic_kernel -> hitting_gemm (K*S >= 64^2) -> backup_kernel per layer
  value norm           two backup_kernel passes, the second with one V per action
  in-place order       gs_sparse_kernel<ONEPASS> -> gs_solve_tma_kernel -> gs_solve_kernel

Every case runs one path on a synthetic MDP, compares it with the plain fp64 oracle (oracle/oracle.py) and asserts
through `colo_solver_path_launches` which path ran and how often.  Bars: 1e-6 relative in f64 mode and 1e-4 in f32 at
the fixed point, rounding level for fixed sweep counts, the stopping tolerance (and at most one sweep apart) for the
in-place order.  The switches that force a path (COLO_NO_SPARSE, COLO_NO_RESIDENT, COLO_DIAM_PATH, COLO_SPARSE_NT,
COLO_GS_NO_TMA) are read once per process, so forced cases run in one child process per setting; the oracle runs
here.  The boundaries of the selection rules are pinned by the counter alone, and the last test checks that the file
reached every path.
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from colosseum_b200._cabi import PATH_KINDS
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = {name: i for i, name in enumerate(PATH_KINDS)}  # COLO_PATH_* of include/colosseum_b200.h
RTOL64, RTOL32 = 1e-6, 1e-4
GAM = float(np.float32(0.9))
TALLY = np.zeros(len(PATH_KINDS), np.int64)  # launches per path over every case of this file (parent and children)


def path_counts():
    from colosseum_b200 import _cabi

    return np.array([_cabi.lib().colo_solver_path_launches(k) for k in range(len(PATH_KINDS))], np.int64)


def sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def resident_fits(S, A, NV, f64):
    from colosseum_b200 import _cabi

    return _cabi.lib().colo_resident_fits(S, A, NV, int(f64), None) == 1


# ------------------------------------------------------------------------------------------------------------ MDPs
def sparse_T(S, A, k, seed):
    """rows of at most k non-zeros: 0.6 on a steering successor (s + 1 for action 0, so every state reaches every
    other; a random state for the others), 0.4 spread over k - 1 random states"""
    rs = np.random.RandomState(seed)
    T = np.zeros((S, A, S), np.float32)
    I, J = np.meshgrid(np.arange(S), np.arange(A), indexing="ij")
    main = rs.randint(S, size=(S, A))
    main[:, 0] = (np.arange(S) + 1) % S
    if k == 1:
        T[I, J, main] = 1.0
        return T
    other = rs.randint(S, size=(S, A, k - 1))
    w = rs.dirichlet(np.ones(k - 1), size=(S, A)).astype(np.float32) * 0.4
    T[I, J, main] += 0.6
    for j in range(k - 1):
        T[I, J, other[..., j]] += w[..., j]
    return T / T.sum(-1, keepdims=True)


def dense_T(S, A, seed, noise=0.05, rare0=False):
    """every entry positive: `noise` spread over all states plus a steering successor as in sparse_T, so hitting times
    stay short and the iterations converge in tens of sweeps.  rare0: state 0 is reached only through the noise, with
    1e-3 of its share (hitting times to 0 in the hundreds of thousands)"""
    rs = np.random.RandomState(seed)
    W = rs.uniform(0.5, 1.5, size=(S, A, S)).astype(np.float32)
    if rare0:
        W[:, :, 0] *= 1e-3
    T = noise * W / W.sum(-1, keepdims=True)
    I, J = np.meshgrid(np.arange(S), np.arange(A), indexing="ij")
    main = rs.randint(S, size=(S, A))
    main[:, 0] = (np.arange(S) + 1) % S
    if rare0:
        main[main == 0] = 1
    T[I, J, main] += 1.0 - noise
    return (T / T.sum(-1, keepdims=True)).astype(np.float32)


def make_T(c, seed):
    return sparse_T(c["S"], c["A"], c["k"], seed) if c.get("k") else dense_T(c["S"], c["A"], seed,
                                                                              rare0=c.get("rare0", False))


def make_mdp(c):
    """T [B,S,A,S], R [B,S,A] (instance b scaled by rscale[b]: instances converge at different sweeps), pi"""
    B = c.get("B", 1)
    S, A = c["S"], c["A"]
    Ts, Rs, pis = [], [], []
    for b in range(B):
        rs = np.random.RandomState(c["seed"] + 1000 * b + 1)
        Ts.append(make_T(c, c["seed"] + b))
        Rs.append((rs.uniform(0, 1, (S, A)) * c.get("rscale", [1.0] * B)[b]).astype(np.float32))
        if c.get("H"):
            pis.append(rs.dirichlet(np.ones(A), size=(c["H"], S)).astype(np.float32))
        else:
            pis.append(rs.dirichlet(np.ones(A), size=S).astype(np.float32))
    return np.stack(Ts), np.stack(Rs), np.stack(pis)


def make_T_epi(c):
    """T_epi [H,S,A,S] of an episodic MDP that may start anywhere (every target is reached in every horizon)"""
    T = make_T(c, c["seed"])
    R = np.zeros(T.shape[:2], np.float32)
    w = np.random.RandomState(c["seed"] + 3).uniform(0.5, 1.5, c["S"])
    T_epi, _, _ = orc.episodic_T(c["H"], T, R, np.arange(c["S"]), w / w.sum())
    return T_epi


def v_of(c):
    return np.random.RandomState(c["seed"] + 7).uniform(-3, 8, c["S"]).astype(np.float32)


# ------------------------------------------------------------------------------------------------------ the GPU side
def run_case(c):
    """runs one case on the GPU; returns its outputs and the launches per solver path it caused"""
    import colosseum_b200.dynamic_programming as dp
    import colosseum_b200.hardness as hd

    prec = c.get("prec", "f64")
    out = {}
    n0 = path_counts()
    op = c["op"]
    if op in ("disc", "gs"):
        T, R, pi = make_mdp(c)
        if op == "gs":
            res = dp._solve_discounted(T, R, pi if c.get("pe") else None, GAM, 1e-3, None, "f32",
                                       sweep_order="gauss_seidel")
        else:
            res = dp._solve_discounted(T, R, pi if c.get("pe") else None, GAM, 1e-10 if prec == "f64" else 1e-5,
                                       None, prec)
        out["Q"], out["V"] = res
        out["iters"] = np.array(dp.last_iterations())
    elif op == "backup":
        T, R, pi = make_mdp(c)
        fold = {"max": orc.FOLD_MAX, "pi": orc.FOLD_PI, "min": orc.FOLD_MIN}[c["fold"]]
        out["Q"], out["V"], out["res"] = dp.bellman_backup(T[0], R[0], v_of(c), GAM, pi[0] if c["fold"] == "pi" else None,
                                                           fold, precision=prec, return_residual=True)
    elif op == "epi":
        T, R, pi = make_mdp(c)
        res = dp._episodic(c["H"], T, R, pi if c.get("pe") else None, c.get("max_value"), prec)
        out["none"] = np.array(res is None)
        if res is not None:
            out["Q"], out["V"] = res
    elif op in ("diam", "epidiam"):
        T = make_T_epi(c) if op == "epidiam" else make_T(c, c["seed"])
        # f32: a few ulps of the largest hitting time (the residual of an f32 iterate does not fall below that)
        eps = 1e-9 if prec == "f64" else (5e-5 if op == "epidiam" else 1e-5)
        res = hd.get_diameter(T, op == "epidiam", c.get("max_value"), precision=prec, epsilon=eps,
                              targets=np.array(c["targets"], np.int32), return_sweeps=True)
        out["none"] = np.array(res is None)
        if res is not None:
            out["d"], out["sweeps"] = np.array(res[0]), np.array(res[1])
    elif op == "norm":
        out["norm"] = np.array(hd.calculate_norm_discounted(make_T(c, c["seed"]), v_of(c), precision=prec))
    else:
        raise ValueError(op)
    out["paths"] = path_counts() - n0
    return out


# ------------------------------------------------------------------------------------------------------ the CPU side
@functools.lru_cache(maxsize=None)
def _oracle(key):
    c = json.loads(key)
    op = c["op"]
    if op == "disc":
        T, R, pi = make_mdp(c)
        return [orc.discounted_f64(T[b], R[b], pi[b] if c.get("pe") else None, gamma=GAM, tol=1e-12)[:2]
                for b in range(len(T))]
    if op == "gs":
        T, R, pi = make_mdp(c)
        return orc.discounted_gs_f32(T[0], R[0], pi[0] if c.get("pe") else None, gamma=GAM, eps=1e-3)
    if op == "backup":
        T, R, pi = make_mdp(c)
        fold = {"max": orc.FOLD_MAX, "pi": orc.FOLD_PI, "min": orc.FOLD_MIN}[c["fold"]]
        return orc.jacobi_sweeps_f64(T[0], R[0], v_of(c), 1, gamma=GAM, pi=pi[0], fold=fold)
    if op == "epi":
        T, R, pi = make_mdp(c)
        return [orc.episodic_f64(c["H"], T[b], R[b], pi[b] if c.get("pe") else None, c.get("max_value"))
                for b in range(len(T))]
    if op == "diam":
        return orc.diameter_continuous_f64(make_T(c, c["seed"]), np.array(c["targets"], np.int32), tol=1e-10)
    if op == "epidiam":
        return orc.diameter_episodic_f64(make_T_epi(c), np.array(c["targets"], np.int32), tol=1e-10)
    if op == "norm":
        return orc.value_norm_f64(make_T(c, c["seed"]), v_of(c).astype(np.float64))
    raise ValueError(op)


PRECISION_FREE = ("prec", "path", "n", "max_value")


def oracle(c):
    """the oracle's answer for case c (shared by both precisions, and by the bounded and unbounded runs of a case
    whose oracle does not see the bound)"""
    drop = PRECISION_FREE[:3] if c["op"] == "epi" else PRECISION_FREE
    return _oracle(json.dumps({k: v for k, v in c.items() if k not in drop}, sort_keys=True))


def check_paths(c, got):
    """exactly the expected path ran: c["path"] = name, c["n"] = its launches (None: at least one, "sweeps": one per
    sweep the solve reports); every other path stayed idle"""
    global TALLY
    paths = np.asarray(got["paths"])
    TALLY += paths
    k = P[c["path"]]
    n = c.get("n")
    if n == "sweeps":
        n = int(got["sweeps"]) * (c["H"] - 1 if c["op"] == "epidiam" else 1)
    seen = {PATH_KINDS[i]: int(v) for i, v in enumerate(paths) if v}
    assert paths[k] >= 1 and (n is None or paths[k] == n), (c, seen)
    assert all(v == 0 for i, v in enumerate(paths) if i != k), (c, seen)


def check_case(c, got):
    check_paths(c, got)
    op, prec = c["op"], c.get("prec", "f64")
    rtol = RTOL64 if prec == "f64" else RTOL32
    ref = oracle(c)
    if op == "disc":
        for b, (Qo, Vo) in enumerate(ref):
            np.testing.assert_allclose(got["V"][b], Vo, rtol=rtol, atol=rtol, err_msg=str(c))
            np.testing.assert_allclose(got["Q"][b], Qo, rtol=rtol, atol=rtol, err_msg=str(c))
        if "rscale" in c:  # instances froze at their own sweeps
            assert len(set(got["iters"].tolist())) > 1, (c, got["iters"])
    elif op == "gs":
        Qo, Vo, ito = ref
        assert abs(int(got["iters"][0]) - ito) <= 1, (c, got["iters"], ito)
        np.testing.assert_allclose(got["V"][0], Vo, atol=1.5e-3, err_msg=str(c))
        np.testing.assert_allclose(got["Q"][0], Qo, atol=1.5e-3, err_msg=str(c))
    elif op == "backup":
        Qo, Vo = ref
        r = 1e-12 if prec == "f64" else 1e-5
        scale = np.abs(Qo).max()
        np.testing.assert_allclose(got["Q"], Qo, rtol=r, atol=r * scale, err_msg=str(c))
        np.testing.assert_allclose(got["V"], Vo, rtol=r, atol=r * scale, err_msg=str(c))
        np.testing.assert_allclose(got["res"], np.abs(Vo - v_of(c)).max(), rtol=r, atol=r * scale, err_msg=str(c))
    elif op == "epi":
        assert bool(got["none"]) == any(o is None for o in ref), (c, [o is None for o in ref])
        if not bool(got["none"]):
            for b, (Qo, Vo) in enumerate(ref):
                np.testing.assert_allclose(got["V"][b], Vo, rtol=rtol, atol=rtol, err_msg=str(c))
                np.testing.assert_allclose(got["Q"][b], Qo, rtol=rtol, atol=rtol, err_msg=str(c))
    elif op in ("diam", "epidiam"):
        expect_none = c.get("max_value") is not None and ref > c["max_value"]
        assert bool(got["none"]) == expect_none, (c, ref)
        if not expect_none:
            assert abs(float(got["d"]) - ref) <= rtol * ref, (c, float(got["d"]), ref)
    elif op == "norm":
        assert abs(float(got["norm"]) - ref) <= (1e-10 if prec == "f64" else RTOL32) * ref, (c, float(got["norm"]), ref)


def run_here(cases):
    for c in cases:
        check_case(c, run_case(c))


CHILD = r"""
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import test_gpu_solver_paths as w
for k, case in enumerate(json.load(open(sys.argv[2]))):
    np.savez(f"{sys.argv[3]}/{k}.npz", **w.run_case(case))
"""
SWITCHES = ("COLO_NO_SPARSE", "COLO_NO_RESIDENT", "COLO_DIAM_PATH", "COLO_SPARSE_NT", "COLO_GS_NO_TMA",
            "COLO_EPISODIC_BATCHED", "COLO_NO_UMMA", "COLO_BACKUP_TMA")


def run_children(tmp_path, setting, cases):
    """the path switches are read once per process: the cases run in one child process with `setting` in its
    environment, the oracle and the checks here"""
    tag = "_".join(f"{k}{v}" for k, v in setting.items())
    d = tmp_path / tag
    d.mkdir()
    (d / "cases.json").write_text(json.dumps(cases))
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env.update(setting)
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(d / "cases.json"), str(d)], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    results = []
    for k, c in enumerate(cases):
        with np.load(d / f"{k}.npz") as z:
            results.append(dict(z))
        check_case(c, results[-1])
    return results


def both(cases):
    """every case in f64 and f32"""
    return [dict(c, prec=p) for c in cases for p in ("f64", "f32")]


def bounded(c, factor):
    """case c with max_value = factor x the oracle's diameter"""
    return dict(c, max_value=float(factor * oracle(c)))


# ------------------------------------------------------------------------------------------------ discounted VI / PE
def test_discounted_sparse_one_cta():
    """sparse_vi_kernel: the whole solve in one CTA with V in shared memory, S from 1 to the 2,048 limit"""
    cases = []
    for i, (S, A, k) in enumerate([(1, 3, 1), (7, 2, 3), (513, 3, 5), (2048, 2, 4), (2048, 1, 4)]):
        for pe in (False, True) if S < 2048 else (A == 1,):
            cases.append(dict(op="disc", S=S, A=A, k=k, B=1 + (S == 513), seed=100 + i, pe=pe, path="SPARSE_VI", n=1))
    run_here(both(cases))


def test_discounted_sparse_sweep():
    """sparse_sweep_kernel: S past the one-CTA limit, one compressed-row launch per sweep"""
    cases = [dict(op="disc", S=2049, A=2, k=4, seed=200, pe=pe, path="SPARSE_SWEEP") for pe in (False, True)]
    cases.append(dict(op="disc", S=3001, A=1, k=4, seed=201, path="SPARSE_SWEEP"))
    run_here(both(cases))


def test_discounted_resident():
    """resident_solve_kernel: dense T that fits a cluster's shared memory, one launch per solve"""
    cases = [dict(op="disc", S=S, A=A, B=2, seed=300 + S, pe=pe, path="RESIDENT", n=1)
             for S, A in ((100, 4), (37, 3)) for pe in (False, True)]
    for c in cases:
        assert resident_fits(c["S"], c["A"], 1, True)
    run_here(both(cases))


def test_discounted_backup_cta():
    """backup_kernel<GROUP_CTA = true>: one CTA per state (B*S < 64*SMs, S*A >= 4096); vector loads (S % 4 == 0),
    scalar loads, and the a0 >= kAT action loop (A = 9); T too large for the resident solver"""
    cases = []
    for i, (S, A) in enumerate([(1024, 4), (1027, 4), (1366, 3), (512, 9)]):
        assert S * A >= 4096 and S < 64 * sms() and not resident_fits(S, A, 1, False)
        cases.append(dict(op="disc", S=S, A=A, seed=400 + i, pe=bool(i % 2), path="BACKUP_CTA"))
    run_here(both(cases))


@pytest.mark.parametrize("fold", ["max", "pi", "min"])
def test_single_backup_cta_matches_fixed_sweep(fold):
    """one bellman_backup per CTA shape against jacobi_sweeps_f64, residual included: rounding level"""
    cases = [dict(op="backup", S=S, A=A, seed=450 + i, fold=fold, path="BACKUP_CTA", n=1)
             for i, (S, A) in enumerate([(1024, 4), (1027, 4), (1366, 3), (512, 9)])]
    run_here(both(cases))


def test_discounted_backup_warp_forced(tmp_path):
    """backup_kernel<GROUP_CTA = false> with the sparse and resident solvers off: S in {33, 130, 512}, A in
    {1, 4, 5, 9}, three instances each freezing at its own sweep"""
    cases = []
    for i, (S, A) in enumerate([(33, 1), (33, 9), (130, 4), (130, 5), (512, 4), (512, 5)]):
        assert S * A < 4096
        cases.append(dict(op="disc", S=S, A=A, B=3, rscale=[1.0, 0.01, 3.0], seed=500 + i, pe=bool(i % 2),
                          path="BACKUP_WARP"))
    run_children(tmp_path, {"COLO_NO_SPARSE": "1", "COLO_NO_RESIDENT": "1"}, both(cases))


# ------------------------------------------------------------------------------------------------ episodic VI / PE
def test_episodic_streaming_layers():
    """one backup_kernel launch per layer: B < 16 and T too large for the resident solver; warp mode (S*A < 4096) and
    CTA mode (S*A = 4096), with a per-layer policy"""
    cases = [dict(op="epi", S=700, A=4, H=5, B=3, seed=600, pe=pe, path="BACKUP_WARP", n=5) for pe in (False, True)]
    cases += [dict(op="epi", S=1024, A=4, H=3, B=2, seed=601, pe=pe, path="BACKUP_CTA", n=3) for pe in (False, True)]
    for c in cases:
        assert not resident_fits(c["S"], c["A"], 1, True)
    run_here(both(cases))


def test_episodic_batched_and_bounds():
    """B >= 16 without a bound: episodic_batched_kernel.  A bound turns it off (resident solver instead), and on the
    resident and streaming paths the answer is None exactly when the oracle's values exceed the bound"""
    small = dict(op="epi", S=40, A=3, H=6, B=16, seed=700)
    cases = [dict(small, path="EPI_BATCHED", n=1), dict(small, pe=True, path="EPI_BATCHED", n=1)]
    for base, path, n in ((small, "RESIDENT", 1), (dict(op="epi", S=700, A=4, H=4, B=3, seed=701), "BACKUP_WARP", 4)):
        vmax = max(Vo.max() for _, Vo in oracle(base))
        for f in (0.999, 1.001):
            cases.append(dict(base, max_value=float(f * vmax), path=path, n=n))
    run_here(both(cases))


# ------------------------------------------------------------------------------------------------ continuous diameter
def sparse_diam(S, K, seed, A=3):
    tg = sorted(set([0, S - 1] + list(np.random.RandomState(seed).choice(S, K, replace=False))))
    tg = [t for t in tg if t in (0, S - 1)] + [t for t in tg if t not in (0, S - 1)]
    return dict(op="diam", S=S, A=A, k=4, seed=seed, targets=[int(t) for t in tg[:K]])


@pytest.mark.parametrize("nt", ["1", "2", "4"])
def test_diameter_sparse_forced_nt(tmp_path, nt):
    """sparse_hitting_kernel<NT> with NT forced to 1, 2 and 4: K in {1, 3, 5, S} (ragged last tiles), targets 0 and
    S - 1, and a bound below the diameter"""
    cases = []
    for i, K in enumerate([1, 3, 5, 130]):
        c = dict(sparse_diam(130, K, 800 + i), path="SPARSE_HIT", n=1)
        cases.append(c)
    cases.append(dict(bounded(cases[2], 0.9)))
    run_children(tmp_path, {"COLO_SPARSE_NT": nt}, both(cases))


def test_diameter_resident_partial_tiles():
    """resident solver, tiles of 4 targets: K % 4 in {1, 2, 3}; the last tile is padded with copies of the last target.
    State 0 is nearly unreachable, so a tile padded with target 0 would overflow the bound the real targets meet"""
    S, A = 60, 3
    assert resident_fits(S, A, 4, True)
    cases = [dict(op="diam", S=S, A=A, seed=900 + K, targets=list(range(S - 1, S - 1 - K, -1)) + [0],
                  path="RESIDENT", n=1) for K in (4, 5, 6)]  # K + 1 targets: 5, 6, 7
    for K in (5, 6, 7):
        hard = dict(op="diam", S=S, A=A, seed=910 + K, rare0=True, targets=list(range(S - 1, S - 1 - K, -1)),
                    path="RESIDENT", n=1)
        cases += [bounded(hard, 3.0), bounded(hard, 0.9)]
    run_here(both(cases))


def test_diameter_gemm_and_umma_selected():
    """K*S >= 128^2 on dense T too large for the resident solver: hitting_gemm in f64 (and in f32 with K < 64),
    hitting_umma in f32 with K >= 64; one launch per sweep; a bound below the diameter gives None"""
    S, A = 448, 6
    assert not resident_fits(S, A, 4, False) and not resident_fits(S, A, 4, True)
    many = dict(op="diam", S=S, A=A, seed=1000, targets=[0, S - 1] + list(range(3, 3 + 62)))  # K = 64
    few = dict(op="diam", S=S, A=A, seed=1001, targets=[0, S - 1] + list(range(5, 5 + 35)))  # K = 37
    assert len(few["targets"]) * S >= 128 * 128
    cases = [dict(many, prec="f64", path="HIT_GEMM", n="sweeps"), dict(many, prec="f32", path="HIT_UMMA", n="sweeps"),
             dict(few, prec="f32", path="HIT_GEMM", n="sweeps")]
    cases += [dict(bounded(c, 0.9), n=None) for c in cases]
    run_here(cases)


def test_diameter_forced_gemm_and_stream(tmp_path):
    """COLO_DIAM_PATH=gemm: the SIMT GEMM in f32 where the tensor cores would run (same number as hitting_umma to
    rounding), S not a multiple of 64; COLO_DIAM_PATH=stream: backup_kernel with pinned targets, warp mode and CTA mode
    (S = 1100, A = 4, K = 3).  Episodic diameters on dense T_epi go to the same children"""
    S, A = 448, 6
    many = dict(op="diam", S=S, A=A, seed=1000, targets=[0, S - 1] + list(range(3, 3 + 62)))
    gemm = [dict(many, path="HIT_GEMM", n="sweeps")]
    gemm += both([dict(op="diam", S=200, A=3, seed=1100, targets=[0, 199] + list(range(1, 40)), path="HIT_GEMM",
                       n="sweeps")])
    gemm = [dict(c, prec=c.get("prec", "f32")) for c in gemm]
    gemm.append(dict(bounded(gemm[-1], 0.9), n=None))
    gemm += both([dict(op="epidiam", S=S_, A=3, H=H, seed=1200 + H, targets=list(range(S_)) if S_ == 37 else
                       [0, S_ - 1] + list(range(1, 19)), path="HIT_GEMM", n="sweeps") for S_, H in ((37, 2), (130, 3))])
    stream = both([dict(op="diam", S=200, A=3, seed=1300, targets=[0, 199, 17, 50, 3], path="BACKUP_WARP", n="sweeps"),
                   dict(op="diam", S=1100, A=4, seed=1301, targets=[0, 1099, 500], path="BACKUP_CTA", n="sweeps")])
    stream.append(dict(bounded(stream[-1], 0.9), n=None))
    stream += both([dict(op="epidiam", S=130, A=3, H=H, seed=1400 + H, targets=list(range(130)), path="BACKUP_WARP",
                         n="sweeps") for H in (2, 7)])
    forced = run_children(tmp_path, {"COLO_DIAM_PATH": "gemm"}, gemm)
    run_children(tmp_path, {"COLO_DIAM_PATH": "stream"}, stream)
    # the tensor cores (selected at this shape) and the forced SIMT GEMM: the same diameter to f32 rounding and the
    # stopping tolerance
    c = dict(many, prec="f32", path="HIT_UMMA", n="sweeps")
    umma = run_case(c)
    check_case(c, umma)
    assert abs(float(umma["d"]) - float(forced[0]["d"])) <= 2e-5 * float(forced[0]["d"]), (umma["d"], forced[0]["d"])


# ------------------------------------------------------------------------------------------------ episodic diameter
@pytest.mark.parametrize("H", [2, 3, 7])
def test_episodic_diameter_paths(H):
    """sparse_episodic_kernel on a sparse T_epi; on a dense T_epi the GEMM (K*S >= 64^2) or the per-layer backup
    (K*S < 64^2) as selected by the shape, both against the oracle and so against each other"""
    cases = [dict(op="epidiam", S=S, A=3, k=3, H=H, seed=1500 + S, targets=[0, S - 1] + list(range(1, 9)),
                  path="SPARSE_EPI", n=1) for S in (37, 130)]
    cases.append(dict(op="epidiam", S=130, A=3, H=H, seed=1600, targets=[0, 129] + list(range(1, 31)), path="HIT_GEMM",
                      n="sweeps"))  # K*S = 4160
    cases.append(dict(op="epidiam", S=130, A=3, H=H, seed=1600, targets=[0, 129] + list(range(1, 30)),
                      path="BACKUP_WARP", n="sweeps"))  # K*S = 4030
    cases.append(dict(op="epidiam", S=37, A=3, H=H, seed=1601, targets=list(range(37)), path="BACKUP_WARP", n="sweeps"))
    run_here(both(cases))


# ------------------------------------------------------------------------------------------------ value norm
def test_value_norm_paths():
    """two backup_kernel passes, the second with one V per action (v_action_stride = S): warp mode, and CTA mode with
    vector (S = 1100) and scalar (S = 1101) loads"""
    cases = [dict(op="norm", S=130, A=3, seed=1700, path="BACKUP_WARP", n=2)]
    cases += [dict(op="norm", S=S, A=4, seed=1701 + S, path="BACKUP_CTA", n=2) for S in (1100, 1101)]
    run_here(both(cases))


# ------------------------------------------------------------------------------------------------ in-place order
def gs_cases():
    # gamma = 0.9: at 0.99 the residual of these MDPs lingers near eps for several sweeps, and an f32 dot product in
    # another summation order (numpy's, or the warp's) stops up to four sweeps away from the sequential oracle
    dense = [dict(op="gs", S=128, A=4, seed=1800, path="GS_TMA", n=1), dict(op="gs", S=130, A=3, seed=1801,
                                                                           pe=True, path="GS_LDG", n=1)]
    # gs_sparse_kernel<ONEPASS>: A * KMp <= 32 (KMp = kmax rounded up to a power of two) and > 32
    sparse = [dict(op="gs", S=S, A=A, k=k, seed=1810 + i, pe=bool(i % 2), path="GS_SPARSE", n=1)
              for i, (S, A, k) in enumerate([(128, 4, 8), (130, 4, 8), (128, 4, 12), (131, 3, 16)])]
    return dense, sparse


def test_in_place_order_paths():
    """the reference's in-place sweeps against the loop-for-loop f32 oracle: TMA-staged dense rows (S % 4 == 0), plain
    loads (S % 4 != 0), compressed rows in one pass (A * KMp <= 32) and in several"""
    dense, sparse = gs_cases()
    run_here(dense + sparse)


def test_in_place_order_ldg_forced(tmp_path):
    """COLO_GS_NO_TMA: gs_solve_kernel on rows the TMA kernel would take (S % 4 == 0)"""
    dense, _ = gs_cases()
    run_children(tmp_path, {"COLO_GS_NO_TMA": "1"}, [dict(dense[0], path="GS_LDG")])


# ------------------------------------------------------------------------------------------------ selection boundaries
def disc_path(T, prec="f32"):
    import colosseum_b200.dynamic_programming as dp

    S, A = T.shape[0], T.shape[1]
    R = np.random.RandomState(S).uniform(0, 1, (S, A)).astype(np.float32)
    n0 = path_counts()
    dp._solve_discounted(T, R, None, GAM, 1e-3, None, prec)
    d = path_counts() - n0
    global TALLY
    TALLY += d
    return {PATH_KINDS[i] for i in np.nonzero(d)[0]}


def with_row(T, nnz):
    T = T.copy()
    T[0, 0] = 0.0
    T[0, 0, :nnz] = 1.0 / nnz
    return T


def test_boundary_compressed_rows():
    """a row of up to 8 non-zeros is always compressed; above that only while 8 * kmax <= S, and never above 256"""
    assert disc_path(with_row(sparse_T(64, 2, 2, 1), 8)) == {"SPARSE_VI"}
    assert disc_path(with_row(sparse_T(72, 2, 2, 2), 9)) == {"SPARSE_VI"}
    assert disc_path(with_row(sparse_T(71, 2, 2, 3), 9)) == {"RESIDENT"}
    assert disc_path(with_row(sparse_T(2048, 1, 2, 4), 256)) == {"SPARSE_VI"}
    assert disc_path(with_row(sparse_T(2048, 1, 2, 5), 257)) == {"BACKUP_WARP"}


def test_boundary_one_cta_sparse_solve():
    assert disc_path(sparse_T(2048, 2, 3, 6)) == {"SPARSE_VI"}
    assert disc_path(sparse_T(2049, 2, 3, 7)) == {"SPARSE_SWEEP"}


def test_boundary_group_cta():
    """one CTA per state below B * rows = 64 * SMs (rows of S * A >= 4096), one warp per state from there"""
    import torch

    import colosseum_b200.dynamic_programming as dp

    N = 64 * sms()
    T = torch.zeros((1, N, 1, N), dtype=torch.float32, device="cuda")
    R = torch.zeros((1, N, 1), dtype=torch.float32, device="cuda")
    for rows, path in ((N - 1, "BACKUP_CTA"), (N, "BACKUP_WARP")):
        vi = dp.BatchedValueIteration(T[:, :rows], R[:, :rows], GAM, precision="f32", S_total=N)
        n0 = path_counts()
        vi.sweep()
        torch.cuda.synchronize()
        d = path_counts() - n0
        global TALLY
        TALLY += d
        assert {PATH_KINDS[i]: int(v) for i, v in enumerate(d) if v} == {path: 1}, rows


def test_boundary_gemm():
    """the multi-target GEMM from K * S = 128^2 (f64; dense T too large for the resident solver)"""
    import colosseum_b200.hardness as hd

    S, A = 512, 4
    assert not resident_fits(S, A, 4, True)
    T = dense_T(S, A, 1900)
    global TALLY
    for K, path in ((128 * 128 // S - 1, "BACKUP_WARP"), (128 * 128 // S, "HIT_GEMM")):
        n0 = path_counts()
        _, sweeps = hd.get_diameter(T, False, targets=np.arange(K, dtype=np.int32), return_sweeps=True)
        d = path_counts() - n0
        TALLY += d
        assert {PATH_KINDS[i]: int(v) for i, v in enumerate(d) if v} == {path: sweeps}, K


# ------------------------------------------------------------------------------------------------ coverage
def test_every_solver_path_was_reached():
    """runs last: the cases above reached every COLO_PATH_* kind at least once"""
    missing = [name for name, n in zip(PATH_KINDS, TALLY) if n == 0]
    assert not missing, missing
