"""GPU parity of every dense step-kernel variant at every row width it is compiled for.

The dense step has one instantiation per row width NCH = ld / 128 = 1..8 (rows of at most 1024 states) for each of
the lean kernel (the common f32 call), the general k-ary kernel (fp32 and fp64), the warp-cooperative kernel
(COLO_STEP_KERNEL=coop, tiles of 8, 16 and 32 envs), plus the long-row kernel (more than 1024 states).  Every case here
runs synthetic MDPs through one of them and compares state, h, step_type, observation, reward bits, discount and both
visitation tables with the C oracle, bit for bit; `colo_step_kernel_launches` proves which variant ran.

The MDPs are built so that the search meets its hard cases: exact ties x == cdf[j] (bisect_right goes past j and past
any flat run of zero-probability states after it) at quad, block and chunk ends, also inside the lean kernel, whose
uniforms are predicted from the Philox stream; deterministic rows onto 0, 3, 4, 31, 32, 127, 128 and S-1; zero tails
(the clamp to the last positive-probability state); zero runs across quad, block and chunk boundaries; all 256 reward
classes, with ids 127, 128 and 255 on the next states the ties select, and different classes at positions 31 and 32.
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from colosseum_b200.tables import MDPTables
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LEAN, KARY, SHORT, LONG, SUCC = range(5)  # COLO_STEP_KIND_* of include/colosseum_b200.h
KIND_NAMES = ["env_step_kary_lean_kernel", "env_step_dense_kary_kernel", "env_step_dense_short_kernel",
              "env_step_dense_kernel", "env_step_succ_kernel"]

# states of each row width: no padding, and one state in the last chunk (plus a few odd sizes)
WIDTH_S = {k: [128 * k, 128 * (k - 1) + 1] for k in range(1, 9)}
WIDTH_S[1] += [2, 3, 33]
WIDTH_S[4] += [465]
LONG_S = [1024, 1025, 1056, 1057, 2049]  # the last short width, then long rows (ld = 1056, 1056, 1088, 2080)

TIE_POS = [0, 1, 2, 3, 4, 31, 32, 35, 127, 128, 131, 255, 383, 511, 639, 767, 895, 1023, 1024, 1055, 1056, 2047]
DET_POS = [0, 3, 4, 31, 32, 127, 128]
SPECIAL_CLS = [127, 128, 255, 7]  # class ids the tie rows' next states carry (7: the Beta class)
N_CLS, BETA_CLS = 256, 7
SEED = 20261020


def u24(w):
    return (w >> 8) * 2.0 ** -24


def philox_u24(seed, env, t):
    return u24(orc.philox(seed, env, t)[0])


def philox_u(seed, env, t, f64):
    """the step kernels' in-kernel next-state uniform: u24 of word 0 (fp32), u53 of words 0 and 1 (fp64)"""
    w = orc.philox(seed, env, t)
    return ((w[0] >> 5) * 2 ** 26 + (w[1] >> 6)) * 2.0 ** -53 if f64 else u24(w[0])


def n_tie_envs(N, S, A):
    return min(N, S * A, 64)


@functools.lru_cache(maxsize=4)
def make_mdp(S, A, H, seed, tie_u=()):
    """A synthetic MDP with a mix of rows (see the module docstring).  Row r = s * A + a < len(tie_u) is an exact tie
    for the uniform tie_u[r] (a multiple of 2^-24): cdf[p..j] == tie_u[r], then a zero run, then the rest of the mass
    at q, so the sampled state is q.  Returns (tables, dyadic rows, {row: (j, q)})."""
    rng = np.random.default_rng(seed)
    R = S * A
    T = np.zeros((R, S), np.float64)
    pos = np.arange(S)
    kind = (np.arange(R) + seed) % 5
    # 0: Dirichlet
    sel = np.nonzero(kind == 0)[0]
    T[sel] = rng.gamma(0.3, size=(len(sel), S))
    # 1: deterministic onto a boundary state
    det = [d for d in DET_POS if d < S] + [S - 1]
    sel = np.nonzero(kind == 1)[0]
    T[sel, np.array(det)[np.arange(len(sel)) % len(det)]] = 1.0
    # 2: zero tail: the last positive state is well before S - 1
    sel = np.nonzero(kind == 2)[0]
    last = rng.integers(0, max(1, S // 2), size=len(sel))
    T[sel] = rng.gamma(0.5, size=(len(sel), S)) * (pos[None, :] <= last[:, None])
    # 3: zero runs across quad, block and chunk boundaries (shifted per row)
    sel = np.nonzero(kind == 3)[0]
    shift = rng.integers(0, 4, size=(len(sel), 1))
    p = (pos[None, :] + shift)
    runs = ((p % 32) >= 29) | ((p % 32) <= 2) | ((p % 128) >= 118) | ((p % 8) == 5)
    T[sel] = rng.gamma(0.5, size=(len(sel), S)) * ~runs
    # 4: dyadic: masses k / 4096 summing to exactly 1, so every CDF entry is exact in fp32 and fp64
    sel = np.nonzero(kind == 4)[0]
    w = rng.gamma(0.2, size=(len(sel), S)) * (((pos[None, :] // 3) % 4) != 1)
    w[:, 0] += 1e-12
    T[sel] = rng.multinomial(4096, w / w.sum(1, keepdims=True)) / 4096.0
    empty = T.sum(1) == 0
    T[empty, S - 1] = 1.0
    T /= T.sum(1, keepdims=True)
    T[kind == 4] = np.round(T[kind == 4] * 4096) / 4096  # exact again after the normalisation
    cls = rng.integers(0, N_CLS, size=(R, S))
    if S > 32:
        cls[:, 32] = (cls[:, 31] + 1 + rng.integers(0, N_CLS - 1, size=R)) % N_CLS
    ties = {}
    targets = [j for j in TIE_POS if j < S - 1]
    for r, v in enumerate(tie_u):
        if not targets:
            break
        j, m = targets[r % len(targets)], r // len(targets)  # the m-th row that ties at j
        p0 = j - min(j, 5) if m % 3 == 1 else j  # a flat run [p0, j] up to the tie
        q = min(S - 1, j + 1 + [0, 1, 4, 29, 97][m % 5])  # then a zero run (j, q)
        T[r] = 0.0
        T[r, p0] = v
        T[r, q] += 1.0 - v
        cls[r, q] = SPECIAL_CLS[r % len(SPECIAL_CLS)]
        ties[r] = (j, q)
    dyadic = np.nonzero((kind == 4) | np.isin(np.arange(R), list(ties)))[0]
    start = np.unique([0, S - 1, S // 2])
    kinds = [("deterministic", (0.5 + k / 256.0,)) for k in range(N_CLS)]
    kinds[BETA_CLS] = ("beta", (2.0, 5.0))
    tb = MDPTables.from_dense(T.reshape(S, A, S).astype(np.float32), rew_kinds=kinds,
                              rew_cls_sas=cls.reshape(S, A, S).astype(np.uint8), start_idx=start,
                              start_prob=rng.dirichlet(np.ones(len(start))), H=H)
    return tb, dyadic, ties


def case_tables(case):
    """the case's MDP; its tie rows are exact for the lean kernel's own uniforms at the first step (t = 1)"""
    S, A, N = case["S"], case["A"], case["N"]
    tie_u = tuple(philox_u24(case["seed"], case["env0"] + e, 1) for e in range(n_tie_envs(N, S, A)))
    return make_mdp(S, A, case["H"], case["seed"], tie_u)


def edges(f64):
    return [0.0, 1.0 - 2.0 ** -24] + ([1.0 - 2.0 ** -53] if f64 else []) + [2.0 ** -30, 0.5]


def step_inputs(case, tb, dyadic, cdf, i, kind):
    """the inputs of step i, the same on both sides: (forced states or None, actions or None, uniforms or None,
    tie envs whose next state is checked against numpy as well)"""
    S, A, N = tb.S, tb.A, case["N"]
    f64 = case["mode"] == "dense_f64"
    rs = np.random.RandomState((case["seed"] * 7919 + i) % 2 ** 32)
    act = rs.randint(A, size=N).astype(np.int32)
    states, u, tie_envs = None, None, []
    if kind == "lean_tie":  # env e < K steps from row e: cdf == its own Philox uniform at the tie
        states = rs.randint(S, size=N).astype(np.int32)
        K = n_tie_envs(N, S, A) if S > 1 else 0
        states[:K], act[:K] = np.arange(K) // A, np.arange(K) % A
        tie_envs = list(range(K))
    elif kind in ("u_tie", "u"):
        u = rs.random_sample(N)
        if kind == "u_tie" and len(dyadic):  # u = cdf[j] / total on dyadic rows: x is exactly a CDF entry
            states = rs.randint(S, size=N).astype(np.int32)
            cands = sorted(set(j for j in TIE_POS if j < S))
            for e in range(min(N, 256)):
                if e % 8 == 5:
                    continue
                r = int(dyadic[(e * 7) % len(dyadic)])
                row = cdf[r // A, r % A, :S]
                flat = np.nonzero(np.diff(row) == 0)[0] + 1
                js = cands + [int(x) for x in flat[:: max(1, len(flat) // 4)][:4]]
                j = js[(e // 3) % len(js)]
                states[e], act[e] = r // A, r % A
                u[e] = float(row[j]) / float(row[S - 1])
                tie_envs.append(e)
        ed = edges(f64)
        sel = np.arange(5, N, 8)
        u[sel] = np.array(ed)[np.arange(len(sel)) % len(ed)]
        u = u.astype(np.float64 if f64 else np.float32)
    return states, act, u, tie_envs


def expected_kind(case, kind, stripped=False):
    if case["S"] > 1024:
        return LONG
    if case.get("force") == "coop":
        return SHORT
    lean_shaped = kind in ("lean_tie", "act")
    if lean_shaped and case["mode"] == "dense_f32" and case.get("force") != "general" and not stripped:
        return LEAN
    return KARY


# ------------------------------------------------------------------------------------------------------ GPU side
def launches():
    from colosseum_b200 import _cabi

    return np.array([_cabi.lib().colo_step_kernel_launches(k) for k in range(5)], np.int64)


def run_case(case, stripped=False):
    """runs the case's plan on the GPU; returns every step's outputs and launch-count deltas"""
    import torch

    from colosseum_b200.batched_mdp import BatchedMDP

    tb, dyadic, _ = case_tables(case)
    f64 = case["mode"] == "dense_f64"
    io = case["io"]
    env = BatchedMDP(tb, case["N"], mode=case["mode"], seed=case["seed"], env_offset=case["env0"],
                     host_io=io != "device", compact_io=io == "compact")
    out = {}
    if not stripped:
        for k in ("cdf", "cdf_mid", "cdf_coarse", "rew_cls_pad"):
            if env.dev.keep.get(k) is not None:
                out[k] = env.dev.keep[k].cpu().numpy()
    else:
        env.dev.c.cdf_mid = env.dev.c.cdf_coarse = env.dev.c.rew_cls_pad = None
    cdf = orc.build_dense_cdf(tb.T, ld=tb.ld, f64=f64)
    env.reset()
    for i, (kind, n) in enumerate(case["plan"]):
        states, act, u, _ = step_inputs(case, tb, dyadic, cdf, i, kind)
        if states is not None:
            env.state.copy_(torch.from_numpy(states))
            env.h.zero_()
            env.step_type.fill_(1)
        before = launches()
        if kind == "rand":
            env.step_async(None, auto_reset=True)
        elif kind == "fused":
            env.random_steps_fused(n, auto_reset=True)
        elif kind == "u" or kind == "u_tie":
            env.step_async(torch.from_numpy(act).cuda(), auto_reset=True, u_next=u)
        elif io == "device":
            env.step_async(torch.from_numpy(act).cuda(), auto_reset=True)
        else:
            env.step_host(torch.from_numpy(act).to(env.action_dtype).pin_memory(), auto_reset=True)
        torch.cuda.synchronize()
        out[f"{i}_launches"] = launches() - before
        # (the host_io fields are views of the pinned output block: copied, the next step overwrites them)
        out[f"{i}_state"] = env.state.cpu().numpy()
        out[f"{i}_h"] = env.h.cpu().numpy()
        out[f"{i}_st"] = (env.step_type_host if env.host_io else env.step_type).cpu().numpy().copy()
        out[f"{i}_obs"] = env.obs.cpu().numpy().astype(np.int32)
        out[f"{i}_reward"] = env.reward.cpu().numpy().copy()
        if env.discount is not None:
            out[f"{i}_discount"] = env.discount.cpu().numpy().copy()
    out["visits_s"] = env.visits_s.cpu().numpy()
    out["visits_sa"] = env.visits_sa.cpu().numpy()
    return out


# ------------------------------------------------------------------------------------------------------ oracle side
def bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def numpy_next(row, S, x):
    """bisect_right over the row, clamped to the first state where the row reaches its total"""
    j = int(np.searchsorted(row[:S], x, side="right"))
    return min(j, int(np.argmax(row[:S] >= row[S - 1])))


def check_case(case, got, stripped=False):
    """replays the case on the oracle and compares every output of `got` with it"""
    tb, dyadic, ties = case_tables(case)
    f64 = case["mode"] == "dense_f64"
    omode = 1 if f64 else 0
    N, S, A = case["N"], tb.S, tb.A
    cdf = orc.build_dense_cdf(tb.T, ld=tb.ld, f64=f64)
    tag = f"{case} stripped={stripped}"
    if "cdf" in got:
        assert np.array_equal(got["cdf"], cdf), tag
    if "cdf_mid" in got:  # the search index against its definition
        assert np.array_equal(got["cdf_mid"], cdf[..., 3::4]), tag
        assert np.array_equal(got["cdf_coarse"], cdf[..., 31::32]), tag
        pad = np.zeros((S, A, tb.ld), np.uint8)
        pad[..., :S] = tb.rew_cls_sas
        assert np.array_equal(got["rew_cls_pad"], pad), tag
    ht = orc.HostTables(S, A, H=tb.H, cdf=cdf, rew_cls_sas=tb.rew_cls_sas, rew_q=tb.rew_q, rmin=tb.rmin, rmax=tb.rmax,
                        start_cum=tb.start_cum, start_idx=tb.start_idx)
    vis_s = np.zeros(S, np.uint64)
    vis_sa = np.zeros((S, A), np.uint64)
    seed, env0 = case["seed"], case["env0"]
    state, h, st, _ = orc.env_reset(ht, N, seed=seed, t=0, visits_s=vis_s, env0=env0)
    t = 1
    for i, (kind, n) in enumerate(case["plan"]):
        where = f"{tag} step {i} ({kind})"
        want = expected_kind(case, kind, stripped)
        d = got[f"{i}_launches"]
        assert d[want] == 1 and d.sum() == 1, f"{where}: expected one launch of {KIND_NAMES[want]}, got {d.tolist()}"
        assert kind != "lean_tie" or t == 1, "the tie rows are built for the uniforms of the first step"
        states, act, u, tie_envs = step_inputs(case, tb, dyadic, cdf, i, kind)
        if states is not None:
            state[:], h[:], st[:] = states, 0, 1
        x_rows = [(e, int(state[e]), int(act[e])) for e in tie_envs]
        if kind in ("rand", "fused"):
            for k in range(n if kind == "fused" else 1):
                r, obs, rc, _ = orc.env_step(ht, omode, state, h, st, action=None, seed=seed, t=t + k, auto_reset=True,
                                             visits_s=vis_s, visits_sa=vis_sa, env0=env0)
            t += n if kind == "fused" else 1
        else:
            r, obs, rc, _ = orc.env_step(ht, omode, state, h, st, action=act.copy(), u_next=u, seed=seed, t=t,
                                         auto_reset=True, visits_s=vis_s, visits_sa=vis_sa, env0=env0)
            t += 1
        assert rc == 0, where
        for e, s, a in x_rows:  # the ties, against a plain numpy bisect_right as well
            row = cdf[s, a]
            uu = philox_u(seed, env0 + e, t - 1, f64) if kind == "lean_tie" else u[e]
            x = row.dtype.type(uu) * row[S - 1]
            assert state[e] == numpy_next(row, S, x), f"{where}: env {e}"
            if kind == "lean_tie" and s * A + a in ties:
                assert state[e] == ties[s * A + a][1], f"{where}: env {e}"
        assert np.array_equal(got[f"{i}_state"], state), where
        assert np.array_equal(got[f"{i}_h"], h), where
        assert np.array_equal(got[f"{i}_st"], st), where
        assert np.array_equal(got[f"{i}_obs"], obs), where
        rg = got[f"{i}_reward"]
        assert np.array_equal(np.isnan(rg), np.isnan(r)), where
        assert np.array_equal(bits(rg)[~np.isnan(r)], bits(r)[~np.isnan(r)]), where
        if f"{i}_discount" in got:
            disc = np.where(st == 1, 1.0, np.where(st == 2, 0.0, np.nan)).astype(np.float32)
            assert np.array_equal(bits(got[f"{i}_discount"]), bits(disc)), where
    assert np.array_equal(got["visits_s"], vis_s.astype(np.int64)), tag
    assert np.array_equal(got["visits_sa"], vis_sa.astype(np.int64)), tag


def a_for(S, i):
    return 1 + (i * 3 + S) % (7 if S <= 256 else 4 if S <= 640 else 3)


# ------------------------------------------------------------------------------------------------------ cases
LEAN_COMBOS = [("host", 4099, 0, 0), ("compact", 37, 3, 1000), ("compact", 4099, 0, 123457), ("host", 1, 5, 7),
               ("device", 37, 7, 5), ("device", 4099, 4, 0)]


@pytest.mark.parametrize("nch", range(1, 9))
def test_lean_kernel_matches_oracle(nch):
    """env_step_kary_lean_kernel<NCH, COMPACT> at every width: int32 host, compact and device-resident I/O, 1 / 37 /
    4099 envs (4099: ragged, and more than 16 counter copies x 128 threads), env offsets, continuous and episodic
    MDPs; the first step forces exact ties on the kernel's own Philox uniforms"""
    sizes = WIDTH_S[nch]
    for i in range(max(4, 2 * len(sizes))):
        io, N, H, env0 = LEAN_COMBOS[i % len(LEAN_COMBOS)]
        S = sizes[(i // 2) % len(sizes)]
        H = H and 3 + (H + nch) % 5
        case = dict(S=S, A=a_for(S, i), H=H, N=N, env0=env0, seed=SEED + 100 * nch + i, mode="dense_f32", io=io,
                    plan=[("lean_tie", 1)] + [("act", 1)] * (3 * H + 10))
        check_case(case, run_case(case))


@pytest.mark.parametrize("mode", ["dense_f32", "dense_f64"])
@pytest.mark.parametrize("nch", range(1, 9))
def test_general_kernel_matches_oracle(nch, mode):
    """env_step_dense_kary_kernel<TC, NCH> at every width in both precisions: supplied uniforms with exact ties at quad,
    block and chunk ends and in flat runs, edge uniforms (0, 1-2^-24, 1-2^-53), random actions, n steps in one launch;
    with and without the search index (which is compared with its definition)"""
    f64 = mode == "dense_f64"
    for i, S in enumerate(WIDTH_S[nch]):
        H = [0, 4][i % 2]
        plan = [("u_tie", 1), ("u", 1), ("u", 1), ("rand", 1), ("rand", 1), ("fused", H + 3)]
        if f64:  # the lean-shaped call in fp64 takes the general kernel
            plan = [("lean_tie", 1), ("act", 1)] + plan
        case = dict(S=S, A=a_for(S, i + nch), H=H, N=[777, 37][i % 2], env0=3 * i, seed=SEED + 10 * nch + i + 5000 * f64,
                    mode=mode, io=["device", "host"][i % 2], plan=plan)
        check_case(case, run_case(case))
        stripped = dict(case, plan=[("lean_tie", 1), ("u_tie", 1), ("act", 1), ("u", 1), ("rand", 1), ("fused", 3)])
        check_case(stripped, run_case(stripped, stripped=True), stripped=True)


@pytest.mark.parametrize("mode", ["dense_f32", "dense_f64"])
@pytest.mark.parametrize("S", LONG_S)
def test_long_rows_match_oracle(S, mode):
    """S = 1024 (the last short width) and S = 1025, 1056, 1057, 2049 (env_step_dense_kernel, ld a multiple of 32 but
    not always of 128): ties, edge uniforms, the lean-shaped call, random actions, n steps in one launch"""
    case = dict(S=S, A=2, H=[0, 5][S % 2], N=777, env0=11, seed=SEED + S + 7 * (mode == "dense_f64"), mode=mode,
                io="device", plan=[("lean_tie", 1), ("u_tie", 1), ("u", 1), ("act", 1), ("rand", 1), ("fused", 3)])
    check_case(case, run_case(case))


# ------------------------------------------------------------------------------------------------------ child processes
CHILD = r"""
import json, sys
import numpy as np
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import test_gpu_step_widths as w
for k, case in enumerate(json.load(open(sys.argv[2]))):
    np.savez(f"{sys.argv[3]}/{k}.npz", **w.run_case(case))
"""


def run_children(tmp_path, force, cases):
    """COLO_STEP_KERNEL is read once per process: the cases run in a child process, the oracle here"""
    spec = tmp_path / f"{force}.json"
    spec.write_text(json.dumps(cases))
    env = {k: v for k, v in os.environ.items() if not k.startswith("COLO_STEP_")}
    env["COLO_STEP_KERNEL"] = force
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(spec), str(tmp_path)], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    for k, case in enumerate(cases):
        with np.load(tmp_path / f"{k}.npz") as z:
            check_case(case, dict(z))


def test_warp_cooperative_kernel_matches_oracle(tmp_path):
    """env_step_dense_short_kernel<TC, NCH, U, TILE> (COLO_STEP_KERNEL=coop) at every width in both precisions; the
    tile follows from N: 37 envs -> 8, 4 x SMs x 32 -> 16, 8 x SMs x 32 -> 32"""
    import torch

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cases = []
    for nch in range(1, 9):
        for m, mode in enumerate(["dense_f32", "dense_f64"]):
            for j, N in enumerate([37, 4 * sms * 32, 8 * sms * 32]):
                S = WIDTH_S[nch][(m + j) % 2]
                plan = [("lean_tie", 1), ("u_tie", 1), ("u", 1), ("act", 1), ("rand", 1)]
                if N == 37:
                    plan += [("fused", 4)]
                cases.append(dict(S=S, A=a_for(S, nch + j), H=[0, 3][j % 2], N=N, env0=17 * j,
                                  seed=SEED + 1000 + 10 * nch + 3 * m + j, mode=mode, io="device", plan=plan,
                                  force="coop"))
    run_children(tmp_path, "coop", cases)


def test_forced_general_kernel_matches_oracle(tmp_path):
    """COLO_STEP_KERNEL=general: the lean-shaped call (supplied actions, in-kernel uniforms, auto-reset) through the
    general k-ary kernel at every width, forced ties included"""
    cases = []
    for nch in range(1, 9):
        for j, (io, N) in enumerate([("device", 4099), ("host", 37)]):
            S = WIDTH_S[nch][j]
            cases.append(dict(S=S, A=a_for(S, nch), H=3 * j, N=N, env0=5 + j, seed=SEED + 2000 + 10 * nch + j,
                              mode="dense_f32", io=io, plan=[("lean_tie", 1)] + [("act", 1)] * (9 * j + 6),
                              force="general"))
    run_children(tmp_path, "general", cases)
