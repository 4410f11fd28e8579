"""GPU tests of the breakpoint table (`colo_mdp_tables.cdf_breaks`) and of the two step kernels that search it.

A dense f32 CDF row with few breakpoints (entries above their predecessor) is a step function: the step kernels'
row search over it returns p_min(k*, m-1), k* = #{k : v_k <= x}.  `DeviceTables` builds, for tables whose rows all have
at most 16 breakpoints and at most one per 8 states, a table of K in {2, 4, 8, 16} entries per row (v, p, reward class,
the reward itself for constant classes), and the f32 step kernels search it in one round.  Here the table is compared
with its numpy definition, the selection rule with its statement, and the kernels with the C oracle, bit for bit:
state, h, step_type, observation, reward bits, discount and both visitation tables.

The synthetic MDPs hold dyadic rows (every CDF entry exact in fp32), rows with fewer breakpoints than K, first
breakpoints at 0 and elsewhere, reward classes 0, 127, 128 and 255 on breakpoints, a constant -0.0 class and a Beta
class; the first step of each lean case forces exact ties x == v_k on the kernel's own Philox uniforms.
"""
import os

import numpy as np
import pytest

from colosseum_b200.tables import MDPTables
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

LEAN, BREAKS, BREAKS_GENERAL = 0, 7, 8  # COLO_STEP_KIND_* of include/colosseum_b200.h
N_KINDS = 9
N_CLS, BETA_CLS, NEG0_CLS = 256, 7, 9
SPECIAL_CLS = [0, 127, 128, 255, BETA_CLS, NEG0_CLS]
INLINE = np.uint32(0x80000000)
SEED = 20261021
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
Q = 2.0 ** -24  # every mass is a multiple of it: CDF entries are exact in fp32 and fp64


def u24(w):
    return (w >> 8) * Q


def philox_u24(seed, env, t):
    return u24(orc.philox(seed, env, t)[0])


def sparse_mdp(S, A, m, H, seed, tie_u=()):
    """S x A rows of 1..m breakpoints (row 0 has exactly m).  Row r < len(tie_u) (m >= 2) has c[p_j] == tie_u[r] for
    some j, so that the uniform tie_u[r] hits breakpoint j exactly and the next state is p_(j+1)."""
    rng = np.random.default_rng(seed)
    R = S * A
    T = np.zeros((R, S), np.float64)
    for r in range(R):
        mr = m if r % 3 == 0 else int(rng.integers(1, m + 1))
        pos = np.sort(rng.choice(S, mr, replace=False))
        if r % 5 == 1:
            pos[0] = 0  # first breakpoint at 0 (elsewhere otherwise)
            pos = np.unique(pos)
            mr = len(pos)
        if r < len(tie_u) and mr >= 2:
            u = int(round(tie_u[r] / Q))
            j = r % (mr - 1) if u > mr else 0
            w = np.ones(mr, np.int64)
            w[0] = u - j  # masses of p_0..p_j sum to u, the rest to 2^24 - u
            w[j + 1] = (1 << 24) - u - (mr - j - 2)
            T[r, pos] = w * Q
        else:
            T[r, pos] = (rng.multinomial(4096 - mr, np.ones(mr) / mr) + 1) / 4096.0
    cls = rng.integers(0, N_CLS, size=(R, S))
    rows = rng.integers(0, R, size=4 * len(SPECIAL_CLS))
    for i, r in enumerate(rows):  # special classes on breakpoints
        nz = np.nonzero(T[r])[0]
        cls[r, nz[i % len(nz)]] = SPECIAL_CLS[i % len(SPECIAL_CLS)]
    kinds = [("deterministic", (0.5 + k / 256.0,)) for k in range(N_CLS)]
    kinds[BETA_CLS] = ("beta", (2.0, 5.0))
    start = np.unique([0, S - 1, S // 2])
    tb = MDPTables.from_dense(T.reshape(S, A, S).astype(np.float32), rew_kinds=kinds,
                              rew_cls_sas=cls.reshape(S, A, S).astype(np.uint8), start_idx=start,
                              start_prob=rng.dirichlet(np.ones(len(start))), H=H, rewards_range=(-0.25, 1.5))
    tb.rew_q[NEG0_CLS] = -0.0
    return tb


def breakpoints(row, S):
    """the definition: p with c[p] > c[p-1], c[-1] := 0 (a row without one: the single entry (0, 0))"""
    c = row[:S]
    p = np.nonzero(c > np.concatenate([[0], c[:-1]]))[0]
    return (p, c[p]) if len(p) else (np.zeros(1, np.int64), np.zeros(1, row.dtype))


def expected_table(tb, cdf, K):
    """[S, A, K] v, p and cls_flags of the table by its definition"""
    S, A = tb.S, tb.A
    v = np.zeros((S, A, K), np.float32)
    p = np.zeros((S, A, K), np.int32)
    for s in range(S):
        for a in range(A):
            pp, vv = breakpoints(cdf[s, a], S)
            assert len(pp) <= K
            p[s, a] = np.concatenate([pp, np.full(K - len(pp), pp[-1])])
            v[s, a] = np.concatenate([vv, np.full(K - len(vv), vv[-1])])
    cls = np.take_along_axis(tb.rew_cls_sas.astype(np.uint32), p, axis=2)
    q = tb.rew_q.view(np.uint32)
    const = np.all(q == q[:, :1], axis=1) & np.isfinite(tb.rew_q[:, 0])
    return v, p, cls | np.where(const[cls], INLINE, np.uint32(0))


def host_tables(tb, cdf):
    return orc.HostTables(tb.S, tb.A, H=tb.H, cdf=cdf, rew_cls_sas=tb.rew_cls_sas, rew_q=tb.rew_q, rmin=tb.rmin,
                          rmax=tb.rmax, start_cum=tb.start_cum, start_idx=tb.start_idx)


def check_table(dev, tb):
    """the built table against its definition; inline rewards against the oracle's draws at several uniforms"""
    K = dev.breaks_k
    cdf = orc.build_dense_cdf(tb.T, ld=tb.ld)
    got = dev.keep["cdf_breaks"].cpu().numpy().reshape(tb.S, tb.A, K, 4)
    v, p, cf = expected_table(tb, cdf, K)
    assert np.array_equal(got[..., 0].view(np.float32), v)
    assert np.array_equal(got[..., 1], p)
    assert np.array_equal(got[..., 2].view(np.uint32), cf)
    inl = (cf & INLINE) != 0
    assert not inl[(cf & ~INLINE) == BETA_CLS].any()
    # one env per (s, a, k) entry: a uniform inside (v_(k-1), v_k) selects p_k; the oracle draws its reward
    s, a, k = [x.ravel() for x in np.meshgrid(np.arange(tb.S), np.arange(tb.A), np.arange(K), indexing="ij")]
    lo = np.where(k > 0, v[s, a, np.maximum(k - 1, 0)], 0.0)
    total = v[s, a, K - 1]
    un = ((lo.astype(np.float64) + v[s, a, k]) / 2 / np.where(total > 0, total, 1)).astype(np.float32)
    ht = host_tables(tb, cdf)
    for ur in (0.0, 0.37, 1.0 - Q):
        state, h, st = s.astype(np.int32), np.zeros(len(s), np.int32), np.ones(len(s), np.uint8)
        r, _, rc, _ = orc.env_step(ht, 0, state, h, st, action=a.astype(np.int32), u_next=un,
                                   u_rew=np.full(len(s), ur, np.float32), seed=1, t=1)
        assert rc == 0
        hit = state == p[s, a, k]
        assert hit[inl[s, a, k]].mean() > 0.99
        sel = hit & inl[s, a, k]
        assert np.array_equal(got[s, a, k, 3][sel].view(np.uint32), r[sel].view(np.uint32)), ur


# ------------------------------------------------------------------------------------------------------ GPU harness
def launches():
    from colosseum_b200 import _cabi

    return np.array([_cabi.lib().colo_step_kernel_launches(k) for k in range(N_KINDS)], np.int64)


def edge_u(N, rs):
    u = rs.random_sample(N).astype(np.float32)
    ed = np.array([0.0, 1.0 - Q, 1.0, -0.25, 0.5], np.float32)
    sel = np.arange(3, N, 7)
    u[sel] = ed[np.arange(len(sel)) % len(ed)]
    return u


def run_and_check(tb, N, seed, env0, io, plan, want):
    """runs `plan` on the GPU and on the oracle side by side, comparing every step; `want(kind)` is the kernel kind
    each step must launch once"""
    import torch

    from colosseum_b200.batched_mdp import BatchedMDP

    env = BatchedMDP(tb, N, mode="dense_f32", seed=seed, env_offset=env0, host_io=io != "device",
                     compact_io=io == "compact")
    assert env.dev.breaks_k > 0
    cdf = env.dev.keep["cdf"].cpu().numpy()
    assert np.array_equal(cdf, orc.build_dense_cdf(tb.T, ld=tb.ld))
    ht = host_tables(tb, cdf)
    vis_s, vis_sa = np.zeros(tb.S, np.uint64), np.zeros((tb.S, tb.A), np.uint64)
    env.reset()
    state, h, st, _ = orc.env_reset(ht, N, seed=seed, t=0, visits_s=vis_s, env0=env0)
    t = 1
    for i, (kind, n) in enumerate(plan):
        rs = np.random.RandomState(seed * 31 + i)
        act = rs.randint(tb.A, size=N).astype(np.int32)
        u = None
        where = f"S={tb.S} N={N} io={io} step {i} ({kind})"
        if kind == "lean_tie":  # env e < S*A steps from row e, whose breakpoint sits on the env's own uniform
            K = min(N, tb.S * tb.A)
            states = rs.randint(tb.S, size=N).astype(np.int32)
            states[:K], act[:K] = np.arange(K) // tb.A, np.arange(K) % tb.A
            env.state.copy_(torch.from_numpy(states))
            env.h.zero_()
            env.step_type.fill_(1)
            state[:], h[:], st[:] = states, 0, 1
        before = launches()
        if kind == "rand":
            env.step_async(None, auto_reset=True)
        elif kind == "fused":
            env.random_steps_fused(n, auto_reset=True)
        elif kind == "u":
            u = edge_u(N, rs)
            env.step_async(torch.from_numpy(act).cuda(), auto_reset=True, u_next=u)
        elif kind == "server":
            buf = torch.zeros(N, dtype=torch.int32).pin_memory()
            env.serve(buf, idle_timeout_ms=500)
            try:
                for k in range(n):
                    a = np.random.RandomState(seed + 7 * k).randint(tb.A, size=N).astype(np.int32)
                    buf.copy_(torch.from_numpy(a))
                    o2, r2, _ = env.step_served()
                    r, obs, rc, _ = orc.env_step(ht, 0, state, h, st, action=a, seed=seed, t=t + k, auto_reset=True,
                                                 visits_s=vis_s, visits_sa=vis_sa, env0=env0)
                    assert rc == 0 and np.array_equal(o2.numpy(), obs), where
                    assert np.array_equal(r2.numpy().view(np.uint32), r.view(np.uint32)), where
            finally:
                env.stop_serving()
            t += n
        elif io == "device":
            env.step_async(torch.from_numpy(act).cuda(), auto_reset=True)
        else:
            env.step_host(torch.from_numpy(act).to(env.action_dtype).pin_memory(), auto_reset=True)
        torch.cuda.synchronize()
        d = launches() - before
        assert d[want(kind)] == 1 and d.sum() == 1, f"{where}: launches {d.tolist()}"
        if kind == "server":
            continue
        if kind in ("rand", "fused"):
            for k in range(n):
                r, obs, rc, _ = orc.env_step(ht, 0, state, h, st, action=None, seed=seed, t=t + k, auto_reset=True,
                                             visits_s=vis_s, visits_sa=vis_sa, env0=env0)
            t += n
        else:
            r, obs, rc, _ = orc.env_step(ht, 0, state, h, st, action=act.copy(), u_next=u, seed=seed, t=t,
                                         auto_reset=True, visits_s=vis_s, visits_sa=vis_sa, env0=env0)
            t += 1
        assert rc == 0, where
        if kind == "lean_tie":  # the tie rows against a plain numpy bisect_right, too
            for e in range(min(N, tb.S * tb.A, 64)):
                row = cdf[e // tb.A, e % tb.A]
                x = np.float32(philox_u24(seed, env0 + e, t - 1)) * row[tb.S - 1]
                j = int(np.searchsorted(row[:tb.S], x, side="right"))
                assert state[e] == min(j, int(np.argmax(row[:tb.S] >= row[tb.S - 1]))), f"{where}: env {e}"
        st_got = (env.step_type_host if env.host_io else env.step_type).cpu().numpy()
        assert np.array_equal(env.state.cpu().numpy(), state), where
        assert np.array_equal(env.h.cpu().numpy(), h), where
        assert np.array_equal(st_got, st), where
        assert np.array_equal(env.obs.cpu().numpy().astype(np.int32), obs), where
        rg = env.reward.cpu().numpy()
        assert np.array_equal(rg.view(np.uint32), r.view(np.uint32)), where
        if env.discount is not None:
            disc = np.where(st == 1, 1.0, np.where(st == 2, 0.0, np.nan)).astype(np.float32)
            assert np.array_equal(env.discount.cpu().numpy().view(np.uint32), disc.view(np.uint32)), where
    assert np.array_equal(env.visits_s.cpu().numpy(), vis_s.astype(np.int64))
    assert np.array_equal(env.visits_sa.cpu().numpy(), vis_sa.astype(np.int64))
    return env


def tie_mdp(S, A, m, H, seed, N, env0):
    """sparse_mdp whose first rows tie on the lean kernel's own uniforms at the first step (t = 1)"""
    tie_u = tuple(philox_u24(seed, env0 + e, 1) for e in range(min(N, S * A, 64)))
    return sparse_mdp(S, A, m, H, seed, tie_u)


# ------------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("m,K", [(1, 2), (2, 2), (3, 4), (4, 4), (5, 8), (8, 8), (9, 16), (16, 16)])
def test_table_matches_definition(m, K):
    """the table of every K, built from rows of up to m breakpoints (fewer in most rows), against its definition"""
    from colosseum_b200.batched_mdp import DeviceTables

    tb = sparse_mdp(max(8 * m, 8) + m % 3, 3, m, 0, SEED + m)
    dev = DeviceTables(tb, "dense_f32")
    assert dev.breaks_k == K
    check_table(dev, tb)


@pytest.mark.parametrize("S,m", [(200, 17), (31, 4), (33, 5)])
def test_no_table_for_dense_rows(S, m):
    """more than 16 breakpoints in a row, or more than one per 8 states: no table, the k-ary lean kernel runs"""
    import torch

    from colosseum_b200.batched_mdp import BatchedMDP

    tb = sparse_mdp(S, 2, m, 0, SEED + S)
    env = BatchedMDP(tb, 64, mode="dense_f32", seed=1)
    assert env.dev.breaks_k == 0 and env.dev.c.cdf_breaks is None
    env.reset()
    before = launches()
    env.step_async(torch.zeros(64, dtype=torch.int32, device="cuda"), auto_reset=True)
    torch.cuda.synchronize()
    assert (launches() - before)[LEAN] == 1


@pytest.mark.parametrize("name", ["c2_deepsea30_prand", "c2_deepsea30", "taxi_epi", "minigridempty5_epi",
                                  "riverswimcontinuous_ergo0", "simplegridcontinuous_ergo1"])
def test_golden_tables(name):
    """the sparse recorded instances get a table, matching its definition; C2 gets K = 2 and the breakpoint lean kernel"""
    import torch

    from colosseum_b200.batched_mdp import BatchedMDP

    g = np.load(os.path.join(GOLDEN, f"inst_{name}.npz"))
    tb = MDPTables.from_golden(g)
    env = BatchedMDP(tb, 1000, mode="dense_f32", seed=3)
    assert env.dev.breaks_k > 0
    if tb.rew_cls_sas is not None:
        check_table(env.dev, tb)
    if name == "c2_deepsea30_prand":
        assert env.dev.breaks_k == 2
    env.reset()
    before = launches()
    env.step_async(torch.zeros(1000, dtype=torch.int32, device="cuda"), auto_reset=True)
    torch.cuda.synchronize()
    assert (launches() - before)[BREAKS] == 1


LEAN_COMBOS = [("host", 4099, 0, 0), ("compact", 37, 3, 1000), ("device", 1, 0, 7), ("device", 65536, 4, 5),
               ("compact", 4099, 0, 123457), ("host", 37, 5, 3)]


@pytest.mark.parametrize("m", [2, 4, 7, 16])
def test_lean_breaks_kernel_matches_oracle(m):
    """env_step_breaks_lean_kernel<K, COMPACT> for each K: int32 host, compact and device I/O, 1 / 37 / 4,099 / 65,536
    envs, env offsets, continuous and episodic; the first step forces exact ties on the kernel's own uniforms"""
    for i, (io, N, H, env0) in enumerate(LEAN_COMBOS[(m % 3):(m % 3) + 4]):
        S = 8 * m + 3 * i
        seed = SEED + 100 * m + i
        tb = tie_mdp(S, 2 + i % 2, m, H, seed, N, env0)
        plan = [("lean_tie", 1)] + [("act", 1)] * (3 * H + 6)
        run_and_check(tb, N, seed, env0, io, plan, lambda kind: BREAKS)


@pytest.mark.parametrize("m", [2, 4, 7, 16])
def test_general_breaks_kernel_matches_oracle(m):
    """env_step_dense_kary_kernel on the table (kind 8): random actions, a fused walk, supplied uniforms with edges
    0, 1-2^-24, 1.0 and a negative value, and the step server"""
    for i, (io, N, H, env0) in enumerate([("device", 4099, 0, 11), ("host", 37, 4, 0)]):
        S = 8 * m + 5 * i
        seed = SEED + 1000 + 10 * m + i
        tb = tie_mdp(S, 3, m, H, seed, N, env0)
        plan = [("lean_tie", 1), ("u", 1), ("rand", 1), ("fused", H + 5), ("u", 1)]
        if io == "host":
            plan += [("server", 6), ("act", 1)]
        run_and_check(tb, N, seed, env0, io, plan,
                      lambda kind: BREAKS if kind in ("lean_tie", "act") else BREAKS_GENERAL)


def test_c2_same_trajectory_with_and_without_table():
    """C2 at 65,536 envs x 50 steps: the breakpoint lean kernel and the k-ary lean kernel (table nulled) emit the same
    TimeSteps, states and visitation counts"""
    import torch

    from colosseum_b200.batched_mdp import BatchedMDP

    g = np.load(os.path.join(GOLDEN, "inst_c2_deepsea30_prand.npz"))
    tb = MDPTables.from_golden(g)
    N = 65536
    gen = torch.Generator().manual_seed(5)
    acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, generator=gen).cuda() for _ in range(50)]

    def run(strip):
        env = BatchedMDP(tb, N, mode="dense_f32", seed=8)
        if strip:
            env.dev.c.cdf_breaks, env.dev.c.cdf_breaks_k = None, 0
        env.reset()
        out = []
        before = launches()
        for a in acts:
            env.step_async(a, auto_reset=True)
            out.append((env.obs.clone(), env.reward.clone().view(torch.int32), env.step_type.clone()))
        torch.cuda.synchronize()
        assert (launches() - before)[LEAN if strip else BREAKS] == len(acts)
        return out, env.state.clone(), env.visits_s.clone(), env.visits_sa.clone()

    ref, got = run(True), run(False)
    for x, y in zip(ref[0], got[0]):
        assert all(torch.equal(p, q) for p, q in zip(x, y))
    assert all(torch.equal(p, q) for p, q in zip(ref[1:], got[1:]))
