"""`BatchedMDP`: N parallel episodes of one MDP advanced on the GPU with the semantics of the reference's
`BaseMDP.reset/step` (colosseum/mdp/base.py:1268-1355).

    env = BatchedMDP(MDPTables.from_mdp(reference_mdp), n_envs=65536, mode="dense_f32")
    ts = env.reset()
    ts = env.step(actions)            # actions: int32 [N] (numpy or CUDA tensor)
    ts, actions = env.random_step()   # BaseMDP.random_step for every env

With n_envs=1, `ts.scalar()` is the reference's scalar dm_env.TimeStep.  Modes:
  dense_f32 / dense_f64   warp-cooperative inverse-CDF search over the dense CDF row of T[s,a,:]
  succ                    successor-list tables in the reference sampler's own order: bit-exact with
                          NextStateSampler.sample for the same fp64 uniform (mdp/utils/custom_samplers.py:49-72)
Uniforms may be supplied (`u_next`, `u_reward`) or come from the in-kernel Philox4x32-10 stream keyed by
(seed; env index, step counter).  There is no CPU path.
"""
import ctypes as C

import numpy as np

from . import _cabi
from .tables import MDPTables
from .timestep import BatchedTimeStep, BoundedArray, DiscreteArray

_MODES = {"dense_f32": 0, "dense_f64": 1, "succ": 2}


class DeviceTables:
    """MDPTables uploaded to the current CUDA device + the `colo_mdp_tables` struct pointing at them.

    breaks=True: for dense_f32 rows of <= 1024 states with at most 16 breakpoints each (CDF entries above their
    predecessor) and at most one per 8 states, also the breakpoint table the f32 step kernels search in one round
    instead of the row (`colo_mdp_tables.cdf_breaks`); `breaks_k` is its entries per row (0: none)."""

    BREAKS_K = (2, 4, 8, 16)

    def __init__(self, tb: MDPTables, mode: str, breaks: bool = True):
        import torch

        _cabi.require_cuda()
        self.host = tb
        self.mode = mode
        dev = "cuda"
        k = {}

        def up(name, arr, dtype):
            if arr is None:
                k[name] = None
            else:
                k[name] = torch.from_numpy(np.ascontiguousarray(arr, dtype)).to(dev)

        up("start_cum", tb.start_cum, np.float64)
        up("start_idx", tb.start_idx, np.int32)
        up("rew_q", tb.rew_q, np.float32)
        c = _cabi.MdpTables()
        c.S, c.A, c.H = tb.S, tb.A, tb.H
        c.rmin, c.rmax = tb.rmin, tb.rmax
        c.n_cls, c.nq = tb.rew_q.shape
        c.n_start = tb.n_start
        if mode == "succ":
            assert tb.succ_cum is not None, "successor tables are required for mode='succ'"
            up("succ_cum", tb.succ_cum, np.float64)
            up("succ_idx", tb.succ_idx, np.int32)
            up("succ_len", tb.succ_len, np.int32)
            up("rew_cls_succ", tb.rew_cls_succ, np.int32)
            c.Ksucc = tb.succ_cum.shape[-1]
        else:
            assert tb.T is not None, "a dense T is required for the dense modes"
            f64 = mode == "dense_f64"
            up("T", tb.T, np.float32)
            ld = tb.ld
            k["cdf"] = torch.empty((tb.S, tb.A, ld), dtype=torch.float64 if f64 else torch.float32, device=dev)
            rc = _cabi.lib().colo_build_dense_cdf(_cabi.ptr(k["T"]), tb.S, tb.A, ld, _cabi.ptr(k["cdf"]), int(f64),
                                                  _cabi.current_stream())
            _cabi.check(rc, "colo_build_dense_cdf")
            c.ld = ld
            short_rows = ld % 128 == 0 and ld <= 1024
            if short_rows:  # two-level search index of the short-row step kernel
                k["cdf_mid"] = torch.empty((tb.S, tb.A, ld // 4), dtype=k["cdf"].dtype, device=dev)
                k["cdf_coarse"] = torch.empty((tb.S, tb.A, ld // 32), dtype=k["cdf"].dtype, device=dev)
                rc = _cabi.lib().colo_build_cdf_index(_cabi.ptr(k["cdf"]), tb.S, tb.A, ld, int(f64),
                                                      _cabi.ptr(k["cdf_mid"]), _cabi.ptr(k["cdf_coarse"]),
                                                      _cabi.current_stream())
                _cabi.check(rc, "colo_build_cdf_index")
            up("rew_cls_sas", tb.rew_cls_sas, np.uint8)
            up("rew_cls_sa", tb.rew_cls_sa, np.int32)
            if short_rows and k["rew_cls_sas"] is not None:  # class rows padded to ld: one aligned read per block
                k["rew_cls_pad"] = torch.nn.functional.pad(k["rew_cls_sas"], (0, ld - tb.S)).contiguous()
        for name in ("cdf", "succ_cum", "succ_idx", "succ_len", "rew_cls_sas", "rew_cls_sa", "rew_cls_succ", "rew_q",
                     "start_cum", "start_idx", "cdf_mid", "cdf_coarse", "rew_cls_pad"):
            setattr(c, name, _cabi.ptr(k.get(name)))
        self.breaks_k = 0
        if breaks and mode == "dense_f32" and short_rows:
            m = C.c_int(0)
            rc = _cabi.lib().colo_count_cdf_breaks(_cabi.ptr(k["cdf"]), tb.S, tb.A, ld, C.byref(m), _cabi.current_stream())
            _cabi.check(rc, "colo_count_cdf_breaks")
            # the density rule of the compressed-row kernels: rows denser than 1 in 8 keep the k-ary row search
            if m.value <= self.BREAKS_K[-1] and 8 * m.value <= tb.S:
                K = next(x for x in self.BREAKS_K if x >= m.value)
                k["cdf_breaks"] = torch.empty((tb.S, tb.A, K, 4), dtype=torch.int32, device=dev)
                rc = _cabi.lib().colo_build_cdf_breaks(C.byref(c), K, _cabi.ptr(k["cdf_breaks"]), _cabi.current_stream())
                _cabi.check(rc, "colo_build_cdf_breaks")
                c.cdf_breaks, c.cdf_breaks_k = _cabi.ptr(k["cdf_breaks"]), K
                self.breaks_k = K
        self.keep = k
        self.c = c


class BatchedMDP:
    VISIT_COPIES = 16  # privatised visitation counters (power of two), summed when read

    def __init__(self, tables: MDPTables, n_envs: int, mode: str = "dense_f32", seed: int = 0,
                 track_visits: bool = True, env_offset: int = 0, host_io: bool = False, stream=None,
                 device_tables=None, scalar_api: bool = False, compact_io: bool = False):
        """scalar_api=True (n_envs must be 1): `reset()` / `step(action: int)` / `random_step()` return the reference's
        SCALAR dm_env.TimeStep (`TimeStep(FIRST, None, None, obs)`, `(MID, r, 1.0, obs)`, `(LAST, r, 0.0, -1)`,
        mdp/base.py:1277,1316-1317), so the object can stand where a `BaseMDP` stood.
        host_io=True: the TimeStep fields (obs, reward, step_type) live in ONE pinned host buffer that the step
        kernel writes directly over PCIe (zero-copy), and `step_host` reads the actions straight from a pinned host
        tensor: an agent running on the host gets its TimeStep with one launch and one stream sync per step, no
        copy launches (include/colosseum_b200.h, colo_env_batch).  stream: a torch.cuda.Stream the host_io lean path
        (`step_host`, `send_host`/`recv_host`) launches on instead of the current stream (see PipelinedBatchedMDP).
        compact_io=True (with host_io): actions cross PCIe as uint8 and observations as int16 (-1 = terminal) --
        8 instead of 13 bytes per env-step; S <= 32767, A <= 256, auto-resetting dense f32 steps with supplied actions."""
        import torch

        assert mode in _MODES
        assert not scalar_api or int(n_envs) == 1, "scalar_api: one env, the reference's own regime"
        self.scalar_api = bool(scalar_api)
        self.torch = torch
        self.tables = tables
        self.dev = device_tables if device_tables is not None else DeviceTables(tables, mode)  # shards share one copy
        self.mode = mode
        self.n_envs = int(n_envs)
        self.seed = int(seed)
        # env_offset: global index of this shard's first env; the Philox counter is (env_offset + i, t), so a
        # batch sharded over GPUs draws exactly the numbers of the unsharded batch
        self.env_offset = int(env_offset)
        N = self.n_envs
        self.state = torch.zeros(N, dtype=torch.int32, device="cuda")
        self.h = torch.zeros(N, dtype=torch.int32, device="cuda")
        # before the first reset() the reference raises (necessary_reset is unset, base.py:405 vs :1272);
        # step_type = LAST + auto_reset=False reproduces that as an error, LAST + auto_reset=True resets.
        # the three TimeStep fields a host-side agent reads back live in ONE buffer (obs | reward | step_type), so an
        # end-to-end step is a single device->host copy
        self.host_io = bool(host_io)
        self.compact_io = bool(compact_io)
        assert not self.compact_io or (self.host_io and mode == "dense_f32" and track_visits and tables.S <= 32767
                                       and tables.A <= 256), "compact_io: host_io dense_f32 batches with counters"
        # (obs | reward | [discount |] step_type).  The device-resident block also carries dm_env's discount, written by
        # the step kernel's epilogue (no eager-PyTorch tail after a step); the pinned-host block does not (4 more
        # bytes per env over PCIe): there the discount is derived from step_type on the host when it is asked for.
        if self.compact_io:  # reward f32 | obs i16 | step_type u8: 7 bytes per env written over PCIe
            self._out = torch.zeros(7 * N, dtype=torch.uint8).pin_memory()
            self.step_type = torch.full((N,), _cabi.STEP_LAST, dtype=torch.uint8, device="cuda")
            self.step_type_host = self._out[6 * N:]
            self.step_type_host.fill_(_cabi.STEP_LAST)
            self.discount = None
        elif self.host_io:
            self._out = torch.zeros(9 * N, dtype=torch.uint8).pin_memory()
            self.step_type = torch.full((N,), _cabi.STEP_LAST, dtype=torch.uint8, device="cuda")  # kernel input too
            self.step_type_host = self._out[8 * N:]
            self.step_type_host.fill_(_cabi.STEP_LAST)
            self.discount = None
        else:
            self._out = torch.zeros(13 * N, dtype=torch.uint8, device="cuda")
            self.step_type = self._out[12 * N:]
            self.step_type.fill_(_cabi.STEP_LAST)
            self.discount = self._out[8 * N: 12 * N].view(torch.float32)
        if self.compact_io:
            self.reward = self._out[: 4 * N].view(torch.float32)
            self.obs = self._out[4 * N: 6 * N].view(torch.int16)
        else:
            self.obs = self._out[: 4 * N].view(torch.int32)
            self.reward = self._out[4 * N: 8 * N].view(torch.float32)
        self.action_dtype = torch.uint8 if self.compact_io else torch.int32
        self.action = torch.zeros(N, dtype=self.action_dtype, device="cuda")
        self.status = torch.zeros(1, dtype=torch.int32, device="cuda")
        vc = self.VISIT_COPIES
        self._visits_s = torch.zeros((vc, tables.S), dtype=torch.int64, device="cuda") if track_visits else None
        self._visits_sa = (torch.zeros((vc, tables.S, tables.A), dtype=torch.int64, device="cuda")
                           if track_visits else None)
        self.t = 0  # launch counter: the Philox stream position
        self._was_reset = False
        # static launch arguments, resolved once (a step is then one ctypes call)
        lib = _cabi.lib()
        self._step_fn = {"dense_f32": (lib.colo_env_step_dense_f32, torch.float32),
                         "dense_f64": (lib.colo_env_step_dense_f64, torch.float64),
                         "succ": (lib.colo_env_step_succ, torch.float64)}[mode]
        self._tb_ref = C.byref(self.dev.c)
        b = _cabi.EnvBatch()
        b.N, b.seed, b.env0 = N, self.seed, self.env_offset
        b.state, b.h, b.step_type = _cabi.ptr(self.state), _cabi.ptr(self.h), _cabi.ptr(self.step_type)
        b.action, b.reward, b.obs = _cabi.ptr(self.action), _cabi.ptr(self.reward), _cabi.ptr(self.obs)
        b.visits_s, b.visits_sa, b.visits_copies = _cabi.ptr(self._visits_s), _cabi.ptr(self._visits_sa), vc
        b.status = _cabi.ptr(self.status)
        b.step_type_mirror = self.step_type_host.data_ptr() if self.host_io else None
        b.discount = _cabi.ptr(self.discount)
        b.io_compact = int(self.compact_io)
        self._batch = b
        self._batch_ref = C.byref(b)
        self._own_action_ptr = b.action
        self._sync = lib.colo_stream_synchronize
        self.stream = stream
        self._stream_ptr = None if stream is None else int(stream.cuda_stream)
        self._stepper = None

    # -- reference attribute surface (base.py:463-503, 1233-1252)
    @property
    def n_states(self):
        return self.tables.S

    @property
    def n_actions(self):
        return self.tables.A

    @property
    def H(self):
        return self.tables.H if self.tables.H > 0 else None

    def is_episodic(self):
        return self.tables.H > 0

    @property
    def T(self):
        """f32 [S,A,S] (mdp/base.py:463-470)"""
        return self.tables.T

    @property
    def R(self):
        """f32 [S,A] expected rewards (mdp/base.py:472-479)"""
        return self.tables.R if self.tables.R is not None else self.tables.expected_rewards().astype(np.float32)

    @property
    def starting_state_distribution(self):
        return self.tables.starting_state_distribution

    @property
    def node_to_index(self):
        return self.tables.node_to_index

    @property
    def index_to_node(self):
        return self.tables.index_to_node

    @property
    def rewards_range(self):
        return (self.tables.rmin, self.tables.rmax)

    def action_spec(self):
        """mdp/base.py:1233-1240"""
        return DiscreteArray(self.tables.A, name="action")

    def observation_spec(self):
        """mdp/base.py:1242-1252: tabular observations unless an emission table was set"""
        if getattr(self, "_emit_table", None) is None:
            return DiscreteArray(self.tables.S, name="observation")
        return BoundedArray(self._emit_shape, np.float32, -np.inf, np.inf, "observation")

    def _u(self, u, dtype):
        if u is None:
            return None
        torch = self.torch
        if isinstance(u, torch.Tensor):
            return u.to(device="cuda", dtype=dtype).contiguous()
        return torch.from_numpy(np.ascontiguousarray(u, {torch.float32: np.float32, torch.float64: np.float64}[dtype])).cuda()

    def _timestep(self):
        torch = self.torch
        if self.host_io:  # host-resident fields: wait for the kernel that writes them
            torch.cuda.current_stream().synchronize()
        N = self.n_envs
        out = self._out.clone()  # ONE copy: the fields of this TimeStep survive the next step
        if self.compact_io:
            reward, obs = out[: 4 * N].view(torch.float32), out[4 * N: 6 * N].view(torch.int16)
        else:
            obs, reward = out[: 4 * N].view(torch.int32), out[4 * N: 8 * N].view(torch.float32)
        if self.host_io:  # host tensors: derive dm_env's discount from step_type on the host (no GPU work)
            st = out[6 * N:] if self.compact_io else out[8 * N:]
            discount = torch.full((N,), float("nan"))
            discount[st == _cabi.STEP_MID] = 1.0
            discount[st == _cabi.STEP_LAST] = 0.0
        else:
            st, discount = out[12 * N:], out[8 * N: 12 * N].view(torch.float32)
        ts = BatchedTimeStep(st, reward, discount, obs)
        return ts.scalar(0) if self.scalar_api else ts

    def reset(self, u_next=None) -> BatchedTimeStep:
        """BaseMDP.reset (base.py:1268-1277) for every env."""
        torch = self.torch
        u = self._u(u_next, torch.float64)
        rc = _cabi.lib().colo_env_reset(self._tb_ref, self._batch_ref, _cabi.ptr(u), self.t, _cabi.current_stream())
        _cabi.check(rc, "colo_env_reset")
        self.t += 1
        self._was_reset = True
        return self._timestep()

    def step_async(self, action=None, auto_reset=False, u_next=None, u_reward=None, check=False):
        """Enqueue one step for all envs on the current stream; results live in self.state / h / step_type /
        reward / obs (CUDA tensors, overwritten by the next step).  action=None plays uniformly random actions
        (BaseMDP.random_step, base.py:1341-1355) and records them in self.action."""
        torch = self.torch
        random_actions = action is None
        act_ptr = self._own_action_ptr
        if not random_actions:
            if isinstance(action, torch.Tensor):
                if (action.is_cuda or (self.host_io and action.is_pinned())) and action.dtype == self.action_dtype \
                        and action.is_contiguous():
                    act_ptr = action.data_ptr()  # read in place (device, or pinned host memory over PCIe): no copy
                else:
                    self.action.copy_(action, non_blocking=True)  # pinned host tensors: async H2D
            else:
                a = np.array(np.broadcast_to(np.asarray(action, np.int32), (self.n_envs,)))
                self.action.copy_(torch.from_numpy(a), non_blocking=True)
        fn, udt = self._step_fn
        un = None if u_next is None else self._u(u_next, udt)
        ur = None if u_reward is None else self._u(u_reward, torch.float32)
        self._batch.action = act_ptr
        rc = fn(self._tb_ref, self._batch_ref, int(random_actions), _cabi.ptr(un), _cabi.ptr(ur), self.t,
                int(bool(auto_reset)), torch.cuda.current_stream().cuda_stream)
        if rc != 0:
            _cabi.check(rc, "colo_env_step")
        self.t += 1
        if check or not auto_reset:
            # the reference asserts `not self.necessary_reset` (base.py:1291); stepping before reset() raises too
            st = int(self.status.item())
            if st == _cabi.BAD_ACTION:
                self.status.zero_()
                raise ValueError(f"an action outside [0, {self.tables.A}) was supplied (the env it belongs to was not stepped)")
            if st == _cabi.NEEDS_RESET:
                self.status.zero_()
                if not self._was_reset:
                    raise AttributeError("step() called before reset() (reference: necessary_reset is unset)")
                raise AssertionError("an episode has terminated: call reset() or step(..., auto_reset=True)")

    def step_host(self, action, auto_reset=False):
        """host_io mode: one launch + one stream sync; `action` is a pinned host int32 tensor read by the kernel
        itself.  Returns host views (obs i32[N], reward f32[N], step_type u8[N]) of the pinned output buffer,
        valid until the next step."""
        assert self.host_io, "construct the BatchedMDP with host_io=True"
        if not (auto_reset and action.dtype == self.action_dtype and action.is_pinned() and action.is_contiguous()):
            self.step_async(action, auto_reset=auto_reset)  # general path (checks, staging copies)
            self._sync(_cabi.current_stream())
            return self.obs, self.reward, self.step_type_host
        # lean path: two ctypes calls (launch, wait); everything else was resolved in __init__
        self.send_host(action)
        return self.recv_host()

    def send_host(self, action):
        """host_io lean path, first half: launch one auto-resetting step reading `action` (pinned int32) in place.
        Goes through a prepared stepper (colo_env_stepper_*): three scalar arguments per call instead of two structs
        and six scalars."""
        st = self._stepper
        if st is None:
            st = self._make_stepper()
        rc = self._stepper_launch(st, action.data_ptr(), self.t)
        if rc != 0:
            _cabi.check(rc, "colo_env_stepper_launch")
        self.t += 1

    def _make_stepper(self):
        stream = self._stream_ptr if self._stream_ptr is not None else _cabi.current_stream()
        out = C.c_void_p()
        rc = _cabi.lib().colo_env_stepper_create(self._tb_ref, self._batch_ref, _MODES[self.mode], stream, C.byref(out))
        _cabi.check(rc, "colo_env_stepper_create")
        self._stepper = out.value
        self._pending = stream
        self._stepper_launch = _cabi.lib().colo_env_stepper_launch
        return self._stepper

    def recv_host(self):
        """second half: wait for the step launched by `send_host`; returns the pinned host views."""
        self._sync(self._pending)
        return self.obs, self.reward, self.step_type_host

    # -- step server: the step kernel stays resident and is driven through a doorbell in pinned host memory
    def serve(self, action, idle_timeout_ms=200, share=1):
        """Start the persistent step kernel (include/colosseum_b200.h, colo_env_server_*).  `action` is the pinned
        int32 [N] buffer the agent writes its actions into before every `post()`; the TimeStep fields arrive in the
        pinned views `wait()` returns.  One step then costs no launch and no stream sync, only PCIe round trips.
        The kernel retires by itself after `idle_timeout_ms` without a step and is restarted transparently."""
        torch = self.torch
        assert self.host_io and not self.compact_io, "construct the BatchedMDP with host_io=True (and without compact_io)"
        assert action.dtype == torch.int32 and action.is_pinned() and action.is_contiguous() \
            and action.numel() == self.n_envs, "action: pinned contiguous int32 [N]"
        assert getattr(self, "_srv", None) is None, "already serving"
        if self.stream is None:
            self.stream = torch.cuda.Stream()
            self._stream_ptr = int(self.stream.cuda_stream)
        torch.cuda.current_stream().synchronize()  # reset()/steps enqueued on the caller's stream are done
        self._srv_action = action
        self._batch.action = action.data_ptr()
        self._srv_words = torch.zeros(32, dtype=torch.int64).pin_memory()  # doorbell [0], done [16]: own cache lines
        self._srv_ctl = torch.zeros(2, dtype=torch.int64, device="cuda")
        torch.cuda.current_stream().synchronize()
        srv = _cabi.EnvServer()
        srv.doorbell_host = self._srv_words.data_ptr()
        srv.done_host = self._srv_words.data_ptr() + 128
        srv.ctl_dev = self._srv_ctl.data_ptr()
        srv.share, srv.idle_timeout_ms = int(share), int(idle_timeout_ms)
        self._srv = srv
        self._srv_ref = C.byref(srv)
        self._served = 0
        self._posted = 0
        lib = _cabi.lib()
        self._srv_post, self._srv_wait = lib.colo_env_server_post, lib.colo_env_server_wait
        self._server_launch()
        return self

    def _server_launch(self):
        mode = {"dense_f32": 0, "dense_f64": 1, "succ": 2}[self.mode]
        rc = _cabi.lib().colo_env_server_start(self._tb_ref, self._batch_ref, self._srv_ref, mode, self.t, self._served,
                                               self._stream_ptr)
        _cabi.check(rc, "colo_env_server_start")

    def post(self):
        """ring the doorbell: the actions in the served buffer are final"""
        self._posted = self._srv_post(self._srv_ref)

    def wait(self, timeout_ms=10000):
        """block until the posted step's TimeStep is in host memory; returns the pinned views (obs, reward, step_type)"""
        rc = self._srv_wait(self._srv_ref, self._posted, timeout_ms)
        if rc != 0:
            if rc != _cabi.SERVER_LAPSED:
                _cabi.check(rc, "colo_env_server_wait")
            self._sync(self._stream_ptr)  # the retired kernel has left the stream
            self._server_launch()         # the doorbell already holds the pending step
            rc = self._srv_wait(self._srv_ref, self._posted, timeout_ms)
            if rc != 0:
                raise _cabi.ColosseumB200Error(f"colo_env_server_wait: rc={rc} after a restart: {_cabi.last_error()}")
        if self._served != self._posted:
            self._served = self._posted
            self.t += 1
        return self.obs, self.reward, self.step_type_host

    def step_served(self):
        self.post()
        return self.wait()

    def stop_serving(self):
        if getattr(self, "_srv", None) is None:
            return
        rc = _cabi.lib().colo_env_server_stop(self._srv_ref, self._stream_ptr)
        self._srv = None
        self._batch.action = self._own_action_ptr
        _cabi.check(rc, "colo_env_server_stop")

    def __del__(self):
        try:
            self.stop_serving()
            if getattr(self, "_stepper", None):
                _cabi.lib().colo_env_stepper_destroy(self._stepper)
                self._stepper = None
        except Exception:
            pass

    # -- checkpoint / resume: the whole state of the batch is three small tensors, the Philox counter and the counters
    def state_dict(self):
        """everything needed to continue the trajectories bit for bit (SURVEY.md section 5, checkpoint/resume)"""
        assert getattr(self, "_srv", None) is None, "stop_serving() before taking a checkpoint"
        self.torch.cuda.current_stream().synchronize()
        d = {"n_envs": self.n_envs, "seed": self.seed, "env_offset": self.env_offset, "t": self.t, "mode": self.mode,
             "was_reset": self._was_reset, "state": self.state.cpu(), "h": self.h.cpu(),
             "step_type": (self.step_type_host if self.host_io else self.step_type).cpu().clone(),
             "obs": self.obs.cpu().clone(), "reward": self.reward.cpu().clone()}
        if self.discount is not None:
            d["discount"] = self.discount.cpu().clone()
        if self._visits_s is not None:
            d["visits_s"], d["visits_sa"] = self._visits_s.sum(0).cpu(), self._visits_sa.sum(0).cpu()
        return d

    def load_state_dict(self, d):
        assert d["n_envs"] == self.n_envs and d["mode"] == self.mode, "checkpoint of another batch shape / sampler mode"
        self.seed, self.env_offset, self.t = int(d["seed"]), int(d["env_offset"]), int(d["t"])
        self._batch.seed, self._batch.env0 = self.seed, self.env_offset
        self._was_reset = bool(d["was_reset"])
        self.state.copy_(d["state"])
        self.h.copy_(d["h"])
        self.step_type.copy_(d["step_type"])
        if self.host_io:
            self.step_type_host.copy_(d["step_type"])
        self.obs.copy_(d["obs"])
        self.reward.copy_(d["reward"])
        if self.discount is not None and "discount" in d:
            self.discount.copy_(d["discount"])
        if self._visits_s is not None and "visits_s" in d:
            self._visits_s.zero_()
            self._visits_sa.zero_()
            self._visits_s[0].copy_(d["visits_s"])
            self._visits_sa[0].copy_(d["visits_sa"])
        self.torch.cuda.current_stream().synchronize()

    def fetch_async(self, host_buffer):
        """one device->host copy of the TimeStep block (obs i32[N] | reward f32[N] | discount f32[N] | step_type
        u8[N]; 13*N bytes, 9*N without the discount in host_io mode) into a pinned uint8 buffer, enqueued on the
        current stream; `split_host` views it as (obs, reward, step_type)."""
        host_buffer.copy_(self._out, non_blocking=True)

    def split_host(self, host_buffer):
        N = self.n_envs
        torch = self.torch
        return (host_buffer[: 4 * N].view(torch.int32), host_buffer[4 * N: 8 * N].view(torch.float32),
                host_buffer[(8 if self.host_io else 12) * N:])

    def step(self, action, auto_reset=False, u_next=None, u_reward=None) -> BatchedTimeStep:
        """BaseMDP.step (base.py:1279-1317) for every env."""
        self.step_async(action, auto_reset, u_next, u_reward)
        return self._timestep()

    def random_step(self, auto_reset=False):
        """BaseMDP.random_step (base.py:1341-1355): returns (BatchedTimeStep, actions)."""
        self.step_async(None, auto_reset)
        if self.scalar_api:
            return self._timestep(), int(self.action.item())
        return self._timestep(), self.action.clone()

    def random_steps(self, n, auto_reset=False):
        """BaseMDP.random_steps (base.py:1319-1339)."""
        return [self.random_step(auto_reset) for _ in range(n)]

    def set_emission_table(self, all_observations):
        """Non-tabular observations (colosseum/emission_maps/base.py:56-76): `all_observations` is the reference's
        precomputed table, f32 [H,S,...] (episodic) or [S,...] (continuous).  `emit_observations()` then returns the
        feature rows of the current TimeStep of every env (zeros past the horizon, :131-132)."""
        torch = self.torch
        t = all_observations if isinstance(all_observations, torch.Tensor) else torch.from_numpy(
            np.ascontiguousarray(all_observations, np.float32))
        t = t.to(device="cuda", dtype=torch.float32).contiguous()
        lead = 2 if self.tables.H > 0 else 1
        assert tuple(t.shape[:lead]) == ((self.tables.H, self.tables.S) if lead == 2 else (self.tables.S,))
        self._emit_shape = tuple(t.shape[lead:])
        self._emit_table = t.reshape(*t.shape[:lead], -1)
        self._emit_out = torch.empty((self.n_envs, self._emit_table.shape[-1]), dtype=torch.float32, device="cuda")

    def set_emission_noise(self, noise_class=None, seed=0, **noise_kwargs):
        """the `noise_class` / `noise_kwargs` of EmissionMap (emission_maps/base.py:85-104): "GaussianUncorrelated"
        (scale=0.1), "StudentTUncorrelated" (df=3), "GaussianCorrelated" (scale=0.1) or "StudentTCorrelated" (scale=0.1),
        by name or by reference class; None switches the noise off"""
        name = None if noise_class is None else getattr(noise_class, "__name__", str(noise_class))
        if name is None:
            self._emit_noise = None
        elif name == "GaussianUncorrelated":
            self._emit_noise = (1, float(noise_kwargs.get("scale", 0.1)), int(seed))
        elif name == "StudentTUncorrelated":
            self._emit_noise = (2, float(noise_kwargs.get("df", 3)), int(seed))
        elif name in ("GaussianCorrelated", "StudentTCorrelated"):
            # the covariance the reference draws ONCE per emission map (noises/gaussian_correlated.py:14-17): the same
            # scipy call on the same RandomState(seed) -> the same W; its Cholesky factor goes to the device
            import scipy.stats

            D = int(self._emit_table.shape[-1])
            rng = np.random.RandomState(int(seed))
            W = np.atleast_2d(scipy.stats.wishart(scale=[float(noise_kwargs.get("scale", 0.1))] * D).rvs(1, rng))
            self._emit_cov = W
            chol = np.linalg.cholesky(W).astype(np.float32)
            self._emit_chol = self.torch.from_numpy(np.ascontiguousarray(chol)).cuda()
            self._emit_noise = (3 if name == "GaussianCorrelated" else 4, float(noise_kwargs.get("df", 1.0)), int(seed))
        else:
            raise NotImplementedError(f"{name}: unknown noise class")
        self._emit_t = 0

    def emit_observations(self):
        """EmissionMap.get_observation for every env (one gather launch, plus one noise launch when a noise is set);
        f32 [N, *shape] CUDA tensor."""
        D = int(self._emit_table.shape[-1])
        rc = _cabi.lib().colo_emit_observations(_cabi.ptr(self._emit_table), _cabi.ptr(self.state), _cabi.ptr(self.h),
                                                _cabi.ptr(self.step_type), self.n_envs, self.tables.H, self.tables.S, D,
                                                _cabi.ptr(self._emit_out), _cabi.current_stream())
        _cabi.check(rc, "colo_emit_observations")
        noise = getattr(self, "_emit_noise", None)
        if noise is not None and noise[0] >= 3:
            kind, df, seed = noise
            rc = _cabi.lib().colo_emit_noise_correlated(_cabi.ptr(self._emit_out), _cabi.ptr(self.step_type), _cabi.ptr(self.h),
                                                        self.n_envs, self.tables.H, D, _cabi.ptr(self._emit_chol), kind - 2, df,
                                                        seed, self._emit_t, self.env_offset, _cabi.current_stream())
            _cabi.check(rc, "colo_emit_noise_correlated")
            self._emit_t += 1
        elif noise is not None:
            kind, param, seed = noise
            period = D if kind == 1 else max(1, int(np.prod(self._emit_shape[1:])))
            rc = _cabi.lib().colo_emit_noise(_cabi.ptr(self._emit_out), _cabi.ptr(self.step_type), _cabi.ptr(self.h),
                                             self.n_envs, self.tables.H, D, period, kind, param, seed, self._emit_t,
                                             self.env_offset, _cabi.current_stream())
            _cabi.check(rc, "colo_emit_noise")
            self._emit_t += 1
        return self._emit_out.view(self.n_envs, *self._emit_shape)

    def random_steps_fused(self, n, auto_reset=True):
        """n random-agent steps of every env in ONE launch (no per-step TimeStep list: state, h, visitation counts
        and the last step's TimeStep fields are what remains) -- bit-identical to n calls of random_step()."""
        self._batch.action = self._own_action_ptr
        rc = _cabi.lib().colo_env_random_steps(self._tb_ref, self._batch_ref, _MODES[self.mode], int(n), self.t,
                                               int(bool(auto_reset)), _cabi.current_stream())
        _cabi.check(rc, "colo_env_random_steps")
        self.t += int(n)
        if not auto_reset and int(self.status.item()) == _cabi.NEEDS_RESET:
            self.status.zero_()
            raise AssertionError("an episode has terminated: call reset() or use auto_reset=True")
        return self._timestep()

    @property
    def visits_s(self):
        """state visitation counts i64[S] (sum of the privatised copies)"""
        return None if self._visits_s is None else self._visits_s.sum(0)

    @property
    def visits_sa(self):
        """state-action visitation counts i64[S,A], counted on the NEXT node as in the reference (base.py:1302-1303)"""
        return None if self._visits_sa is None else self._visits_sa.sum(0)

    def get_visitation_counts(self, state_only=True):
        """base.py:1357-1373, as arrays indexed by state index (and action)."""
        return self.visits_s if state_only else self.visits_sa

    def reset_visitation_counts(self):
        """base.py:1375-1382"""
        if self._visits_s is not None:
            self._visits_s.zero_()
            self._visits_sa.zero_()


class MixedBatchedMDP:
    """One batch whose envs belong to different MDP instances, stepped by ONE launch per reset / step / fused random
    steps whatever the number of instances (include/colosseum_b200.h, colo_mixed_tables).  Instance i owns the
    contiguous envs `segment(i)`; there, with the instance's own tables, H, action range and seed `seed[i]`, the batch
    is bit-identical to `BatchedMDP(tables[i], n_envs[i], mode, seed=seed[i])` driven by the same calls.

        env = MixedBatchedMDP([inst.tables for inst in suite], 1024, mode="succ", seed=0)
        env.reset()
        env.random_steps_fused(1000)
        env.get_visitation_counts(3)      # instance 3's state counts

    `n_envs` and `seed` are an int for every instance or one value per instance.  Observations are state indices within
    the env's own instance.  Host I/O, compact I/O, the pipelines, the step server and emission maps are single-MDP."""
    VISIT_COPIES = BatchedMDP.VISIT_COPIES

    def __init__(self, tables, n_envs, mode: str = "succ", seed=0, track_visits: bool = True):
        import torch

        assert mode in _MODES
        self.torch = torch
        self.tables = list(tables)
        n = len(self.tables)
        assert n >= 1, "a mixed batch needs at least one instance"
        sizes = [int(n_envs)] * n if np.ndim(n_envs) == 0 else [int(x) for x in n_envs]
        seeds = [int(seed)] * n if np.ndim(seed) == 0 else [int(x) for x in seed]
        assert len(sizes) == n and len(seeds) == n, "n_envs and seed: one value, or one per instance"
        assert all(x >= 1 for x in sizes), "every instance needs at least one env"
        self.mode = mode
        self.sizes = np.array(sizes, np.int64)
        self.offsets = np.concatenate([[0], np.cumsum(self.sizes)[:-1]]).astype(np.int64)
        self.seeds = np.array(seeds, np.uint64)
        self.n_envs = int(self.sizes.sum())
        self.n_states = np.array([tb.S for tb in self.tables], np.int64)
        self.n_actions = np.array([tb.A for tb in self.tables], np.int64)
        self.H = np.array([tb.H for tb in self.tables], np.int64)  # 0: continuous
        self._s_off = np.concatenate([[0], np.cumsum(self.n_states)]).astype(np.int64)
        self._sa_off = np.concatenate([[0], np.cumsum(self.n_states * self.n_actions)]).astype(np.int64)
        # the single-MDP upload, reused as is: in the dense modes it also builds the short-row search index (cdf_mid,
        # cdf_coarse, rew_cls_pad) for rows of <= 1024 states, which the mixed kernels do not read -- a few build
        # launches per instance at construction and up to about half the bytes of an f32 dense CDF again.  The
        # breakpoint table, which they do not read either, is not built.
        self.dev = []
        for i, tb in enumerate(self.tables):
            try:
                self.dev.append(DeviceTables(tb, mode, breaks=False))
            except AssertionError as e:
                raise AssertionError(f"instance {i}: {e}") from None
        self._c_tables = (_cabi.MdpTables * n)(*[d.c for d in self.dev])
        self._handle = None
        self._make_handle()
        N = self.n_envs
        # i32[N]: the instance of every env, for the caller.  It mirrors the env -> instance map the handle uploaded for
        # the kernels (same sizes, same order; both fixed at construction) -- the kernels never read this copy.
        self.instance = torch.repeat_interleave(torch.arange(n, dtype=torch.int32),
                                                torch.from_numpy(self.sizes)).to("cuda")
        self.state = torch.zeros(N, dtype=torch.int32, device="cuda")
        self.h = torch.zeros(N, dtype=torch.int32, device="cuda")
        # obs i32 | reward f32 | discount f32 | step_type u8, as BatchedMDP's device-resident block (one clone per TimeStep)
        self._out = torch.zeros(13 * N, dtype=torch.uint8, device="cuda")
        self.obs = self._out[: 4 * N].view(torch.int32)
        self.reward = self._out[4 * N: 8 * N].view(torch.float32)
        self.discount = self._out[8 * N: 12 * N].view(torch.float32)
        self.step_type = self._out[12 * N:]
        self.step_type.fill_(_cabi.STEP_LAST)  # stepping before reset() is flagged, as in BatchedMDP
        self.action = torch.zeros(N, dtype=torch.int32, device="cuda")
        self.status = torch.zeros(1, dtype=torch.int32, device="cuda")
        vc = self.VISIT_COPIES
        size = _cabi.lib().colo_mixed_visits_size
        self._visits_s = torch.zeros((vc, size(self._handle, 0)), dtype=torch.int64, device="cuda") if track_visits else None
        self._visits_sa = torch.zeros((vc, size(self._handle, 1)), dtype=torch.int64, device="cuda") if track_visits else None
        self.t = 0
        self._was_reset = False
        self._udt = torch.float32 if mode == "dense_f32" else torch.float64
        b = _cabi.EnvBatch()
        b.N = N  # seed / env0 are not used by the mixed calls: every env takes them from its instance
        b.state, b.h, b.step_type = _cabi.ptr(self.state), _cabi.ptr(self.h), _cabi.ptr(self.step_type)
        b.action, b.reward, b.obs = _cabi.ptr(self.action), _cabi.ptr(self.reward), _cabi.ptr(self.obs)
        b.visits_s, b.visits_sa, b.visits_copies = _cabi.ptr(self._visits_s), _cabi.ptr(self._visits_sa), vc
        b.status = _cabi.ptr(self.status)
        b.discount = _cabi.ptr(self.discount)
        self._batch = b
        self._batch_ref = C.byref(b)
        self._own_action_ptr = b.action

    # BatchedMDP's helpers read only these of its attributes
    host_io = compact_io = scalar_api = False
    _u = BatchedMDP._u
    _timestep = BatchedMDP._timestep

    def _make_handle(self):
        n = len(self.tables)
        out = C.c_void_p()
        rc = _cabi.lib().colo_mixed_tables_create(self._c_tables, n, (C.c_longlong * n)(*self.sizes.tolist()),
                                                  (C.c_ulonglong * n)(*self.seeds.tolist()), _MODES[self.mode],
                                                  _cabi.current_stream(), C.byref(out))
        _cabi.check(rc, "colo_mixed_tables_create")
        if self._handle is not None:
            _cabi.lib().colo_mixed_tables_destroy(self._handle)
        self._handle = out.value

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _cabi.lib().colo_mixed_tables_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    @property
    def n_instances(self):
        return len(self.tables)

    def segment(self, i: int) -> slice:
        """the envs of instance i"""
        return slice(int(self.offsets[i]), int(self.offsets[i] + self.sizes[i]))

    def action_spec(self, i: int):
        return DiscreteArray(int(self.n_actions[i]), name="action")

    def observation_spec(self, i: int):
        return DiscreteArray(int(self.n_states[i]), name="observation")

    def reset(self, u_next=None) -> BatchedTimeStep:
        """BaseMDP.reset for every env, from its own instance's start distribution"""
        u = self._u(u_next, self.torch.float64)
        rc = _cabi.lib().colo_mixed_env_reset(self._handle, self._batch_ref, _cabi.ptr(u), self.t, _cabi.current_stream())
        _cabi.check(rc, "colo_mixed_env_reset")
        self.t += 1
        self._was_reset = True
        return self._timestep()

    def step_async(self, action=None, auto_reset=False, u_next=None, u_reward=None, check=False):
        """BatchedMDP.step_async over all envs: action=None plays uniformly random actions in [0, A_i) of every env's
        instance and records them in self.action"""
        torch = self.torch
        random_actions = action is None
        act_ptr = self._own_action_ptr
        if not random_actions:
            if isinstance(action, torch.Tensor) and action.is_cuda and action.dtype == torch.int32 and action.is_contiguous():
                act_ptr = action.data_ptr()
            elif isinstance(action, torch.Tensor):
                self.action.copy_(action, non_blocking=True)
            else:
                a = np.array(np.broadcast_to(np.asarray(action, np.int32), (self.n_envs,)))
                self.action.copy_(torch.from_numpy(a), non_blocking=True)
        un = None if u_next is None else self._u(u_next, self._udt)
        ur = None if u_reward is None else self._u(u_reward, torch.float32)
        self._batch.action = act_ptr
        rc = _cabi.lib().colo_mixed_env_step(self._handle, self._batch_ref, int(random_actions), _cabi.ptr(un),
                                             _cabi.ptr(ur), self.t, int(bool(auto_reset)),
                                             torch.cuda.current_stream().cuda_stream)
        if rc != 0:
            _cabi.check(rc, "colo_mixed_env_step")
        self.t += 1
        if check or not auto_reset:
            st = int(self.status.item())
            if st == _cabi.BAD_ACTION:
                self.status.zero_()
                raise ValueError("an action outside [0, A) of its env's instance was supplied (that env was not stepped)")
            if st == _cabi.NEEDS_RESET:
                self.status.zero_()
                if not self._was_reset:
                    raise AttributeError("step() called before reset() (reference: necessary_reset is unset)")
                raise AssertionError("an episode has terminated: call reset() or step(..., auto_reset=True)")

    def step(self, action, auto_reset=False, u_next=None, u_reward=None) -> BatchedTimeStep:
        self.step_async(action, auto_reset, u_next, u_reward)
        return self._timestep()

    def random_step(self, auto_reset=False):
        """BaseMDP.random_step for every env: returns (BatchedTimeStep, actions)"""
        self.step_async(None, auto_reset)
        return self._timestep(), self.action.clone()

    def random_steps(self, n, auto_reset=False):
        return [self.random_step(auto_reset) for _ in range(n)]

    def random_steps_fused(self, n, auto_reset=True):
        """n random-agent steps of every env in ONE launch -- bit-identical to n calls of random_step()"""
        self._batch.action = self._own_action_ptr
        rc = _cabi.lib().colo_mixed_env_random_steps(self._handle, self._batch_ref, int(n), self.t, int(bool(auto_reset)),
                                                     _cabi.current_stream())
        _cabi.check(rc, "colo_mixed_env_random_steps")
        self.t += int(n)
        if not auto_reset and int(self.status.item()) == _cabi.NEEDS_RESET:
            self.status.zero_()
            raise AssertionError("an episode has terminated: call reset() or use auto_reset=True")
        return self._timestep()

    def get_visitation_counts(self, i: int, state_only=True):
        """instance i's counts (base.py:1357-1373): i64[S_i], or i64[S_i, A_i] counted on the NEXT node"""
        if self._visits_s is None:
            return None
        if state_only:
            return self._visits_s[:, int(self._s_off[i]): int(self._s_off[i + 1])].sum(0)
        S, A = int(self.n_states[i]), int(self.n_actions[i])
        return self._visits_sa[:, int(self._sa_off[i]): int(self._sa_off[i + 1])].sum(0).view(S, A)

    def reset_visitation_counts(self):
        if self._visits_s is not None:
            self._visits_s.zero_()
            self._visits_sa.zero_()

    def state_dict(self):
        """everything needed to continue the trajectories bit for bit"""
        self.torch.cuda.current_stream().synchronize()
        d = {"sizes": self.sizes.copy(), "seeds": self.seeds.copy(), "t": self.t, "mode": self.mode,
             "was_reset": self._was_reset, "state": self.state.cpu(), "h": self.h.cpu(),
             "step_type": self.step_type.cpu().clone(), "obs": self.obs.cpu().clone(),
             "reward": self.reward.cpu().clone(), "discount": self.discount.cpu().clone()}
        if self._visits_s is not None:
            d["visits_s"], d["visits_sa"] = self._visits_s.sum(0).cpu(), self._visits_sa.sum(0).cpu()
        return d

    def load_state_dict(self, d):
        assert np.array_equal(d["sizes"], self.sizes) and d["mode"] == self.mode, \
            "checkpoint of another batch shape / sampler mode"
        if not np.array_equal(d["seeds"], self.seeds):
            self.seeds = np.array(d["seeds"], np.uint64)
            self._make_handle()
        self.t = int(d["t"])
        self._was_reset = bool(d["was_reset"])
        for name in ("state", "h", "step_type", "obs", "reward", "discount"):
            getattr(self, name).copy_(d[name])
        if self._visits_s is not None and "visits_s" in d:
            self._visits_s.zero_()
            self._visits_sa.zero_()
            self._visits_s[0].copy_(d["visits_s"])
            self._visits_sa[0].copy_(d["visits_sa"])
        self.torch.cuda.current_stream().synchronize()


def split_sizes(n: int, groups: int):
    """sizes and offsets of `groups` contiguous shards of n items, the first n % groups shards one item larger"""
    assert 1 <= groups <= n
    base, extra = divmod(int(n), int(groups))
    sizes = [base + (1 if g < extra else 0) for g in range(groups)]
    offsets = [sum(sizes[:g]) for g in range(groups)]
    return sizes, offsets


class PipelinedBatchedMDP:
    """N parallel envs split into `groups` contiguous shards, each a host_io BatchedMDP on its own stream, stepped in
    a software pipeline: while the host agent reads group g's TimeStep and writes its next actions, the other
    groups' step kernels are doing their PCIe reads/writes.  Env i of group g is global env offsets[g] + i
    (`env_offset`), so the trajectories are those of the unsplit batch; N need not be a multiple of `groups`
    (`sizes`, `offsets`).

        env = PipelinedBatchedMDP(tables, 65536, groups=2); env.reset()
        for g in range(env.groups): env.send(g, actions[g])         # prime
        while ...:
            for g in range(env.groups):
                obs, reward, step_type = env.recv(g)                 # group g's TimeStep (pinned host views)
                ...agent writes actions[g] (pinned int32)...
                env.send(g, actions[g])
    """

    def __init__(self, tables: MDPTables, n_envs: int, groups: int = 2, mode: str = "dense_f32", seed: int = 0,
                 track_visits: bool = True, env_offset: int = 0, compact_io: bool = False):
        import torch

        self._serving = False
        self.compact_io = bool(compact_io)  # uint8 actions in, int16 observations out (BatchedMDP.compact_io)

        self.groups = int(groups)
        self.n_envs = int(n_envs)
        self.sizes, self.offsets = split_sizes(self.n_envs, self.groups)
        self.per_group = self.sizes[0]
        dev = DeviceTables(tables, mode)
        self.shards = [BatchedMDP(tables, self.sizes[g], mode=mode, seed=seed, track_visits=track_visits,
                                  env_offset=env_offset + self.offsets[g], host_io=True,
                                  stream=torch.cuda.Stream(), device_tables=dev, compact_io=compact_io)
                       for g in range(groups)]
        torch.cuda.synchronize()  # the buffers were initialised on the default stream

    def reset(self):
        import torch

        out = []
        for sh in self.shards:
            with torch.cuda.stream(sh.stream):
                out.append(sh.reset())
        return out

    def serve(self, actions, idle_timeout_ms=200):
        """switch every group to its persistent step kernel (BatchedMDP.serve); `actions[g]` is group g's pinned
        action buffer, from then on `send(g)` takes no argument"""
        for sh, a in zip(self.shards, actions):
            sh.serve(a, idle_timeout_ms=idle_timeout_ms, share=self.groups)
        self._serving = True
        return self

    def stop_serving(self):
        for sh in self.shards:
            sh.stop_serving()
        self._serving = False

    def send(self, g: int, action=None):
        if self._serving:
            self.shards[g].post()
        else:
            self.shards[g].send_host(action)

    def recv(self, g: int):
        return self.shards[g].wait() if self._serving else self.shards[g].recv_host()

    def run_native(self, action_ring, n_steps, on_timestep=None, threads=False):
        """`n_steps` steps of every env with the recv/send loop run by the library (colo_env_pipeline_run): step i of
        group g reads `action_ring[i % len(action_ring)][g]` (pinned int32 tensors).  `on_timestep`: an optional
        ctypes callback `void(void* user, int group, int step)` -- a host agent written in C -- called when group g's
        TimeStep of `step` is in the pinned views (`shards[g].obs / reward / step_type_host`) and before its next
        launch.  Bit-identical to `n_steps` rounds of recv / send.  `threads=True`: one host thread per group
        (colo_env_pipeline_run_threads; `on_timestep` is then called on the group's own thread)."""
        import ctypes as C

        assert not self._serving
        G, Rn = self.groups, len(action_ring)
        for sh in self.shards:
            if sh._stepper is None:
                sh._make_stepper()
        hs = (C.c_void_p * G)(*[sh._stepper for sh in self.shards])
        ring = (C.c_void_p * (Rn * G))()
        for i, acts in enumerate(action_ring):
            for g, a in enumerate(acts):
                assert a.dtype == self.shards[g].action_dtype and a.is_pinned() and a.numel() == self.sizes[g]
                ring[i * G + g] = a.data_ptr()
        t0 = self.shards[0].t
        assert all(sh.t == t0 for sh in self.shards)
        run = _cabi.lib().colo_env_pipeline_run_threads if threads else _cabi.lib().colo_env_pipeline_run
        rc = run(hs, G, ring, Rn, t0, int(n_steps), on_timestep, None)
        _cabi.check(rc, "colo_env_pipeline_run_threads" if threads else "colo_env_pipeline_run")
        for sh in self.shards:
            sh.t += int(n_steps)
        return [(sh.obs, sh.reward, sh.step_type_host) for sh in self.shards]

    def run_queued(self, action_ring, n_steps, on_timestep=None, graph=True):
        """`run_native` without a stream synchronisation and a launch on the host per group-step
        (colo_env_pipeline_run_queued): every group's steps sit on a library-owned stream behind stream memory
        operations -- wait (go == i) -> step kernel -> write (done = i) -- enqueued ahead of time (`graph=True`: as
        replays of one CUDA graph of >= 64 steps per group), and the host loop per group-step is: spin on the pinned
        `done` word, `on_timestep`, store the pinned `go` word.  Same arguments, same order of events and bit-identical
        TimeSteps as `run_native`; the action ring must stay alive (and, for the graphs to be reused, the same) between
        calls."""
        import ctypes as C

        assert not self._serving
        G, Rn = self.groups, len(action_ring)
        for sh in self.shards:
            if sh._stepper is None:
                sh._make_stepper()
        if getattr(self, "_pipeline", None) is None:
            hs = (C.c_void_p * G)(*[sh._stepper for sh in self.shards])
            out = C.c_void_p()
            _cabi.check(_cabi.lib().colo_env_pipeline_create(hs, G, C.byref(out)), "colo_env_pipeline_create")
            self._pipeline = out.value
        ring = (C.c_void_p * (Rn * G))()
        for i, acts in enumerate(action_ring):
            for g, a in enumerate(acts):
                assert a.dtype == self.shards[g].action_dtype and a.is_pinned() and a.numel() == self.sizes[g]
                ring[i * G + g] = a.data_ptr()
        t0 = self.shards[0].t
        assert all(sh.t == t0 for sh in self.shards)
        rc = _cabi.lib().colo_env_pipeline_run_queued(self._pipeline, ring, Rn, t0, int(n_steps), on_timestep, None,
                                                      1 if graph else 0)
        _cabi.check(rc, "colo_env_pipeline_run_queued")
        for sh in self.shards:
            sh.t += int(n_steps)
        return [(sh.obs, sh.reward, sh.step_type_host) for sh in self.shards]

    def __del__(self):
        try:
            if getattr(self, "_pipeline", None):
                _cabi.lib().colo_env_pipeline_destroy(self._pipeline)
                self._pipeline = None
        except Exception:
            pass

    def step_all(self, actions):
        """one step of every env: launches all groups, then waits for each (actions: list of pinned int32 [N/groups])"""
        for sh, a in zip(self.shards, actions):
            sh.send_host(a)
        return [sh.recv_host() for sh in self.shards]

    def get_visitation_counts(self, state_only=True):
        tot = None
        for sh in self.shards:
            v = sh.get_visitation_counts(state_only)
            tot = v if tot is None else tot + v
        return tot
