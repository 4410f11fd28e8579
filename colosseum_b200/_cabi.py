"""ctypes binding of libcolosseum_b200.so (include/colosseum_b200.h).

There is no CPU fallback: if the CUDA library is missing this module raises at first use, loudly.
PyTorch is used only as the device-buffer / stream provider (tensor.data_ptr(), torch.cuda.current_stream()).
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("COLO_B200_LIB") or os.path.join(_PKG, "_lib", "libcolosseum_b200.so")  # env: kernel-variant probes only

OK, OVERFLOW, MAX_ITER, NEEDS_RESET, SERVER_LAPSED, BAD_ACTION = 0, 1, 2, 3, 4, 5
FOLD_MAX, FOLD_PI, FOLD_MIN = 0, 1, 2
STEP_FIRST, STEP_MID, STEP_LAST = 0, 1, 2
# step-kernel variants of colo_step_kernel_launches (include/colosseum_b200.h, COLO_STEP_KIND_*)
STEP_KIND_LEAN, STEP_KIND_KARY, STEP_KIND_SHORT, STEP_KIND_LONG, STEP_KIND_SUCC = 0, 1, 2, 3, 4
STEP_KIND_MIXED_SUCC, STEP_KIND_MIXED_DENSE = 5, 6
STEP_KIND_BREAKS, STEP_KIND_BREAKS_GENERAL = 7, 8


class ColosseumB200Error(RuntimeError):
    pass


class BackupArgs(C.Structure):
    """mirror of `colo_backup_args`"""

    _fields_ = [
        ("T", C.c_void_p), ("R", C.c_void_p), ("pi", C.c_void_p),
        ("V_in", C.c_void_p), ("V_out", C.c_void_p), ("Q", C.c_void_p),
        ("t_stride", C.c_longlong), ("r_stride", C.c_longlong), ("pi_stride", C.c_longlong),
        ("v_in_stride", C.c_longlong), ("v_out_stride", C.c_longlong), ("q_stride", C.c_longlong),
        ("v_action_stride", C.c_longlong),
        ("B", C.c_int), ("S", C.c_int), ("A", C.c_int), ("fold", C.c_int),
        ("gamma", C.c_double), ("r_const", C.c_double),
        ("resid", C.c_void_p), ("resid_vs_out", C.c_int),
        ("active", C.c_void_p),
        ("max_abs", C.c_double), ("overflow_signed", C.c_int), ("overflow_flag", C.c_void_p),
        ("row0", C.c_int), ("nrows", C.c_int),
        ("pin_index", C.c_void_p), ("pin_value", C.c_double),
        ("exclude_index", C.c_void_p), ("exclude_value", C.c_double),
        ("V_out_peers", C.c_void_p), ("n_peers", C.c_int),
    ]


class MdpTables(C.Structure):
    """mirror of `colo_mdp_tables` (device pointers)"""

    _fields_ = [
        ("S", C.c_int), ("A", C.c_int), ("H", C.c_int), ("ld", C.c_int),
        ("cdf", C.c_void_p),
        ("succ_cum", C.c_void_p), ("succ_idx", C.c_void_p), ("succ_len", C.c_void_p), ("Ksucc", C.c_int),
        ("rew_cls_sas", C.c_void_p), ("rew_cls_sa", C.c_void_p), ("rew_cls_succ", C.c_void_p),
        ("rew_q", C.c_void_p), ("n_cls", C.c_int), ("nq", C.c_int),
        ("rmin", C.c_float), ("rmax", C.c_float),
        ("start_cum", C.c_void_p), ("start_idx", C.c_void_p), ("n_start", C.c_int),
        ("cdf_mid", C.c_void_p), ("cdf_coarse", C.c_void_p), ("rew_cls_pad", C.c_void_p),
        ("cdf_breaks", C.c_void_p), ("cdf_breaks_k", C.c_int),
    ]


class ResidentArgs(C.Structure):
    """mirror of `colo_resident_args`"""

    _fields_ = [
        ("T", C.c_void_p), ("R", C.c_void_p), ("pi", C.c_void_p), ("V", C.c_void_p), ("Q", C.c_void_p),
        ("t_stride", C.c_longlong), ("r_stride", C.c_longlong),
        ("B", C.c_int), ("S", C.c_int), ("A", C.c_int), ("NV", C.c_int), ("fold", C.c_int),
        ("gamma", C.c_double), ("r_const", C.c_double), ("eps", C.c_double),
        ("max_abs", C.c_double), ("overflow_signed", C.c_int),
        ("max_iter", C.c_longlong), ("episodic_H", C.c_int),
        ("pin_index", C.c_void_p), ("pin_value", C.c_double),
        ("iters_out", C.c_void_p), ("status_out", C.c_void_p),
    ]


class EnvBatch(C.Structure):
    """mirror of `colo_env_batch` (device pointers)"""

    _fields_ = [
        ("N", C.c_longlong), ("seed", C.c_ulonglong), ("env0", C.c_ulonglong),
        ("state", C.c_void_p), ("h", C.c_void_p), ("step_type", C.c_void_p), ("action", C.c_void_p),
        ("reward", C.c_void_p), ("obs", C.c_void_p), ("visits_s", C.c_void_p), ("visits_sa", C.c_void_p),
        ("visits_copies", C.c_int), ("status", C.c_void_p), ("step_type_mirror", C.c_void_p),
        ("discount", C.c_void_p), ("io_compact", C.c_int),
    ]


class EnvServer(C.Structure):
    """mirror of `colo_env_server`"""

    _fields_ = [("doorbell_host", C.c_void_p), ("done_host", C.c_void_p), ("ctl_dev", C.c_void_p),
                ("share", C.c_int), ("idle_timeout_ms", C.c_uint)]


class ActorArgs(C.Structure):
    """mirror of `colo_actor_args`"""

    _fields_ = [("epsilon_schedule", C.c_void_p), ("temperature_schedule", C.c_void_p), ("t0", C.c_longlong),
                ("len", C.c_int), ("boltzmann", C.c_int), ("boltzmann_temperature", C.c_double)]


class QLearningArgs(C.Structure):
    """mirror of `colo_qlearning_args`"""

    _fields_ = [
        ("N", C.c_longlong), ("seed", C.c_ulonglong), ("env0", C.c_ulonglong),
        ("state", C.c_void_p), ("h", C.c_void_p), ("cnt", C.c_void_p), ("Q", C.c_void_p), ("Q_main", C.c_void_p),
        ("V", C.c_void_p), ("mu", C.c_void_p), ("sigma", C.c_void_p), ("beta", C.c_void_p),
        ("ucb_type", C.c_int),
        ("c_1", C.c_double), ("c_2", C.c_double), ("min_at", C.c_double), ("log_term", C.c_double),
        ("sqrt_h7sa", C.c_double), ("H_eff", C.c_double), ("gamma", C.c_double), ("span_approx", C.c_double),
        ("epsilon_greedy", C.c_double), ("cum_reward", C.c_void_p), ("n_episodes", C.c_void_p),
        ("trace", C.c_void_p), ("actor", ActorArgs),
    ]


class PsrlArgs(C.Structure):
    """mirror of `colo_psrl_args`"""

    _fields_ = [
        ("N", C.c_longlong), ("seed", C.c_ulonglong), ("env0", C.c_ulonglong),
        ("state", C.c_void_p), ("h", C.c_void_p), ("Q", C.c_void_p), ("dir_hyper", C.c_void_p),
        ("nig_hyper", C.c_void_p), ("epsilon_greedy", C.c_double), ("cum_reward", C.c_void_p),
        ("n_episodes", C.c_void_p), ("trace", C.c_void_p), ("reward_model", C.c_int), ("actor", ActorArgs),
    ]


class Ucrl2Args(C.Structure):
    """mirror of `colo_ucrl2_args`"""

    _fields_ = [
        ("N", C.c_longlong), ("seed", C.c_ulonglong), ("env0", C.c_ulonglong),
        ("state", C.c_void_p), ("t", C.c_void_p), ("cum_reward", C.c_void_p), ("Q", C.c_void_p),
        ("Nsas", C.c_void_p), ("Nsa", C.c_void_p), ("P", C.c_void_p), ("est_r", C.c_void_p), ("var_r", C.c_void_p),
        ("hold", C.c_void_p), ("nu", C.c_void_p), ("seen", C.c_void_p), ("ep_len", C.c_void_p), ("ep_log", C.c_void_p),
        ("log_cap", C.c_int), ("ended", C.c_void_p), ("iteration", C.c_void_p), ("episode", C.c_void_p),
        ("delta", C.c_void_p), ("epsilon_greedy", C.c_double), ("trace", C.c_void_p), ("trace_t0", C.c_longlong),
        ("trace_steps", C.c_int), ("actor", ActorArgs),
    ]


class PsrlcArgs(C.Structure):
    """mirror of `colo_psrlc_args`"""

    _fields_ = [
        ("N", C.c_longlong), ("seed", C.c_ulonglong), ("env0", C.c_ulonglong),
        ("state", C.c_void_p), ("t", C.c_void_p), ("cum_reward", C.c_void_p), ("Q", C.c_void_p), ("psi", C.c_int),
        ("dir_hyper", C.c_void_p), ("nig_hyper", C.c_void_p), ("reward_model", C.c_int),
        ("Nsas", C.c_void_p), ("Nsa", C.c_void_p), ("nu", C.c_void_p), ("ended", C.c_void_p), ("episode", C.c_void_p),
        ("epsilon_greedy", C.c_double), ("trace", C.c_void_p), ("trace_t0", C.c_longlong), ("trace_steps", C.c_int),
        ("actor", ActorArgs),
    ]


class SuiteInstance(C.Structure):
    """mirror of `colo_suite_instance` (HOST pointers)"""

    _fields_ = [
        ("S", C.c_int), ("A", C.c_int), ("H", C.c_int), ("K", C.c_int),
        ("T", C.c_void_p), ("R", C.c_void_p), ("succ_cum", C.c_void_p), ("succ_idx", C.c_void_p),
        ("succ_len", C.c_void_p), ("rew_cls_succ", C.c_void_p), ("rew_q", C.c_void_p),
        ("n_cls", C.c_int), ("nq", C.c_int), ("rmin", C.c_float), ("rmax", C.c_float),
        ("start_idx", C.c_void_p), ("start_cum", C.c_void_p), ("start_prob", C.c_void_p), ("n_start", C.c_int),
        ("node_h", C.c_void_p), ("node_s", C.c_void_p), ("n_nodes", C.c_int), ("deterministic", C.c_int),
    ]


class SuiteConfig(C.Structure):
    """mirror of `colo_suite_config`"""

    _fields_ = [("n_envs", C.c_longlong), ("n_steps", C.c_int), ("seed", C.c_ulonglong), ("eps", C.c_double),
                ("max_cf_bytes", C.c_size_t), ("diameter", C.c_int)]


class SuiteResult(C.Structure):
    """mirror of `colo_suite_result`"""

    _fields_ = [("status", C.c_int), ("visits_total", C.c_double), ("mean_reward_last_step", C.c_double),
                ("gaps", C.c_double), ("value_norm", C.c_double), ("diameter", C.c_double),
                ("diameter_sweeps", C.c_double), ("step_s", C.c_double), ("hardness_s", C.c_double),
                ("error", C.c_char * 160)]


_P = C.c_void_p
_LL = C.c_longlong
_ULL = C.c_ulonglong
_I = C.c_int
_F = C.c_float
_D = C.c_double

# name -> (restype, argtypes); every symbol include/colosseum_b200.h declares
PROTOTYPES = {
    "colo_last_error": (C.c_char_p, []),
    "colo_version": (_I, []),
    "colo_launch_count": (_ULL, []),
    "colo_reset_launch_count": (None, []),
    "colo_backup_tma_sweeps": (_ULL, []),
    "colo_step_kernel_launches": (_ULL, [_I]),
    "colo_stream_synchronize": (_I, [_P]),
    "colo_backup_f32": (_I, [C.POINTER(BackupArgs), _P]),
    "colo_backup_f64acc": (_I, [C.POINTER(BackupArgs), _P]),
    "colo_resident_fits": (_I, [_I, _I, _I, _I, C.POINTER(C.c_int)]),
    "colo_resident_solve_f32": (_I, [C.POINTER(ResidentArgs), _P]),
    "colo_resident_solve_f64acc": (_I, [C.POINTER(ResidentArgs), _P]),
    "colo_solve_work_bytes": (C.c_size_t, [_LL, _LL, _I]),
    "colo_solve_discounted_f32": (_I, [_P, _P, _P, _I, _I, _I, _F, _F, _F, _LL, _I, _P, _P, _P, _P, _P]),
    "colo_solve_discounted_f64acc": (_I, [_P, _P, _P, _I, _I, _I, _D, _D, _D, _LL, _I, _P, _P, _P, _P, _P]),
    "colo_solve_discounted_gs_f32": (_I, [_P, _P, _P, _I, _I, _I, _F, _F, _F, _LL, _I, _P, _P, _P, _P, _P]),
    "colo_solve_discounted_gs_f64acc": (_I, [_P, _P, _P, _I, _I, _I, _D, _D, _D, _LL, _I, _P, _P, _P, _P, _P]),
    "colo_suite_release_caches": (_I, []),
    "colo_suite_run": (_I, [C.POINTER(SuiteInstance), _I, C.POINTER(SuiteConfig), C.POINTER(SuiteResult), _I]),
    "colo_continuous_form_values_f32": (_I, [_P, _P, _I, _I, _I, _D, _P, _P, _P, _I, _D, _I, _P, C.POINTER(C.c_double), _P]),
    "colo_continuous_form_values_f64acc": (_I, [_P, _P, _I, _I, _I, _D, _P, _P, _P, _I, _D, _I, _P, C.POINTER(C.c_double), _P]),
    "colo_hitting_umma_sweeps_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "colo_episodic_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _F, _P, _P, _P]),
    "colo_episodic_policies_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "colo_episodic_policies_f64acc": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "colo_episodic_f64acc": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _D, _P, _P, _P]),
    "colo_diameter_continuous_work_bytes": (C.c_size_t, [_I, _I, _I]),
    "colo_diameter_continuous_f32": (_I, [_P, _P, _I, _I, _I, _F, _F, _LL, _P, _P, _P]),
    "colo_diameter_continuous_f64acc": (_I, [_P, _P, _I, _I, _I, _D, _D, _LL, _P, _P, _P]),
    "colo_diameter_continuous_gs_work_bytes": (C.c_size_t, [_I, _I, _I]),
    "colo_diameter_continuous_gs_f32": (_I, [_P, _P, _I, _I, _I, _F, _F, _LL, _P, _P, _P]),
    "colo_diameter_continuous_gs_f64acc": (_I, [_P, _P, _I, _I, _I, _D, _D, _LL, _P, _P, _P]),
    "colo_diameter_episodic_work_bytes": (C.c_size_t, [_I, _I, _I, _I, _I]),
    "colo_diameter_episodic_f32": (_I, [_P, _P, _I, _I, _I, _I, _F, _F, _LL, _P, _P, _P]),
    "colo_diameter_episodic_f64acc": (_I, [_P, _P, _I, _I, _I, _I, _D, _D, _LL, _P, _P, _P]),
    "colo_value_norm_work_bytes": (C.c_size_t, [_I, _I, _I]),
    "colo_value_norm_f32": (_I, [_P, _P, _I, _I, _P, _P, _P]),
    "colo_value_norm_f64acc": (_I, [_P, _P, _I, _I, _P, _P, _P]),
    "colo_bias_series_work_bytes": (C.c_size_t, [_I]),
    "colo_bias_series_f64": (_I, [_P, _P, _I, _I, _P, _P, _P]),
    "colo_gaps_f64": (_I, [_P, _P, _P, _LL, _I, _D, _P, _P]),
    "colo_env_reset": (_I, [C.POINTER(MdpTables), C.POINTER(EnvBatch), _P, _ULL, _P]),
    "colo_env_step_dense_f32": (_I, [C.POINTER(MdpTables), C.POINTER(EnvBatch), _I, _P, _P, _ULL, _I, _P]),
    "colo_env_step_dense_f64": (_I, [C.POINTER(MdpTables), C.POINTER(EnvBatch), _I, _P, _P, _ULL, _I, _P]),
    "colo_env_step_succ": (_I, [C.POINTER(MdpTables), C.POINTER(EnvBatch), _I, _P, _P, _ULL, _I, _P]),
    "colo_env_random_steps": (_I, [C.POINTER(MdpTables), C.POINTER(EnvBatch), _I, _I, _ULL, _I, _P]),
    "colo_mixed_tables_create": (_I, [C.POINTER(MdpTables), _I, C.POINTER(C.c_longlong), C.POINTER(C.c_ulonglong), _I,
                                      _P, C.POINTER(C.c_void_p)]),
    "colo_mixed_tables_destroy": (None, [_P]),
    "colo_mixed_visits_size": (_LL, [_P, _I]),
    "colo_mixed_env_reset": (_I, [_P, C.POINTER(EnvBatch), _P, _ULL, _P]),
    "colo_mixed_env_step": (_I, [_P, C.POINTER(EnvBatch), _I, _P, _P, _ULL, _I, _P]),
    "colo_mixed_env_random_steps": (_I, [_P, C.POINTER(EnvBatch), _I, _ULL, _I, _P]),
    "colo_emit_noise_correlated": (_I, [_P, _P, _P, _LL, _I, _I, _P, _I, _D, _ULL, _ULL, _ULL, _P]),
    "colo_env_pipeline_run": (_I, [_P, _I, _P, _I, _ULL, _I, _P, _P]),
    "colo_env_pipeline_run_threads": (_I, [_P, _I, _P, _I, _ULL, _I, _P, _P]),
    "colo_env_pipeline_create": (_I, [_P, _I, C.POINTER(C.c_void_p)]),
    "colo_env_pipeline_run_queued": (_I, [_P, _P, _I, _ULL, _I, _P, _P, _I]),
    "colo_env_pipeline_destroy": (None, [_P]),
    "colo_env_stepper_create": (_I, [C.POINTER(MdpTables), C.POINTER(EnvBatch), _I, _P, C.POINTER(C.c_void_p)]),
    "colo_env_stepper_launch": (_I, [_P, _P, _ULL]),
    "colo_env_stepper_destroy": (None, [_P]),
    "colo_env_server_start": (_I, [C.POINTER(MdpTables), C.POINTER(EnvBatch), C.POINTER(EnvServer), _I, _ULL, _ULL, _P]),
    "colo_env_server_post": (_ULL, [C.POINTER(EnvServer)]),
    "colo_env_server_wait": (_I, [C.POINTER(EnvServer), _ULL, C.c_uint]),
    "colo_env_server_stop": (_I, [C.POINTER(EnvServer), _P]),
    "colo_qlearning_episodic_steps": (_I, [C.POINTER(MdpTables), C.POINTER(QLearningArgs), _I, _ULL, _P]),
    "colo_qlearning_continuous_steps": (_I, [C.POINTER(MdpTables), C.POINTER(QLearningArgs), _I, _ULL, _P]),
    "colo_psrl_episodic_steps": (_I, [C.POINTER(MdpTables), C.POINTER(PsrlArgs), _I, _ULL, _P]),
    "colo_ucrl2_steps": (_I, [C.POINTER(MdpTables), C.POINTER(Ucrl2Args), _LL, _P]),
    "colo_ucrl2_bounds": (_I, [C.POINTER(Ucrl2Args), _I, _I, _P, _I, _D, _D, _D, _I, _P, _P, _P]),
    "colo_ucrl2_model_update": (_I, [C.POINTER(Ucrl2Args), _I, _I, _P, _I, _P]),
    "colo_psrlc_steps": (_I, [C.POINTER(MdpTables), C.POINTER(PsrlcArgs), _LL, _P]),
    "colo_psrlc_sample_models": (_I, [C.POINTER(PsrlcArgs), _I, _I, _P, _I, _D, _I, C.c_float, _I, _P, _P, _P]),
    "colo_psrlc_finish_episode": (_I, [C.POINTER(PsrlcArgs), _I, _I, _P, _I, _P]),
    "colo_sample_nig_rewards": (_I, [_P, _LL, _LL, _ULL, _ULL, _P, _P]),
    "colo_sample_nn_rewards": (_I, [_P, _LL, _LL, _ULL, _ULL, _P, _P]),
    "colo_emit_noise": (_I, [_P, _P, _P, _LL, _I, _I, _I, _I, _D, _ULL, _ULL, _ULL, _P]),
    "colo_emit_observations": (_I, [_P, _P, _P, _P, _LL, _I, _I, _I, _P, _P]),
    "colo_build_dense_cdf": (_I, [_P, _I, _I, _I, _P, _I, _P]),
    "colo_build_cdf_index": (_I, [_P, _I, _I, _I, _I, _P, _P, _P]),
    "colo_count_cdf_breaks": (_I, [_P, _I, _I, _I, C.POINTER(C.c_int), _P]),
    "colo_build_cdf_breaks": (_I, [C.POINTER(MdpTables), _I, _P, _P]),
    "colo_extended_vi_work_bytes": (C.c_size_t, [_I, _I]),
    "colo_extended_vi_f32": (_I, [_P, _P, _P, _P, _I, _I, _D, _D, _LL, _P, _P, _P, _P, _P]),
    "colo_extended_vi_f64acc": (_I, [_P, _P, _P, _P, _I, _I, _D, _D, _LL, _P, _P, _P, _P, _P]),
    "colo_extended_vi_batched_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _D, _D, _LL, _P, _P, _P, _P, _P, _P]),
    "colo_extended_vi_batched_f64acc": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _D, _D, _LL, _P, _P, _P, _P, _P, _P]),
    "colo_sample_dirichlet_rows": (_I, [_P, _LL, _I, _LL, _ULL, _ULL, _P, _P]),
    "colo_sample_dirichlet_rows_fast": (_I, [_P, _LL, _I, _LL, _ULL, _ULL, _P, _P]),
    "colo_average_rewards_work_bytes": (C.c_size_t, [_I, _I]),
    "colo_average_rewards_f64": (_I, [_P, _P, _P, _I, _I, _I, _D, _I, _P, _P, _P, _P, _P]),
    "colo_policy_chain": (_I, [_P, _P, _P, _I, _I, _P, _P, _P]),
    "colo_stationary_distribution_work_bytes": (C.c_size_t, [_I]),
    "colo_stationary_distribution_f64": (_I, [_P, _I, _P, _D, _I, _P, _P, _P, _P]),
    "colo_lazy_transpose": (_I, [_P, _I, _P, _P]),
    "colo_power_iteration_work_bytes": (C.c_size_t, [_I]),
    "colo_power_iteration_f64": (_I, [_P, _I, _P, _D, _LL, _P, _P, _P, _P]),
    "colo_build_episodic_tensor": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "colo_build_continuous_form": (_I, [_P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "colo_synth_dense_rows": (_I, [_P, _P, _I, _I, _I, _I, _ULL, _P]),
}

_lib = None


def lib():
    """The loaded CUDA library.  Raises ColosseumB200Error if it has not been built (no fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ColosseumB200Error(
                f"{LIB_PATH} is missing: build it with `python -m colosseum_b200.build` "
                "(colosseum_b200 has no CPU or PyTorch fallback path)"
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)  # AttributeError here == header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def last_error():
    msg = lib().colo_last_error()
    return msg.decode() if msg else ""


def check(rc, what):
    """raise on CUDA / argument errors; pass the reference-level statuses (0..3) back to the caller"""
    if rc < 0:
        raise ColosseumB200Error(f"{what}: {last_error()} (rc={rc})")
    return rc


def ptr(t):
    """device pointer of a torch tensor (or None)"""
    return None if t is None else t.data_ptr()


def current_stream():
    """raw cudaStream_t of torch's current stream on the current device"""
    import torch

    return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise ColosseumB200Error("colosseum_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    lib()
