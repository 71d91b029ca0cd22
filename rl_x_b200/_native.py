"""ctypes binding of the C-ABI library (include/rlx_b200.h).  No CPU fallback: if the library cannot be loaded or a call
fails, a RuntimeError is raised (the reference's Runner logs it and closes the envs, runner.py:340-352)."""
import ctypes as C
import os

import numpy as np

from . import build as _build

RLX_PPO_NSEG = 13
RLX_PPO_NMETRIC = 8
METRIC_NAMES = ("pg_loss", "critic_loss", "entropy_loss", "approx_kl", "clip_fraction", "policy_grad_norm", "critic_grad_norm", "count")

c_float_p = C.c_void_p  # raw device / host addresses are passed as integers


class PpoDims(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("hidden", C.c_int32)]


class Pcg64(C.Structure):
    _fields_ = [("s", C.c_uint64 * 6)]


class PpoForwardArgs(C.Structure):
    _fields_ = [
        ("dims", PpoDims),
        ("n", C.c_int64),
        ("params", C.c_void_p),
        ("obs", C.c_void_p),
        ("noise", C.c_void_p),
        ("rng_seed", C.c_uint64),
        ("rng_offset", C.c_uint64),
        ("act_low", C.c_void_p),
        ("act_high", C.c_void_p),
        ("clip_rescale", C.c_int32),
        ("deterministic", C.c_int32),
        ("action", C.c_void_p),
        ("env_action", C.c_void_p),
        ("logp", C.c_void_p),
        ("value", C.c_void_p),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_size_t),
    ]


class PpoHparams(C.Structure):
    _fields_ = [
        ("clip_range", C.c_float),
        ("entropy_coef", C.c_float),
        ("critic_coef", C.c_float),
        ("max_grad_norm", C.c_float),
        ("adam_beta1", C.c_float),
        ("adam_beta2", C.c_float),
        ("adam_eps", C.c_float),
        ("ratio_delta_metric", C.c_float),
    ]


class PpoMinibatchArgs(C.Structure):
    _fields_ = [
        ("dims", PpoDims),
        ("m", C.c_int64),
        ("m_global", C.c_int64),
        ("states", C.c_void_p),
        ("actions", C.c_void_p),
        ("log_probs", C.c_void_p),
        ("advantages", C.c_void_p),
        ("returns", C.c_void_p),
        ("adv_stats", C.c_void_p),
        ("params", C.c_void_p),
        ("grads", C.c_void_p),
        ("exp_avg", C.c_void_p),
        ("exp_avg_sq", C.c_void_p),
        ("lr", C.c_void_p),
        ("step_count", C.c_void_p),
        ("hp", PpoHparams),
        ("metrics", C.c_void_p),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_size_t),
        ("states_ld", C.c_int64),
        ("states_ones_col", C.c_int32),
        ("reserved2", C.c_int32),
    ]


class SacDims(C.Structure):
    _fields_ = [("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("hidden", C.c_int32), ("log_std_min", C.c_float), ("log_std_max", C.c_float)]


class SacUpdateArgs(C.Structure):
    _fields_ = [("dims", SacDims), ("batch", C.c_int64)] + [(n, C.c_void_p) for n in (
        "policy", "q", "log_alpha", "states", "next_states", "actions", "rewards", "terminations", "eps_next", "eps_cur", "act_low", "act_high")] + [
        ("gamma", C.c_float), ("tau", C.c_float), ("target_entropy", C.c_float), ("adam_beta1", C.c_float), ("adam_beta2", C.c_float),
        ("adam_eps", C.c_float)] + [(n, C.c_void_p) for n in (
        "g_policy", "m_policy", "v_policy", "g_q", "m_q", "v_q", "g_log_alpha", "m_log_alpha", "v_log_alpha", "lr", "steps", "metrics", "workspace")] + [
        ("workspace_bytes", C.c_size_t)]



class LstmDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("obs_dim", "act_dim", "hidden", "enc_dim", "lstm_dim", "options")]


class LstmMinibatchArgs(C.Structure):
    _fields_ = ([("dims", LstmDims), ("T", C.c_int64), ("n_env", C.c_int64)] +
                [(n, C.c_void_p) for n in ("states", "actions", "log_probs", "advantages", "returns", "dones", "init_c", "init_h", "adv_stats",
                                           "policy_params", "critic_params", "policy_grads", "critic_grads")] +
                [(n, C.c_float) for n in ("clip_range", "entropy_coef", "critic_coef", "reserved")] +
                [("metrics", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)])


class LstmStepArgs(C.Structure):
    _fields_ = ([("dims", LstmDims), ("n", C.c_int64)] +
                [(k, C.c_void_p) for k in ("obs", "c", "h", "noise", "policy_params", "critic_params", "act_low", "act_high")] +
                [("clip_rescale", C.c_int32), ("reserved", C.c_int32)] +
                [(k, C.c_void_p) for k in ("action", "env_action", "logp", "value", "workspace")] + [("workspace_bytes", C.c_size_t)])


RLX_LSTM_POLICY_NSEG, RLX_LSTM_CRITIC_NSEG = 22, 6
RLX_LSTM_OPT_FILM, RLX_LSTM_OPT_SHARED_ENCODER = 1, 2
LSTM_POLICY_SEGMENTS = ("We1", "be1", "g1", "n1", "We2", "be2", "g2", "n2", "Wi", "Wh", "bh", "gl", "nl", "Wt1", "bt1", "Wt2", "bt2", "Wm", "bm", "logstd",
                        "Wf", "bf")
LSTM_CRITIC_SEGMENTS = ("Wc1", "bc1", "Wc2", "bc2", "Wc3", "bc3")


RLX_FASTSAC_POLICY_NSEG, RLX_FASTSAC_Q_NSEG = 16, 14


class FastSacDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("obs_dim", "act_dim", "nr_atoms")]


class FastSacHparams(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("gamma", "tau", "v_min", "v_max", "target_entropy", "log_std_min", "log_std_max", "weight_decay",
                                         "adam_beta1", "adam_beta2", "adam_eps", "max_grad_norm", "clipped_double_q")]


class FastSacUpdateArgs(C.Structure):
    _fields_ = ([("dims", FastSacDims), ("n", C.c_int64)] +
                [(k, C.c_void_p) for k in ("states", "next_states", "actions", "rewards", "dones", "truncations", "effective_n_steps", "noise",
                                           "action_scale", "policy_params", "policy_grads", "policy_m", "policy_v", "q_params", "q_grads", "q_m", "q_v",
                                           "q_target_params", "log_alpha", "alpha_state", "lr", "steps")] +
                [("hp", FastSacHparams), ("metrics", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)])

RLX_SAC_NMETRIC = 12
RLX_COMM_MAX_WORLD = 16
RLX_COMM_HANDLE_BYTES = 64
SAC_METRIC_NAMES = ("entropy/alpha", "entropy/entropy", "gradients/policy_grad_norm", "gradients/critic_grad_norm", "gradients/entropy_grad_norm",
                    "loss/q_loss", "loss/policy_loss", "loss/entropy_loss", "q_value/q_value")

_SIGNATURES = {
    # name: (restype, argtypes)
    "rlx_version": (C.c_int, []),
    "rlx_last_error_string": (C.c_char_p, []),
    "rlx_set_aux_gemm_engine": (C.c_int, [C.c_int]),
    "rlx_aux_tc_gemm_count": (C.c_uint64, []),
    "rlx_launch_count": (C.c_uint64, []),
    "rlx_reset_launch_count": (None, []),
    "rlx_add_launch_count": (None, [C.c_uint64]),
    "rlx_timing_begin": (C.c_int, []),
    "rlx_timing_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "rlx_kernel_class_name": (C.c_char_p, [C.c_int]),
    "rlx_set_gemm_engine": (C.c_int, [C.c_int]),
    "rlx_set_head_engine": (C.c_int, [C.c_int]),
    "rlx_set_gae_tma": (C.c_int, [C.c_int]),
    "rlx_set_autocast_bf16": (C.c_int, [C.c_int]),
    "rlx_set_tc_pair": (C.c_int, [C.c_int, C.c_int]),
    "rlx_get_gemm_engine": (C.c_int, []),
    "rlx_pcg64_seed": (C.c_int, [C.c_uint64, C.POINTER(Pcg64)]),
    "rlx_pcg64_next64": (C.c_uint64, [C.POINTER(Pcg64)]),
    "rlx_pcg64_next32": (C.c_uint32, [C.POINTER(Pcg64)]),
    "rlx_pcg64_shuffle_i64": (C.c_int, [C.POINTER(Pcg64), C.c_void_p, C.c_int64]),
    "rlx_pcg64_integers_i64": (C.c_int, [C.POINTER(Pcg64), C.c_int64, C.c_void_p, C.c_int64]),
    "rlx_pcg64_choice_i64": (C.c_int, [C.POINTER(Pcg64), C.c_int64, C.c_int64, C.c_void_p]),
    "rlx_replay_sample_nstep_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p,
                                              C.c_int64, C.c_int64] + [C.c_void_p] * 15),
    "rlx_lstm_param_layout": (C.c_int, [C.POINTER(LstmDims), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "rlx_lstm_minibatch_workspace_bytes": (C.c_size_t, [C.POINTER(LstmDims), C.c_int64, C.c_int64]),
    "rlx_set_lstm_persistent": (C.c_int, [C.c_int]),
    "rlx_lstm_persistent_launch_count": (C.c_uint64, []),
    "rlx_lstm_ppo_minibatch_fwdbwd_f32": (C.c_int, [C.POINTER(LstmMinibatchArgs), C.c_void_p]),
    "rlx_lstm_step_f32": (C.c_int, [C.POINTER(LstmStepArgs), C.c_void_p]),
    "rlx_lstm_mask_carry_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "rlx_lstm_critic_forward_f32": (C.c_int, [C.POINTER(LstmDims), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rlx_mean_popstd_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rlx_optax_clip_adam_f32": (C.c_int, [C.c_void_p] * 4 + [C.c_int64, C.c_void_p, C.c_void_p] + [C.c_float] * 4 + [C.c_void_p] * 3),
    "rlx_gather_env_columns_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "rlx_fastsac_param_layout": (C.c_int, [C.POINTER(FastSacDims), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "rlx_fastsac_workspace_bytes": (C.c_size_t, [C.POINTER(FastSacDims), C.c_int64]),
    "rlx_fastsac_critic_update_f32": (C.c_int, [C.POINTER(FastSacUpdateArgs), C.c_void_p]),
    "rlx_fastsac_policy_update_f32": (C.c_int, [C.POINTER(FastSacUpdateArgs), C.c_void_p]),
    "rlx_fastsac_act_f32": (C.c_int, [C.POINTER(FastSacDims), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int64, C.c_void_p,
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "rlx_fastsac_normalize_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "rlx_ppo_param_count": (C.c_int64, [C.POINTER(PpoDims)]),
    "rlx_ppo_param_layout": (C.c_int, [C.POINTER(PpoDims), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "rlx_ppo_forward_workspace_bytes": (C.c_size_t, [C.POINTER(PpoDims), C.c_int64]),
    "rlx_ppo_forward_f32": (C.c_int, [C.POINTER(PpoForwardArgs), C.c_void_p]),
    "rlx_critic_forward_f32": (C.c_int, [C.POINTER(PpoDims), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rlx_rollout_store_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rlx_rollout_store_stats_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rlx_gae_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rlx_gather_minibatch_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64] + [C.c_void_p] * 10 + [C.c_int64, C.c_void_p]),
    "rlx_debug_gemm_f32": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "rlx_advantage_stats_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "rlx_segment_moments_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rlx_ppo_minibatch_workspace_bytes": (C.c_size_t, [C.POINTER(PpoDims), C.c_int64]),
    "rlx_ppo_minibatch_fwdbwd_f32": (C.c_int, [C.POINTER(PpoMinibatchArgs), C.c_void_p]),
    "rlx_gradnorm_clip_adam_f32": (C.c_int, [C.POINTER(PpoMinibatchArgs), C.c_void_p]),
    "rlx_ppo_update_epoch_f32": (C.c_int, [C.POINTER(PpoMinibatchArgs), C.c_int64, C.c_int64, C.c_void_p]),
    "rlx_comm_create": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_void_p)]),
    "rlx_comm_export_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rlx_comm_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rlx_comm_send_buffer": (C.c_void_p, [C.c_void_p]),
    "rlx_comm_stage_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "rlx_comm_allreduce_sum_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "rlx_comm_destroy": (C.c_int, [C.c_void_p]),
    "rlx_ppo_update_epoch_sharded_f32": (C.c_int, [C.POINTER(PpoMinibatchArgs), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rlx_replay_sample_gather_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64] + [C.c_void_p] * 10 + [C.c_void_p]),
    "rlx_polyak_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p]),
    "rlx_sac_policy_param_count": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "rlx_sac_q_param_count": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "rlx_sac_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int64]),
    "rlx_sac_act_f32": (C.c_int, [C.POINTER(SacDims), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rlx_sac_update_f32": (C.c_int, [C.POINTER(SacUpdateArgs), C.c_void_p]),
}

_lib = None


def library_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load (building in-tree first if needed) the native library.  Raises RuntimeError when impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if not os.path.exists(path) or (build_if_missing and not _build.is_fresh()):
        if not build_if_missing:
            raise RuntimeError(f"rl_x_b200: native library missing: {path} (run `python -m rl_x_b200.build`)")
        try:
            _build.build()
        except Exception as e:  # stale-but-present library is still usable on a box without nvcc
            if not os.path.exists(path):
                raise RuntimeError(f"rl_x_b200: cannot build native library: {e}") from e
    try:
        lib = C.CDLL(path)
    except OSError as e:
        raise RuntimeError(f"rl_x_b200: cannot load native library {path}: {e}") from e
    missing = []
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            missing.append(name)
            continue
        fn.restype = res
        fn.argtypes = args
    if missing:
        raise RuntimeError(f"rl_x_b200: native library lacks symbols: {missing}")
    # process-wide default of the FastSAC / PPO+LSTM GEMM engine (their configs say gemm_engine="auto" = leave it alone): lets a whole test
    # run or a bench leg select the tensor engine from outside, e.g. RLX_AUX_GEMM_ENGINE=1 python -m pytest tests/test_gpu_zzzz_fastsac.py
    if os.environ.get("RLX_AUX_GEMM_ENGINE", "") in ("0", "1"):
        lib.rlx_set_aux_gemm_engine(int(os.environ["RLX_AUX_GEMM_ENGINE"]))
    if os.environ.get("RLX_LSTM_PERSISTENT", "") in ("0", "1"):   # same idea for the one-launch-per-direction LSTM recurrence
        lib.rlx_set_lstm_persistent(int(os.environ["RLX_LSTM_PERSISTENT"]))
    _lib = lib
    return lib


def exported_symbols():
    return list(_SIGNATURES)


def last_error():
    return load().rlx_last_error_string().decode("utf-8", "replace")


def check(rc, what=""):
    if rc != 0:
        raise RuntimeError(f"rl_x_b200 native call failed ({what}, code {rc}): {last_error()}")


RLX_NKCLASS = 14


def timing_begin():
    check(load().rlx_timing_begin(), "rlx_timing_begin")


def timing_end():
    """{class name: dict(ms, launches, flops, bytes)} of everything launched since timing_begin()."""
    lib = load()
    ms, fl, by = (C.c_double * RLX_NKCLASS)(), (C.c_double * RLX_NKCLASS)(), (C.c_double * RLX_NKCLASS)()
    n = (C.c_uint64 * RLX_NKCLASS)()
    check(lib.rlx_timing_end(ms, n, fl, by), "rlx_timing_end")
    return {lib.rlx_kernel_class_name(i).decode(): dict(ms=ms[i], launches=int(n[i]), flops=fl[i], bytes=by[i]) for i in range(RLX_NKCLASS)}


def ptr(t):
    """Device/host address of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def stream_ptr(device=None):
    import torch

    if not torch.cuda.is_available():
        return None
    return torch.cuda.current_stream(device).cuda_stream


# ------------------------------------------------------------------------------------------------ host RNG (numpy-compatible)
class Pcg64Generator:
    """Restatement-free binding of the library's PCG64 stream; mirrors the subset of numpy.random.Generator the reference uses
    (`shuffle` ppo.py:276, `integers` sac/pytorch/replay_buffer.py:33-34, `choice` espo.py:256)."""

    def __init__(self, seed):
        self._lib = load()
        self.state = Pcg64()
        check(self._lib.rlx_pcg64_seed(C.c_uint64(int(seed)), C.byref(self.state)), "pcg64_seed")

    def shuffle(self, a):
        if not (isinstance(a, np.ndarray) and a.dtype == np.int64 and a.ndim == 1 and a.flags.c_contiguous):
            raise TypeError("shuffle expects a contiguous 1-D int64 numpy array")
        check(self._lib.rlx_pcg64_shuffle_i64(C.byref(self.state), a.ctypes.data, a.shape[0]), "pcg64_shuffle")

    def integers(self, high, size):
        out = np.empty(int(size), dtype=np.int64)
        check(self._lib.rlx_pcg64_integers_i64(C.byref(self.state), int(high), out.ctypes.data, out.shape[0]), "pcg64_integers")
        return out

    def choice(self, a, size, replace=False):
        """Generator.choice(int population, size, replace=False) (espo.py:256)."""
        if replace or not isinstance(a, (int, np.integer)):
            raise NotImplementedError("only choice(int, size, replace=False) is mirrored")
        out = np.empty(int(size), dtype=np.int64)
        check(self._lib.rlx_pcg64_choice_i64(C.byref(self.state), int(a), out.shape[0], out.ctypes.data), "pcg64_choice")
        return out

    def next_uint64(self):
        return int(self._lib.rlx_pcg64_next64(C.byref(self.state)))

    def next_uint32(self):
        return int(self._lib.rlx_pcg64_next32(C.byref(self.state)))


# ------------------------------------------------------------------------------------------------ layout helpers
SEGMENT_NAMES = ("W1p", "W1c", "b1p", "b1c", "W2p", "W2c", "b2p", "b2c", "W3p", "W3c", "b3p", "b3c", "logstd")


def ppo_layout(obs_dim, act_dim, hidden):
    lib = load()
    d = PpoDims(obs_dim, act_dim, hidden)
    off = (C.c_int64 * (RLX_PPO_NSEG + 1))()
    crit = (C.c_int32 * RLX_PPO_NSEG)()
    check(lib.rlx_ppo_param_layout(C.byref(d), off, crit), "ppo_param_layout")
    return list(off), list(crit)


def segment_shapes(obs_dim, act_dim, hidden):
    H, O, A = hidden, obs_dim, act_dim
    return {"W1p": (H, O), "W1c": (H, O), "b1p": (H,), "b1c": (H,), "W2p": (H, H), "W2c": (H, H), "b2p": (H,), "b2c": (H,),
            "W3p": (A, H), "W3c": (1, H), "b3p": (A,), "b3c": (1,), "logstd": (1, A)}


# reference state_dict key <-> segment (policy.py:45-52, critic.py:29-35)
POLICY_KEYS = {"policy_mean.0.weight": "W1p", "policy_mean.0.bias": "b1p", "policy_mean.2.weight": "W2p", "policy_mean.2.bias": "b2p",
               "policy_mean.4.weight": "W3p", "policy_mean.4.bias": "b3p", "policy_logstd": "logstd"}
CRITIC_KEYS = {"critic.0.weight": "W1c", "critic.0.bias": "b1c", "critic.2.weight": "W2c", "critic.2.bias": "b2c",
               "critic.4.weight": "W3c", "critic.4.bias": "b3c"}
