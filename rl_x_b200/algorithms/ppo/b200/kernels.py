"""Thin torch-tensor front end of the C-ABI entry points used by the PPO plugin (include/rlx_b200.h).
Every function here ends in exactly one native call; there is no alternative implementation behind it."""
import ctypes as C

import numpy as np
import torch

from rl_x_b200 import _native as nt


def _f32(t, name):
    if t is None:
        return None
    if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise TypeError(f"{name}: expected a contiguous float32 CUDA tensor, got {t.dtype} on {t.device} (contiguous={t.is_contiguous()})")
    return t.data_ptr()


def _bool_u8(t, name):
    if t is None:
        return None
    if not (t.is_cuda and t.dtype in (torch.bool, torch.uint8) and t.is_contiguous()):
        raise TypeError(f"{name}: expected a contiguous bool/uint8 CUDA tensor")
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class PpoKernels:
    """Binds the library for one (obs_dim, act_dim, hidden) network shape."""

    def __init__(self, obs_dim, act_dim, hidden):
        self.lib = nt.load()
        self.dims = nt.PpoDims(int(obs_dim), int(act_dim), int(hidden))
        self.obs_dim, self.act_dim, self.hidden = int(obs_dim), int(act_dim), int(hidden)
        n = self.lib.rlx_ppo_param_count(C.byref(self.dims))
        if n <= 0:
            raise RuntimeError(f"rl_x_b200: unsupported network shape obs={obs_dim} act={act_dim} hidden={hidden}: {nt.last_error()}")
        self.param_count = int(n)
        self.offsets, self.is_critic = nt.ppo_layout(obs_dim, act_dim, hidden)

    # ---------------------------------------------------------------------------------------------- workspaces
    def forward_workspace(self, n, device):
        nbytes = self.lib.rlx_ppo_forward_workspace_bytes(C.byref(self.dims), int(n))
        return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)

    def minibatch_workspace(self, m, device):
        nbytes = self.lib.rlx_ppo_minibatch_workspace_bytes(C.byref(self.dims), int(m))
        return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)

    # ------------------------------------------------------------------------------------------------ forward
    def forward(self, params, obs, workspace, **kw):
        nt.check(self.lib.rlx_ppo_forward_f32(C.byref(self.forward_args(params, obs, workspace, **kw)), _stream()), "rlx_ppo_forward_f32")

    def forward_prepared(self, a):
        nt.check(self.lib.rlx_ppo_forward_f32(C.byref(a), _stream()), "rlx_ppo_forward_f32")

    def forward_args(self, params, obs, workspace, *, noise=None, rng_seed=0, rng_offset=0, act_low=None, act_high=None,
                     clip_rescale=True, deterministic=False, action=None, env_action=None, logp=None, value=None):
        a = nt.PpoForwardArgs()
        a.dims = self.dims
        a.n = obs.shape[0]
        a.params = _f32(params, "params")
        a.obs = _f32(obs, "obs")
        a.noise = _f32(noise, "noise")
        a.rng_seed, a.rng_offset = int(rng_seed), int(rng_offset)
        a.act_low, a.act_high = _f32(act_low, "act_low"), _f32(act_high, "act_high")
        a.clip_rescale, a.deterministic = int(bool(clip_rescale)), int(bool(deterministic))
        a.action, a.env_action = _f32(action, "action"), _f32(env_action, "env_action")
        a.logp, a.value = _f32(logp, "logp"), _f32(value, "value")
        a.workspace, a.workspace_bytes = workspace.data_ptr(), workspace.numel()
        return a

    def critic_forward(self, params, obs, value, workspace):
        nt.check(self.lib.rlx_critic_forward_f32(C.byref(self.dims), _f32(params, "params"), _f32(obs, "obs"), obs.shape[0],
                                                 _f32(value, "value"), workspace.data_ptr(), workspace.numel(), _stream()),
                 "rlx_critic_forward_f32")

    def rollout_store(self, reward, terminated, truncated, next_obs, rewards_row, terminations_row, next_obs_dst, done_count, episode_stats=None):
        """episode_stats: (episode_return [n], episode_length [n], done_return_row [n], done_length_row [n]) or None."""
        n = reward.shape[0] if reward is not None else next_obs.shape[0]
        es = [_f32(t, "episode_stats") for t in episode_stats] if episode_stats is not None else [None] * 4
        nt.check(self.lib.rlx_rollout_store_stats_f32(_f32(reward, "reward"), _bool_u8(terminated, "terminated"), _bool_u8(truncated, "truncated"),
                                                      _f32(next_obs, "next_obs"), n, self.obs_dim, _f32(rewards_row, "rewards_row"),
                                                      _f32(terminations_row, "terminations_row"), _f32(next_obs_dst, "next_obs_dst"),
                                                      done_count.data_ptr() if done_count is not None else None, *es, _stream()),
                 "rlx_rollout_store_stats_f32")

    # ---------------------------------------------------------------------------------------------------- GAE
    def gae(self, rewards, terminations, values, gamma, gae_lambda, advantages, returns, next_values=None, last_value=None):
        T, N = rewards.shape
        nt.check(self.lib.rlx_gae_f32(_f32(rewards, "rewards"), _f32(terminations, "terminations"), _f32(values, "values"),
                                      _f32(next_values, "next_values"), _f32(last_value, "last_value"), T, N, float(gamma),
                                      float(gae_lambda), _f32(advantages, "advantages"), _f32(returns, "returns"), _stream()),
                 "rlx_gae_f32")

    # ------------------------------------------------------------------------------------------------- gather
    def gather(self, idx, states, actions, log_probs, advantages, returns, out_states, out_actions, out_log_probs,
               out_advantages, out_returns, count=None, out_states_ld=0):
        if not (idx.is_cuda and idx.dtype == torch.int64 and idx.is_contiguous()):
            raise TypeError("idx: expected a contiguous int64 CUDA tensor")
        count = idx.shape[0] if count is None else int(count)
        nt.check(self.lib.rlx_gather_minibatch_f32(idx.data_ptr(), count, self.obs_dim, self.act_dim, _f32(states, "states"),
                                                   _f32(actions, "actions"), _f32(log_probs, "log_probs"), _f32(advantages, "advantages"),
                                                   _f32(returns, "returns"), _f32(out_states, "out_states"), _f32(out_actions, "out_actions"),
                                                   _f32(out_log_probs, "out_log_probs"), _f32(out_advantages, "out_advantages"),
                                                   _f32(out_returns, "out_returns"), int(out_states_ld), _stream()), "rlx_gather_minibatch_f32")

    def advantage_stats(self, adv, count, mb, stats):
        nt.check(self.lib.rlx_advantage_stats_f32(_f32(adv, "adv"), int(count), int(mb), _f32(stats, "stats"), _stream()),
                 "rlx_advantage_stats_f32")

    def segment_moments(self, x, offsets, gsum, gcount, out):
        """offsets: int64 CUDA tensor [nseg+1]; gsum/gcount None -> segment sums, else centred sums of squares."""
        if not (offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()):
            raise TypeError("offsets: expected a contiguous int64 CUDA tensor")
        nt.check(self.lib.rlx_segment_moments_f32(_f32(x, "x"), offsets.data_ptr(), offsets.numel() - 1, _f32(gsum, "gsum"), _f32(gcount, "gcount"),
                                                  _f32(out, "out"), _stream()), "rlx_segment_moments_f32")

    # ------------------------------------------------------------------------------------------------- update
    def minibatch_args(self, *, m, m_global, states, actions, log_probs, advantages, returns, adv_stats, params, grads, exp_avg,
                       exp_avg_sq, lr, step_count, hp, metrics, workspace, states_ld=0, states_ones_col=False):
        a = nt.PpoMinibatchArgs()
        a.dims = self.dims
        a.m, a.m_global = int(m), int(m_global)
        a.states, a.actions = _f32(states, "states"), _f32(actions, "actions")
        a.log_probs, a.advantages, a.returns = _f32(log_probs, "log_probs"), _f32(advantages, "advantages"), _f32(returns, "returns")
        a.adv_stats = _f32(adv_stats, "adv_stats")
        a.params, a.grads = _f32(params, "params"), _f32(grads, "grads")
        a.exp_avg, a.exp_avg_sq = _f32(exp_avg, "exp_avg"), _f32(exp_avg_sq, "exp_avg_sq")
        a.lr = _f32(lr, "lr")
        a.step_count = step_count.data_ptr() if step_count is not None else None
        a.hp = hp
        a.metrics = _f32(metrics, "metrics")
        a.workspace, a.workspace_bytes = workspace.data_ptr(), workspace.numel()
        a.states_ld, a.states_ones_col = int(states_ld), int(bool(states_ones_col))
        return a

    def debug_gemm(self, engine, layout, epilogue, A, B, C, M, N, K, bias=None, aux=None):
        nt.check(self.lib.rlx_debug_gemm_f32(int(engine), int(layout), int(epilogue), M, N, K, _f32(A, "A"), A.stride(0), _f32(B, "B"), B.stride(0),
                                             _f32(C, "C"), C.stride(0), _f32(bias, "bias"), _f32(aux, "aux"), aux.stride(0) if aux is not None else 0,
                                             _stream()), "rlx_debug_gemm_f32")

    def states_pitch(self):
        """Row pitch (floats) of the gathered-states buffer: obs_dim plus a constant-one column, rounded up to 16 bytes."""
        return (self.obs_dim + 1 + 3) // 4 * 4

    def fwdbwd(self, args):
        nt.check(self.lib.rlx_ppo_minibatch_fwdbwd_f32(C.byref(args), _stream()), "rlx_ppo_minibatch_fwdbwd_f32")

    def clip_adam(self, args):
        nt.check(self.lib.rlx_gradnorm_clip_adam_f32(C.byref(args), _stream()), "rlx_gradnorm_clip_adam_f32")

    def update_epoch(self, first_args, count, mb):
        nt.check(self.lib.rlx_ppo_update_epoch_f32(C.byref(first_args), int(count), int(mb), _stream()), "rlx_ppo_update_epoch_f32")

    def update_epoch_sharded(self, first_args, counts, global_counts, comm):
        """counts / global_counts: contiguous int64 numpy arrays [num_mb]; comm: PeerComm."""
        assert counts.dtype == np.int64 and global_counts.dtype == np.int64 and len(counts) == len(global_counts)
        nt.check(self.lib.rlx_ppo_update_epoch_sharded_f32(C.byref(first_args), len(counts), counts.ctypes.data, global_counts.ctypes.data,
                                                           comm.handle, _stream()), "rlx_ppo_update_epoch_sharded_f32")


def make_hparams(clip_range, entropy_coef, critic_coef, max_grad_norm, beta1=0.9, beta2=0.999, eps=1e-8, ratio_delta_metric=False):
    """ratio_delta_metric: False = metrics[4] is the clip fraction (PPO); True / "mean" = mean |ratio - 1|; "median" = torch.median(|ratio - 1|) (ESPO)."""
    code = 2.0 if ratio_delta_metric == "median" else (1.0 if ratio_delta_metric else 0.0)
    return nt.PpoHparams(float(clip_range), float(entropy_coef), float(critic_coef), float(max_grad_norm), float(beta1), float(beta2),
                         float(eps), code)


class PeerComm:
    """The library's NVLink peer-memory gradient exchange (rlx_comm_*, include/rlx_b200.h; SURVEY.md §8 e).

    `dist` is an initialised torch.distributed module: it is used ONCE, to pass the 64-byte CUDA-IPC handles around and as the
    setup barrier; the all-reduces themselves are the library's own kernel.  Raises RuntimeError when the GPUs cannot map each
    other's memory (the caller may then fall back to NCCL)."""

    def __init__(self, dist, nfloats, device):
        self.lib = nt.load()
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        if self.world > nt.RLX_COMM_MAX_WORLD:
            raise RuntimeError(f"PeerComm supports up to {nt.RLX_COMM_MAX_WORLD} ranks")
        self.nfloats = int(nfloats)
        self.handle = C.c_void_p()
        with torch.cuda.device(device):
            nt.check(self.lib.rlx_comm_create(self.rank, self.world, self.nfloats, C.byref(self.handle)), "rlx_comm_create")
            mine = np.zeros(nt.RLX_COMM_HANDLE_BYTES, dtype=np.uint8)
            nt.check(self.lib.rlx_comm_export_handle(self.handle, mine.ctypes.data), "rlx_comm_export_handle")
            gathered = [torch.zeros(nt.RLX_COMM_HANDLE_BYTES, dtype=torch.uint8, device=device) for _ in range(self.world)]
            dist.all_gather(gathered, torch.from_numpy(mine).to(device))
            handles = np.ascontiguousarray(torch.stack(gathered).cpu().numpy())
            rc = self.lib.rlx_comm_connect(self.handle, handles.ctypes.data)
            ok = torch.tensor([1 if rc == 0 else 0], device=device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)  # every rank takes the same decision
            if int(ok.item()) == 0:
                err = self.lib.rlx_last_error_string().decode() if rc != 0 else "a peer rank could not map this rank's buffer"
                self.close()
                raise RuntimeError("PeerComm: " + err)

    def stage(self, src, n=None):
        """copies src into the slot the next all-reduce reads (the PPO epoch writes its gradient there directly instead)."""
        n = src.numel() if n is None else int(n)
        nt.check(self.lib.rlx_comm_stage_f32(self.handle, _f32(src, "src"), n, _stream()), "rlx_comm_stage_f32")

    def allreduce_sum(self, out, n=None):
        n = out.numel() if n is None else int(n)
        nt.check(self.lib.rlx_comm_allreduce_sum_f32(self.handle, _f32(out, "out"), n, _stream()), "rlx_comm_allreduce_sum_f32")

    def close(self):
        if self.handle:
            self.lib.rlx_comm_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
