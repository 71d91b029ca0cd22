"""PPO with the reference's plugin surface (rl_x/algorithms/ppo/pytorch/ppo.py), executed by hand-written sm_100a kernels.

Same constructor / train / test / save / load / general_properties contract and the same metric names as the reference
class `PPO` (ppo.py:22-486).  What differs is where the work happens:

  reference (ppo.py)                                   this build
  ---------------------------------------------------  -------------------------------------------------------------
  acting: 2 compiled modules + ~10 kernels + .item()   1 native call per step (3 kernels) + 1 store kernel, no host sync
          per step (:203-246)
  next_values: critic over all next_states (:253-254)  TORCH envs: one critic pass over the last next_state (SURVEY §8 a5)
  GAE: TorchScript loop over T (:110-118)              1 kernel, bit-exact
  shuffle: numpy Generator.shuffle on host (:276)      same PCG64 stream restated in C (bit-exact), overlapped with GPU work
  6 index-gathers + 7 .item() per minibatch (:283-294) 1 gather per epoch; whole epoch launched from C; 1 metrics D2H/iteration
  autograd + clip_grad_norm_ + Adam (:121-166)         fused GEMM / loss / clip+Adam kernels on one flat parameter buffer
  single device                                        env-sharded data parallel, one NCCL all-reduce per minibatch

There is no CPU path: a missing CUDA device or native library raises.
"""
import logging
import os
import time
from collections import deque

import numpy as np
import torch
import torch.nn as nn

from rl_x_b200 import _native as nt
from rl_x_b200.algorithms.ppo.b200.batch import Batch
from rl_x_b200.algorithms.ppo.b200.general_properties import GeneralProperties
from rl_x_b200.algorithms.ppo.b200.kernels import PeerComm, PpoKernels, make_hparams
from rl_x_b200.algorithms.ppo.b200 import sharding
from rl_x_b200.environments.types import DataInterfaceType, same_member

rlx_logger = logging.getLogger("rl_x")


def init_reference_parameters(obs_dim, act_dim, hidden, std_dev, seed):
    """Initial weights bit-identical to the reference for the same seed: torch.manual_seed(seed) (ppo.py:73), then the
    policy's three nn.Linear layers (constructor init followed by orthogonal_/constant_, policy.py:45-58) and the critic's
    (critic.py:29-41), created on the CPU in that order.  Returns {reference state_dict key: tensor}."""
    torch.manual_seed(seed)

    def layer(i, o, std):
        lin = nn.Linear(i, o)
        nn.init.orthogonal_(lin.weight, std)
        nn.init.constant_(lin.bias, 0.0)
        return lin

    out = {}
    pol = [layer(obs_dim, hidden, np.sqrt(2)), layer(hidden, hidden, np.sqrt(2)), layer(hidden, act_dim, 0.01)]
    for idx, lin in zip((0, 2, 4), pol):
        out[f"policy_mean.{idx}.weight"], out[f"policy_mean.{idx}.bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
    out["policy_logstd"] = torch.full((1, act_dim), np.log(std_dev).item())
    cri = [layer(obs_dim, hidden, np.sqrt(2)), layer(hidden, hidden, np.sqrt(2)), layer(hidden, 1, 1.0)]
    for idx, lin in zip((0, 2, 4), cri):
        out[f"critic.{idx}.weight"], out[f"critic.{idx}.bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
    return out


# torch.optim.Adam(module.parameters()) numbers the parameters in nn.Module.parameters() order: the module's OWN Parameters first
# (policy_logstd, reference policy.py:52), then the children's (policy_mean.0.weight, ...).  state_dict() uses the same order.  The
# reference modules are torch.compile wrappers (policy.py:27, critic.py:19): the installed torch strips their "_orig_mod." prefix in
# state_dict() (what the executed reference wrote here: tests/golden/ppo_ref_checkpoint.model), older builds kept it - load accepts both,
# save writes the bare names like the installed torch.
POLICY_PARAM_ORDER = ("policy_logstd", "policy_mean.0.weight", "policy_mean.0.bias", "policy_mean.2.weight", "policy_mean.2.bias",
                      "policy_mean.4.weight", "policy_mean.4.bias")
CRITIC_PARAM_ORDER = ("critic.0.weight", "critic.0.bias", "critic.2.weight", "critic.2.bias", "critic.4.weight", "critic.4.bias")
COMPILED_PREFIX = "_orig_mod."


class FlatParameters:
    """One flat fp32 device buffer for policy + critic (layout: include/rlx_b200.h), with named views that carry the
    reference's state_dict keys so checkpoints interoperate (ppo.py:426-451)."""

    def __init__(self, kernels, device):
        self.k = kernels
        self.flat = torch.zeros(kernels.param_count, dtype=torch.float32, device=device)
        self.shapes = nt.segment_shapes(kernels.obs_dim, kernels.act_dim, kernels.hidden)

    def view(self, flat, seg):
        i = nt.SEGMENT_NAMES.index(seg)
        return flat[self.k.offsets[i]:self.k.offsets[i + 1]].view(self.shapes[seg])

    def load_named(self, named, flat=None):
        flat = self.flat if flat is None else flat
        for keys in (nt.POLICY_KEYS, nt.CRITIC_KEYS):
            for key, seg in keys.items():
                src = named[key] if key in named else named["_orig_mod." + key]  # torch.compile'd reference modules prefix keys
                self.view(flat, seg).copy_(torch.as_tensor(src, dtype=torch.float32).reshape(self.shapes[seg]))

    def state_dicts(self, flat=None, prefix=""):
        """(policy, critic) dicts in the reference's state_dict() order; prefix="_orig_mod." gives the compiled modules' keys."""
        flat = self.flat if flat is None else flat
        pol = {prefix + key: self.view(flat, nt.POLICY_KEYS[key]).detach().cpu().clone() for key in POLICY_PARAM_ORDER}
        cri = {prefix + key: self.view(flat, nt.CRITIC_KEYS[key]).detach().cpu().clone() for key in CRITIC_PARAM_ORDER}
        return pol, cri

    def adam_state_dict(self, order, keys, exp_avg, exp_avg_sq, step, lr):
        """torch.optim.Adam.state_dict() of the reference's optimiser over one net (ppo.py:83-84,426-436): parameter i is order[i]."""
        state = {i: {"step": torch.tensor(float(step)), "exp_avg": self.view(exp_avg, keys[key]).detach().cpu().clone(),
                     "exp_avg_sq": self.view(exp_avg_sq, keys[key]).detach().cpu().clone()} for i, key in enumerate(order)}
        group = {"lr": lr, "betas": (0.9, 0.999), "eps": 1e-08, "weight_decay": 0, "amsgrad": False, "maximize": False, "foreach": None,
                 "capturable": False, "differentiable": False, "fused": None, "decoupled_weight_decay": False, "params": list(range(len(order)))}
        return {"state": state, "param_groups": [group]}

    def load_adam_state(self, opt_state, order, keys, exp_avg, exp_avg_sq):
        """Inverse of adam_state_dict for a checkpoint written by the reference or by save().  Returns the step count; a parameter whose
        moment shape does not match the layout raises (a silently permuted optimiser state is worse than no state)."""
        st, step = opt_state["state"], 0.0
        for i, key in enumerate(order):
            if i not in st:
                continue  # the reference saves an empty state before the first optimiser step
            seg = keys[key]
            for name, dst in (("exp_avg", exp_avg), ("exp_avg_sq", exp_avg_sq)):
                src = torch.as_tensor(st[i][name], dtype=torch.float32)
                if tuple(src.shape) != tuple(self.shapes[seg]):
                    raise ValueError(f"optimizer state {i} ({key}): {name} has shape {tuple(src.shape)}, expected {tuple(self.shapes[seg])}")
                self.view(dst, seg).copy_(src)
            step = max(step, float(st[i]["step"]))
        return step


class PermutationStream:
    """Background producer of the epoch permutations (ppo.py:273-276).

    The permutation sequence depends only on the PCG64 stream and the batch size — never on data — so it is generated ahead of
    time on a host thread (the native shuffle releases the GIL) into pinned staging slots while the GPU is busy with the rollout
    and the previous epochs.  Order of RNG consumption is exactly the reference's: per iteration one np.arange(B), then nr_epochs
    successive in-place shuffles.  For the env-sharded update the thread also extracts the rows this rank owns."""

    def __init__(self, rng, batch_size, nr_epochs, slot_rows, transform=None, depth_iterations=2):
        import queue
        import threading
        self.rng, self.B, self.E, self.transform = rng, int(batch_size), int(nr_epochs), transform
        self.nslots = max(2, depth_iterations) * self.E
        pool = torch.zeros(self.nslots, max(int(slot_rows), 1), dtype=torch.int64).pin_memory()  # one pinned allocation
        self.slots = [pool[i] for i in range(self.nslots)]
        self.free = queue.Queue()
        for i in range(self.nslots):
            self.free.put(i)
        self.ready = queue.Queue()
        self.stop = False
        self.error = None
        self.thread = threading.Thread(target=self._run, name="rlx-permutations", daemon=True)
        self.thread.start()

    def _run(self):
        try:
            while not self.stop:
                idx = np.arange(self.B)  # int64, re-created every iteration (ppo.py:273)
                for _ in range(self.E):
                    slot = self.free.get()
                    if slot is None or self.stop:
                        return
                    self.rng.shuffle(idx)
                    if self.transform is None:
                        self.slots[slot].numpy()[:] = idx
                        self.ready.put((slot, self.B, None))
                    else:
                        local_idx, counts = self.transform(idx)
                        self.slots[slot].numpy()[:local_idx.shape[0]] = local_idx
                        self.ready.put((slot, int(local_idx.shape[0]), counts))
        except Exception as e:  # surfaced to the training thread
            self.error = e
            self.ready.put(None)

    def next(self):
        item = self.ready.get()
        if item is None:
            raise RuntimeError(f"permutation thread failed: {self.error}")
        slot, count, counts = item
        return slot, self.slots[slot], count, counts

    def release(self, slots):
        for s_ in slots:
            self.free.put(s_)

    def close(self):
        self.stop = True
        self.free.put(None)


class PPO:
    def __init__(self, config, train_env, eval_env, run_path, writer):
        self.config = config
        self.train_env = train_env
        self.eval_env = eval_env
        self.writer = writer

        self.save_model = config.runner.save_model
        self.save_path = os.path.join(run_path, "models")
        self.track_console = config.runner.track_console
        self.track_tb = config.runner.track_tb
        self.track_wandb = config.runner.track_wandb
        self.seed = config.environment.seed
        self.total_timesteps = config.algorithm.total_timesteps
        self.nr_envs = config.environment.nr_envs
        self.learning_rate = config.algorithm.learning_rate
        self.anneal_learning_rate = config.algorithm.anneal_learning_rate
        self.nr_steps = config.algorithm.nr_steps
        self.nr_epochs = config.algorithm.nr_epochs
        self.minibatch_size = config.algorithm.minibatch_size
        self.gamma = config.algorithm.gamma
        self.gae_lambda = config.algorithm.gae_lambda
        self.clip_range = config.algorithm.clip_range
        self.entropy_coef = config.algorithm.entropy_coef
        self.critic_coef = config.algorithm.critic_coef
        self.max_grad_norm = config.algorithm.max_grad_norm
        self.std_dev = config.algorithm.std_dev
        self.action_clipping_and_rescaling = config.algorithm.action_clipping_and_rescaling
        self.nr_hidden_units = config.algorithm.nr_hidden_units
        self.evaluation_frequency = config.algorithm.evaluation_frequency
        self.evaluation_episodes = config.algorithm.evaluation_episodes

        # ---- data-parallel topology: one process per GPU, envs sharded over ranks (SURVEY §8 e)
        import torch.distributed as dist
        self.dist = dist if (dist.is_available() and dist.is_initialized()) else None
        if config.algorithm.get("ignore_process_group", False):
            self.dist = None  # a single-GPU instance inside a multi-rank job (bench.py's sharded-vs-single parity check)
        self.world_size = self.dist.get_world_size() if self.dist else 1
        self.rank = self.dist.get_rank() if self.dist else 0
        self.global_nr_envs = self.nr_envs * self.world_size
        self.batch_size = self.global_nr_envs * self.nr_steps          # global batch (ppo.py:54)
        self.local_batch_size = self.nr_envs * self.nr_steps
        self.nr_minibatches = self.batch_size // self.minibatch_size   # ppo.py:55
        self.exact_global_permutation = bool(config.algorithm.get("exact_global_permutation", True))
        self.gradient_exchange = str(config.algorithm.get("gradient_exchange", "peer"))  # "peer": library kernel over NVLink; "nccl"
        if self.gradient_exchange not in ("peer", "nccl"):
            raise ValueError("gradient_exchange must be 'peer' or 'nccl'")
        if str(config.algorithm.get("peer_exchange_algorithm", "auto")) not in ("auto", "one_shot"):
            raise ValueError("peer_exchange_algorithm must be 'auto' or 'one_shot': the one-shot kernel is the only peer all-reduce "
                             "(the two-shot kernel was removed)")
        self.peer_comm = None
        self._seg_cache = None

        if self.evaluation_frequency % (self.nr_steps * self.nr_envs) != 0 and self.evaluation_frequency != -1:
            raise ValueError("Evaluation frequency must be a multiple of the number of steps and environments.")
        # the reference's mixed-precision mode (ppo.py:98-107,123,155,208,253): autocast(bf16) around acting, next-values and both loss
        # functions.  Here: the same roundings inside the kernels, bf16 values carried in fp32 storage, one tensor-core pass per product
        # (rlx_set_autocast_bf16).  Single GPU for now: the sharded update would round every rank's partial gradient instead of the sum.
        self.bf16_mixed_precision_training = bool(config.algorithm.get("bf16_mixed_precision_training", False))
        if self.bf16_mixed_precision_training and self.world_size > 1:
            raise NotImplementedError("rl_x_b200 PPO: bf16_mixed_precision_training is single-GPU in this build.")
        if config.algorithm.device != "gpu" or not torch.cuda.is_available():
            raise RuntimeError("rl_x_b200 PPO needs a CUDA device (algorithm.device=gpu); there is no CPU fallback.")
        self.device = torch.device("cuda", torch.cuda.current_device())
        rlx_logger.info(f"Using device: {self.device}")

        # Replicas must start from identical weights and (reference-exact mode) walk one permutation stream: both derive from RANK 0's
        # seed, whatever per-rank environment.seed the launcher used to decorrelate the env streams.
        self.model_seed = int(self.seed)
        if self.dist:
            t = torch.tensor([self.model_seed], dtype=torch.int64, device=self.device)
            self.dist.broadcast(t, src=0)
            self.model_seed = int(t.item())
        self.rng = nt.Pcg64Generator(self.model_seed)  # np.random.default_rng(self.seed), ppo.py:72

        self.os_shape = self.train_env.single_observation_space.shape
        self.as_shape = self.train_env.single_action_space.shape
        if len(self.os_shape) != 1 or len(self.as_shape) != 1:
            raise ValueError("rl_x_b200 PPO supports flat observations and flat continuous actions only.")
        obs_dim, act_dim = int(self.os_shape[0]), int(self.as_shape[0])
        for attr in ("policy_observation_indices", "critic_observation_indices"):
            ind = getattr(self.train_env, attr, None)
            if ind is not None and not np.array_equal(np.asarray(ind), np.arange(obs_dim)):
                raise ValueError(f"rl_x_b200 PPO does not implement a non-identity {attr} (policy.py:14, critic.py:10).")

        self.kernels = PpoKernels(obs_dim, act_dim, self.nr_hidden_units)
        engine = config.algorithm.get("gemm_engine", "auto")
        lib = self.kernels.lib
        lib.rlx_set_gemm_engine({"simt": 0, "tcgen05": 1, "auto": 1}[engine])
        self.params = FlatParameters(self.kernels, self.device)
        self.params.load_named(init_reference_parameters(obs_dim, act_dim, self.nr_hidden_units, self.std_dev, self.model_seed))
        if self.dist:
            self.dist.broadcast(self.params.flat, src=0)  # bit-identical replicas even if a rank's torch build initialises differently
        P = self.kernels.param_count
        self.exp_avg = torch.zeros(P, dtype=torch.float32, device=self.device)
        self.exp_avg_sq = torch.zeros(P, dtype=torch.float32, device=self.device)
        self.grads = torch.zeros(P + nt.RLX_PPO_NMETRIC, dtype=torch.float32, device=self.device)  # metrics ride in the tail (one all-reduce)
        if self.world_size > 1 and self.gradient_exchange == "peer" and self.peer_comm is None:
            try:
                self.peer_comm = PeerComm(self.dist, P + nt.RLX_PPO_NMETRIC, self.device)
            except RuntimeError as err:  # GPUs without peer access: NCCL carries the gradient instead (slower, same numbers up to sum order)
                rlx_logger.warning(f"{err}; falling back to gradient_exchange='nccl'")
                self.gradient_exchange = "nccl"
        self.adam_step = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.lr_dev = torch.full((1,), float(self.learning_rate), dtype=torch.float32, device=self.device)
        self.lr_iteration = 0
        self.hp = self._make_hparams()

        low = np.asarray(torch.as_tensor(self.train_env.single_action_space.low).cpu(), dtype=np.float32).reshape(-1)
        high = np.asarray(torch.as_tensor(self.train_env.single_action_space.high).cpu(), dtype=np.float32).reshape(-1)
        self.env_as_low = torch.from_numpy(np.broadcast_to(low, (act_dim,)).copy()).to(self.device)
        self.env_as_high = torch.from_numpy(np.broadcast_to(high, (act_dim,)).copy()).to(self.device)

        self.is_torch_data_interface = same_member(self.train_env.general_properties.data_interface_type, DataInterfaceType.TORCH)
        self.rollout_noise = config.algorithm.get("rollout_noise", "philox")
        self.noise_seed = (int(self.seed) * 0x9E3779B1 + 0x7F4A7C15 * self.rank) & 0xFFFFFFFFFFFFFFFF
        self.noise_offset = 0

        if self.save_model:
            os.makedirs(self.save_path)
            self.best_mean_return = -np.inf
        self._alloc_done = False

    # ------------------------------------------------------------------------------------------------ buffers
    def _allocate(self):
        if self._alloc_done:
            return
        dev, T, N = self.device, self.nr_steps, self.nr_envs
        obs, act = self.kernels.obs_dim, self.kernels.act_dim
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
        self.batch = Batch(
            states=z(T + 1, N, obs),
            next_states=None if self.is_torch_data_interface else z(T, N, obs),
            actions=z(T, N, act), rewards=z(T, N), values=z(T, N), terminations=z(T, N), log_probs=z(T, N),
            advantages=z(T, N), returns=z(T, N),
        )
        self.env_action = z(N, act)
        self.last_value = z(N)
        self.next_values = None if self.is_torch_data_interface else z(T, N)
        self.done_count = torch.zeros(1, dtype=torch.int64, device=dev)
        Bl = self.local_batch_size
        # gathered states carry a constant-one column (pitch rounded to 16 B): the tensor-core dW1 GEMM emits db1 from it
        self.ldx = self.kernels.states_pitch()
        self.g_states, self.g_actions = z(Bl, self.ldx), z(Bl, act)
        self.g_log_probs, self.g_advantages, self.g_returns = z(Bl), z(Bl), z(Bl)
        self.perm_dev = torch.zeros(Bl, dtype=torch.int64, device=dev)
        self._perm_stream = None
        self._perm_slots_in_flight = []
        self.nmb_epoch = -(-self.batch_size // self.minibatch_size)  # ceil: a short last minibatch is processed (ppo.py:277-279)
        self.adv_stats = z(self.nmb_epoch, 2)
        self.seg_tmp = z(2, -(-self.nmb_epoch // 4) * 4)  # rows padded to 16 bytes: rlx_comm_allreduce_sum_f32 wants an aligned destination
        self.metrics_dev = z(self.nr_epochs * self.nmb_epoch, nt.RLX_PPO_NMETRIC)
        self.metrics_host = torch.zeros(self.nr_epochs * self.nmb_epoch, nt.RLX_PPO_NMETRIC).pin_memory()
        self.ev_dev = z(4)
        self.fwd_ws = self.kernels.forward_workspace(max(N, 1) if self.is_torch_data_interface else T * N, dev)
        mb_rows = min(self.minibatch_size, self.batch_size)
        if self.world_size > 1:
            mb_rows = min(mb_rows, Bl)  # a rank can own at most all of its rows in one minibatch
        self.train_ws = self.kernels.minibatch_workspace(mb_rows, dev)
        self.lr_host = torch.zeros(1, dtype=torch.float32).pin_memory()
        if not self.is_torch_data_interface:
            # pinned staging, double-buffered so that step t+1 can be staged while the copies of step t are still in flight
            self.h_action = torch.zeros(N, act).pin_memory()
            self.h_obs = [torch.zeros(N, obs).pin_memory() for _ in range(2)]
            # reward | terminated | truncated of one step travel as ONE packed copy (4N + N + N bytes) instead of three tiny ones
            self.h_pack = [torch.zeros(6 * N, dtype=torch.uint8).pin_memory() for _ in range(2)]
            self.h_pack_np = [(p.numpy()[:4 * N].view(np.float32), p.numpy()[4 * N:5 * N].view(np.bool_), p.numpy()[5 * N:].view(np.bool_))
                              for p in self.h_pack]
            self.h_done_idx = [torch.zeros(N, dtype=torch.int64).pin_memory() for _ in range(2)]   # finished episodes of one step:
            self.h_finals = [torch.zeros(N, obs).pin_memory() for _ in range(2)]                   # env indices and final observations
            self.d_done_idx = torch.zeros(N, dtype=torch.int64, device=dev)
            self.d_finals = z(N, obs)
            self.h2d_done = [torch.cuda.Event() for _ in range(2)]
            self.h2d_pending = [False, False]
            self.action_ready = torch.cuda.Event()
            self.d_pack = torch.zeros(6 * N, dtype=torch.uint8, device=dev)
            self.d_reward = self.d_pack[:4 * N].view(torch.float32)
            self.d_term = self.d_pack[4 * N:5 * N].view(torch.bool)
            self.d_trunc = self.d_pack[5 * N:].view(torch.bool)
            self.d_obs = z(N, obs)
        self.noise_buf = z(N, act) if self.rollout_noise == "torch" else None
        # device-side episode statistics for TORCH-interface envs (SURVEY.md §8 f1; semantics of warp_torch/environment.py:159-178 and
        # wrappers.py:15-33): running return / length per env, and per rollout step the return / length of the episodes that ended there.
        # Read back ONCE per iteration with the metric records - no per-step .cpu() as in the reference's wrapper.
        self.device_episode_stats = self.is_torch_data_interface and bool(self.config.algorithm.get("device_episode_statistics", True))
        if self.device_episode_stats:
            self.ep_return, self.ep_length = z(N), z(N)
            self.done_stats_dev = z(2, T, N)   # [0] finished-episode return, [1] finished-episode length (0 = none ended)
            self.done_stats_host = torch.zeros(2, T, N).pin_memory()
        b = self.batch
        self._fwd_args = [self.kernels.forward_args(self.params.flat, b.states[t], self.fwd_ws, rng_seed=self.noise_seed, act_low=self.env_as_low,
                                                    act_high=self.env_as_high, clip_rescale=self.action_clipping_and_rescaling,
                                                    action=b.actions[t], env_action=self.env_action, logp=b.log_probs[t], value=b.values[t])
                          for t in range(T)]
        self._store_rows = [(b.rewards[t], b.terminations[t], b.states[t + 1]) for t in range(T)]
        self._stat_rows = ([(self.ep_return, self.ep_length, self.done_stats_dev[0, t], self.done_stats_dev[1, t]) for t in range(T)]
                           if self.device_episode_stats else [None] * T)
        self._alloc_done = True

    # ------------------------------------------------------------------------------------------------- acting
    def _policy_step(self, state, step):
        """ref: policy.get_action_logprob + critic.get_value + buffer writes of action/value/log_prob (ppo.py:207-209,233,238,243)."""
        noise = self._draw_noise(step)
        a = self._fwd_args[step]  # pointer table of this rollout slot, built once (the buffers never move)
        a.noise = noise.data_ptr() if noise is not None else None
        a.rng_offset = self.noise_offset
        self.kernels.forward_prepared(a)
        self.noise_offset += 1

    def _draw_noise(self, step):
        """Standard-normal draws for Normal.sample() (policy.py:66).  None = in-kernel Philox stream; `rollout_noise=torch`
        injects torch.randn draws; tests override this hook to teacher-force the reference's samples."""
        if self.noise_buf is not None:
            return self.noise_buf.normal_()
        return None

    @staticmethod
    def _as_host_tensor(x, dtype):
        t = torch.from_numpy(np.ascontiguousarray(x, dtype=dtype))
        return t

    def _h2d(self, src_np, dtype, staging, dst):
        """Host -> device copy of one env output.  Arrays that already live in pinned memory (e.g. a simulator's own staging
        buffers) are copied directly; pageable arrays go through this step's pinned slot first."""
        t = self._as_host_tensor(src_np, dtype)
        if t.is_pinned():
            dst.copy_(t, non_blocking=True)
        else:
            staging.copy_(t)
            dst.copy_(staging, non_blocking=True)

    def _to_device_obs(self, obs_np, dst, slot=0):
        self._h2d(obs_np, np.float32, self.h_obs[slot], dst)

    def _collect_rollout(self, state_is_in_slot0):
        """ref: the acting loop, ppo.py:203-246."""
        b, env, T = self.batch, self.train_env, self.nr_steps
        step_info_collection = {}
        saving_returns = []
        dones_host = 0
        self.done_count.zero_()
        for step in range(T):
            state = b.states[step]
            self._policy_step(state, step)
            if self.is_torch_data_interface:
                next_state, reward, terminated, truncated, info = env.step(self.env_action)
                if reward.dtype != torch.float32:
                    reward = reward.float()
                terminated = terminated if terminated.dtype == torch.bool else terminated.bool()
                truncated = truncated if truncated.dtype == torch.bool else truncated.bool()
                rr, tr, ns = self._store_rows[step]
                self.kernels.rollout_store(reward.contiguous(), terminated.contiguous(), truncated.contiguous(), next_state.contiguous(),
                                           rr, tr, ns, self.done_count, self._stat_rows[step])
            else:
                self.h_action.copy_(self.env_action, non_blocking=True)
                self.action_ready.record()
                self.action_ready.synchronize()  # the simulator needs the actions on the host (ppo.py:211-213)
                next_state, reward, terminated, truncated, info = env.step(self.h_action.numpy())
                slot = step & 1
                if self.h2d_pending[slot]:
                    self.h2d_done[slot].synchronize()  # the pinned slot of step-2 must have been consumed
                self._h2d(next_state, np.float32, self.h_obs[slot], b.states[step + 1])
                h_reward, h_term, h_trunc = self.h_pack_np[slot]
                np.copyto(h_reward, reward, casting="same_kind")
                np.copyto(h_term, terminated, casting="unsafe")
                np.copyto(h_trunc, truncated, casting="unsafe")
                self.d_pack.copy_(self.h_pack[slot], non_blocking=True)
                # next_states[step] = next_state with final observations patched in for finished episodes (ppo.py:217-223)
                self.kernels.rollout_store(self.d_reward, self.d_term, self.d_trunc, b.states[step + 1], b.rewards[step],
                                           b.terminations[step], b.next_states[step], None)
                # Host-side bookkeeping of finished episodes runs while the copies above are in flight; nothing below blocks the host, so
                # the next step's kernels are queued behind the copies instead of being launched after them.
                done = np.logical_or(terminated, truncated)
                if done.any():
                    idx = np.nonzero(done)[0]
                    k = len(idx)
                    batch_getter = getattr(env, "get_final_observations_batch", None)  # optional vectorised form of the per-index call
                    if batch_getter is not None:
                        finals = np.asarray(batch_getter(info, idx), dtype=np.float32)
                    else:
                        finals = np.stack([np.asarray(env.get_final_observation_at_index(info, int(i)), dtype=np.float32) for i in idx])
                    # next_states[step][idx] = finals, staged through this step's pinned slot (stream order keeps it after rollout_store)
                    self.h_done_idx[slot][:k].copy_(torch.from_numpy(idx))
                    self.h_finals[slot][:k].copy_(torch.from_numpy(np.ascontiguousarray(finals)))
                    self.d_done_idx[:k].copy_(self.h_done_idx[slot][:k], non_blocking=True)
                    self.d_finals[:k].copy_(self.h_finals[slot][:k], non_blocking=True)
                    b.next_states[step].index_copy_(0, self.d_done_idx[:k], self.d_finals[:k])
                    values_getter = getattr(env, "get_final_info_values_batch", None)
                    if values_getter is not None:
                        saving_returns.extend(values_getter(info, "episode_return", idx))
                    else:
                        for i in idx:
                            saving_returns.append(env.get_final_info_value_at_index(info, "episode_return", int(i)))
                    dones_host += k
                self.h2d_done[slot].record()
                self.h2d_pending[slot] = True
            for key, info_value in env.get_logging_info_dict(info).items():
                step_info_collection.setdefault(key, []).extend(info_value)
        return step_info_collection, saving_returns, dones_host

    # ------------------------------------------------------------------------------------ advantages / returns
    def _compute_advantages(self):
        """ref: ppo.py:253-258."""
        b, k = self.batch, self.kernels
        if self.is_torch_data_interface:
            k.critic_forward(self.params.flat, b.states[self.nr_steps], self.last_value, self.fwd_ws)
            k.gae(b.rewards, b.terminations, b.values, self.gamma, self.gae_lambda, b.advantages, b.returns, last_value=self.last_value)
        else:
            k.critic_forward(self.params.flat, b.next_states.view(-1, k.obs_dim), self.next_values.view(-1), self.fwd_ws)
            k.gae(b.rewards, b.terminations, b.values, self.gamma, self.gae_lambda, b.advantages, b.returns, next_values=self.next_values)

    # ---------------------------------------------------------------------------------------------- optimising
    def _first_minibatch_args(self, metrics_row0):
        return self.kernels.minibatch_args(
            m=0, m_global=1, states=self.g_states, actions=self.g_actions, log_probs=self.g_log_probs, advantages=self.g_advantages,
            returns=self.g_returns, adv_stats=self.adv_stats, params=self.params.flat, grads=self.grads, exp_avg=self.exp_avg,
            exp_avg_sq=self.exp_avg_sq, lr=self.lr_dev, step_count=self.adam_step, hp=self.hp, metrics=metrics_row0, workspace=self.train_ws,
            states_ld=self.ldx, states_ones_col=True)

    def _optimize(self):
        """ref: ppo.py:265-294 (epochs x shuffled minibatches)."""
        b, k = self.batch, self.kernels
        T, N, obs, act = self.nr_steps, self.nr_envs, k.obs_dim, k.act_dim
        flat_states = b.states[:T].view(T * N, obs)
        flat_actions = b.actions.view(T * N, act)
        lp, adv, ret = b.log_probs.view(-1), b.advantages.view(-1), b.returns.view(-1)
        mbs = self.minibatch_size
        for epoch in range(self.nr_epochs):
            slot, perm_pinned, count, counts = self._perm_stream.next()  # self.rng.shuffle(batch_indices), done ahead of time
            self._perm_slots_in_flight.append(slot)
            row0 = epoch * self.nmb_epoch
            self.perm_dev.copy_(perm_pinned, non_blocking=True)
            if self.world_size == 1:
                k.gather(self.perm_dev, flat_states, flat_actions, lp, adv, ret, self.g_states, self.g_actions, self.g_log_probs,
                         self.g_advantages, self.g_returns, out_states_ld=self.ldx)
                k.advantage_stats(self.g_advantages, self.batch_size, mbs, self.adv_stats)
                k.update_epoch(self._first_minibatch_args(self.metrics_dev[row0]), self.batch_size, mbs)
            else:
                if counts is None:  # rank-local shuffle: fixed local minibatch size
                    counts = sharding.global_minibatch_sizes(self.local_batch_size, mbs // self.world_size)
                self._optimize_epoch_sharded(count, counts, epoch, flat_states, flat_actions, lp, adv, ret)

    def _optimize_epoch_sharded(self, local_count, counts, epoch, flat_states, flat_actions, lp, adv, ret):
        """Reference-exact data parallelism: every rank walks the same global permutation, computes the gradient SUM over the
        rows it owns, one all-reduce(sum) per minibatch makes the full-minibatch gradient (divided by the global minibatch
        size inside the kernels), then every rank applies the identical clip+Adam step (SURVEY §8 e)."""
        k, dist = self.kernels, self.dist
        mbs, row0 = self.minibatch_size, epoch * self.nmb_epoch
        k.gather(self.perm_dev, flat_states, flat_actions, lp, adv, ret, self.g_states, self.g_actions, self.g_log_probs,
                 self.g_advantages, self.g_returns, count=local_count, out_states_ld=self.ldx)
        offsets = np.concatenate([[0], np.cumsum(counts)])
        global_counts = sharding.global_minibatch_sizes(self.batch_size, mbs)
        assert len(global_counts) == len(counts)
        # global per-minibatch advantage mean / unbiased std: two small all-reduces per epoch (advantages are frozen during the update)
        key = np.asarray(counts, dtype=np.int64).tobytes()
        if self._seg_cache is None or self._seg_cache[0] != key:  # rank-local shuffles: the same split every epoch
            self._seg_cache = (key, torch.from_numpy(offsets.astype(np.int64)).to(self.device),
                               torch.from_numpy(global_counts.astype(np.float32)).to(self.device))
        seg_offsets, gc = self._seg_cache[1], self._seg_cache[2]
        sums, ssq = self.seg_tmp[0, :len(counts)], self.seg_tmp[1, :len(counts)]
        k.segment_moments(self.g_advantages, seg_offsets, None, None, sums)
        self._allreduce_small(sums)
        k.segment_moments(self.g_advantages, seg_offsets, sums, gc, ssq)
        self._allreduce_small(ssq)
        self.adv_stats[:, 0] = sums / gc
        self.adv_stats[:, 1] = torch.sqrt(ssq / (gc - 1.0))
        P = k.param_count
        if self.peer_comm is not None:
            # the whole epoch is one native call: fwdbwd -> peer all-reduce -> clip+Adam per minibatch, no host in between
            first = self.kernels.minibatch_args(
                m=0, m_global=1, states=self.g_states, actions=self.g_actions, log_probs=self.g_log_probs, advantages=self.g_advantages,
                returns=self.g_returns, adv_stats=self.adv_stats, params=self.params.flat, grads=self.grads, exp_avg=self.exp_avg,
                exp_avg_sq=self.exp_avg_sq, lr=self.lr_dev, step_count=self.adam_step, hp=self.hp, metrics=self.metrics_dev[row0],
                workspace=self.train_ws, states_ld=self.ldx, states_ones_col=True)
            k.update_epoch_sharded(first, np.ascontiguousarray(counts, dtype=np.int64), np.ascontiguousarray(global_counts, dtype=np.int64),
                                   self.peer_comm)
            return
        for i in range(len(counts)):
            a = self.kernels.minibatch_args(
                m=int(counts[i]), m_global=int(global_counts[i]), states=self.g_states[offsets[i]:], actions=self.g_actions[offsets[i]:],
                log_probs=self.g_log_probs[offsets[i]:], advantages=self.g_advantages[offsets[i]:], returns=self.g_returns[offsets[i]:],
                adv_stats=self.adv_stats[i], params=self.params.flat, grads=self.grads, exp_avg=self.exp_avg, exp_avg_sq=self.exp_avg_sq,
                lr=self.lr_dev, step_count=self.adam_step, hp=self.hp, metrics=self.grads[P:], workspace=self.train_ws,
                states_ld=self.ldx, states_ones_col=True)
            k.fwdbwd(a)
            dist.all_reduce(self.grads)          # gradient + metric sums, 1.32 MB (host-launched NCCL: the baseline exchange)
            k.clip_adam(a)                       # writes the two grad norms into grads[P+5..P+6]
            self.metrics_dev[row0 + i].copy_(self.grads[P:])

    def _allreduce_small(self, t):
        """in-place sum over ranks of a small contiguous float32 tensor, through whichever exchange carries the gradient."""
        if self.peer_comm is not None:
            self.peer_comm.stage(t)
            self.peer_comm.allreduce_sum(t)
        else:
            self.dist.all_reduce(t)

    def _explained_variance(self):
        """ref: ppo.py:298-300, computed on the device instead of on the host."""
        b = self.batch
        y_true, y_pred = b.returns.view(-1), b.values.view(-1)
        if self.world_size == 1:
            var_y = torch.var(y_true, unbiased=False)
            ev = 1.0 - torch.var(y_true - y_pred, unbiased=False) / var_y
            return var_y, ev
        n = torch.tensor([float(self.batch_size)], device=self.device)
        s = torch.stack([y_true.sum(), (y_true - y_pred).sum()])
        self.dist.all_reduce(s)
        m = s / n
        q = torch.stack([((y_true - m[0]) ** 2).sum(), ((y_true - y_pred - m[1]) ** 2).sum()])
        self.dist.all_reduce(q)
        return q[0] / n[0], 1.0 - q[1] / q[0]

    def _set_learning_rate(self, lr):
        self.lr_host[0] = lr
        self.lr_dev.copy_(self.lr_host, non_blocking=True)

    def current_learning_rate(self):
        if not self.anneal_learning_rate:
            return self.learning_rate
        total_iters = int(self.total_timesteps // self.batch_size)  # LinearLR(1 -> 0, total_iters), ppo.py:87-88
        return self.learning_rate * (1.0 - min(self.lr_iteration, total_iters) / max(total_iters, 1))

    # ---------------------------------------------------------------------------------------------------- train
    def train(self):
        self._begin_training()
        try:
            while self.global_step < self.total_timesteps:
                self._train_iteration()
        finally:
            self._end_training()

    def _end_training(self):
        if self._perm_stream is not None:
            self._perm_stream.close()
            self._perm_stream = None

    def _begin_training(self):
        """Everything PPO.train() does before its while loop (ppo.py:169-193)."""
        self._allocate()
        self._select_precision()
        b, k = self.batch, self.kernels
        self.set_train_mode()
        self.saving_return_buffer = deque(maxlen=100 * self.nr_envs)
        state, _ = self.train_env.reset()
        if self.device_episode_stats:
            self.ep_return.zero_()
            self.ep_length.zero_()
        if self.is_torch_data_interface:
            k.rollout_store(None, None, None, state.float().contiguous(), None, None, b.states[0], None)
        else:
            self._to_device_obs(state, b.states[0])
        if self._perm_stream is None:  # starts shuffling right away: the first permutations are ready before the first rollout ends
            self._perm_stream = self._make_index_stream()
        self.global_step = 0
        self.nr_updates = 0
        self.nr_episodes = 0
        self.prev_saving_end_time = None
        self.logging_time_prev = None
        self.iteration_times = []

    def _optimization_metrics(self, m, ev_host):
        """m: the per-minibatch metric records of this iteration [nr_epochs * minibatches, RLX_PPO_NMETRIC] (ppo.py:285-310)."""
        optimization_metrics = {
            "loss/policy_gradient_loss": m[:, 0].mean(),
            "loss/critic_loss": m[:, 1].mean(),
            "loss/entropy_loss": m[:, 2].mean(),
            "policy_ratio/clip_fraction": m[:, 4].mean(),
            "gradients/policy_grad_norm": m[:, 5].mean(),
            "gradients/critic_grad_norm": m[:, 6].mean(),
        }
        # the reference logs get_last_lr() AFTER scheduler.step() (ppo.py:302-307)
        optimization_metrics["lr/learning_rate"] = self.current_learning_rate()
        optimization_metrics["v_value/explained_variance"] = np.nan if float(ev_host[0]) == 0 else float(ev_host[1])
        optimization_metrics["policy_ratio/approx_kl"] = m[-self.nmb_epoch:, 3].mean()  # last epoch only (approx_kl_divs reset at ppo.py:275)
        optimization_metrics["policy/std_dev"] = float(np.mean(np.exp(self.params.view(self.params.flat, "logstd").cpu().numpy())))
        self.nr_updates += self.nr_epochs * self.nr_minibatches
        return optimization_metrics

    def _make_hparams(self):
        return make_hparams(self.clip_range, self.entropy_coef, self.critic_coef, self.max_grad_norm)

    def _make_index_stream(self):
        """Background producer of the epoch permutations (ppo.py:273-276)."""
        if self.world_size > 1 and self.exact_global_permutation:
            # reference-exact: every rank walks the same GLOBAL permutation and keeps the rows it owns (host work O(global batch))
            transform = lambda perm: sharding.local_rows_of_permutation(perm, self.minibatch_size, self.global_nr_envs, self.nr_envs, self.rank)
            return PermutationStream(self.rng, self.batch_size, self.nr_epochs, self.local_batch_size, transform)
        if self.world_size > 1:
            # scalable: each rank shuffles only its own rows with its own PCG64 stream; global minibatch k = union of the ranks'
            # local minibatches k (host work O(local batch), same collectives)
            if self.minibatch_size % self.world_size != 0:
                raise ValueError("minibatch_size must be divisible by the world size when exact_global_permutation=False")
            self.local_rng = nt.Pcg64Generator((int(self.model_seed) * 1000003 + 7919 * (self.rank + 1)) & 0xFFFFFFFFFFFFFFFF)
            return PermutationStream(self.local_rng, self.local_batch_size, self.nr_epochs, self.local_batch_size, None)
        return PermutationStream(self.rng, self.batch_size, self.nr_epochs, self.local_batch_size, None)

    def _select_precision(self):
        """The precision mode is a library-wide switch: select this instance's before every pass through the kernels."""
        self.kernels.lib.rlx_set_autocast_bf16(1 if self.bf16_mixed_precision_training else 0)

    def _train_iteration(self):
        """One pass of the reference's while-loop body (ppo.py:195-393): acting, advantages, optimising, eval, save, log."""
        self._select_precision()
        b, k = self.batch, self.kernels
        start_time = time.time()
        time_metrics = {}
        steps_metrics = {}
        if self.logging_time_prev:
            time_metrics["time/logging_time_prev"] = self.logging_time_prev

        # Acting
        if self.global_step > 0:  # the observation after the last step of the previous rollout is the first state of this one
            k.rollout_store(None, None, None, b.states[self.nr_steps], None, None, b.states[0], None)
        step_info_collection, saving_returns, dones_host = self._collect_rollout(True)
        self.saving_return_buffer.extend(saving_returns)
        self.global_step += self.nr_steps * self.global_nr_envs
        global_step = self.global_step
        acting_end_time = time.time()
        time_metrics["time/acting_time"] = acting_end_time - start_time

        # Calculating advantages and returns
        self._compute_advantages()
        calc_adv_return_end_time = time.time()
        time_metrics["time/calc_adv_and_return_time"] = calc_adv_return_end_time - acting_end_time

        # Optimizing
        self._set_learning_rate(self.current_learning_rate())
        self._optimize()
        var_y, ev = self._explained_variance()
        ev_pair = torch.stack([var_y, ev])
        lr_used = self.current_learning_rate()
        if self.anneal_learning_rate:
            self.lr_iteration += 1  # policy_scheduler.step(); critic_scheduler.step()  (ppo.py:302-304)

        # the only device->host transfers of the iteration: per-minibatch metric records, explained variance, done count
        self.metrics_host.copy_(self.metrics_dev, non_blocking=True)
        if self.device_episode_stats:
            self.done_stats_host.copy_(self.done_stats_dev, non_blocking=True)
        ev_host = ev_pair.cpu()
        dones_this_rollout = dones_host if not self.is_torch_data_interface else int(self.done_count.item())
        if self.device_episode_stats and dones_this_rollout > 0:
            # what the reference's wrapper would have handed over step by step (`v[done_mask].tolist()`, wrappers.py:29-32): finished
            # episodes in step order, env order within a step
            lengths = self.done_stats_host[1].numpy()
            mask = lengths > 0
            finished_returns = self.done_stats_host[0].numpy()[mask]
            step_info_collection.setdefault("episode_return", []).extend(finished_returns.tolist())
            step_info_collection.setdefault("episode_length", []).extend(lengths[mask].tolist())
            self.saving_return_buffer.extend(finished_returns.tolist())
        if self._perm_stream is not None:  # the .cpu()/.item() above synchronised the stream: the staged permutations were consumed
            self._perm_stream.release(self._perm_slots_in_flight)
            self._perm_slots_in_flight = []
        if self.dist:
            t = torch.tensor([dones_this_rollout], device=self.device)
            self.dist.all_reduce(t)
            dones_this_rollout = int(t.item())
        self.nr_episodes += dones_this_rollout
        optimization_metrics = self._optimization_metrics(self.metrics_host.numpy(), ev_host)

        optimizing_end_time = time.time()
        time_metrics["time/optimizing_time"] = optimizing_end_time - calc_adv_return_end_time

        # Evaluating
        evaluation_metrics = {}
        if global_step % self.evaluation_frequency == 0 and self.evaluation_frequency != -1:
            evaluation_metrics = self._evaluate()
        evaluating_end_time = time.time()
        time_metrics["time/evaluating_time"] = evaluating_end_time - optimizing_end_time

        # Saving (only when episodes finished this update, ppo.py:353-357)
        if self.save_model and dones_this_rollout > 0 and len(self.saving_return_buffer) > 0 and self.rank == 0:
            mean_return = np.mean(self.saving_return_buffer)
            if mean_return > self.best_mean_return:
                self.best_mean_return = mean_return
                self.save()

        saving_end_time = time.time()
        if self.prev_saving_end_time:
            time_metrics["time/sps"] = int((self.nr_steps * self.global_nr_envs) / (saving_end_time - self.prev_saving_end_time))
            self.iteration_times.append(saving_end_time - self.prev_saving_end_time)
        self.prev_saving_end_time = saving_end_time
        time_metrics["time/saving_time"] = saving_end_time - evaluating_end_time

        # Logging
        self.start_logging(global_step)
        steps_metrics["steps/nr_env_steps"] = global_step
        steps_metrics["steps/nr_updates"] = self.nr_updates
        steps_metrics["steps/nr_episodes"] = self.nr_episodes

        rollout_info_metrics = {}
        env_info_metrics = {}
        for info_name, values in step_info_collection.items():
            metric_group = "rollout" if info_name in ["episode_return", "episode_length"] else "env_info"
            metric_dict = rollout_info_metrics if metric_group == "rollout" else env_info_metrics
            mean_value = np.mean(values)
            if mean_value == mean_value:
                metric_dict[f"{metric_group}/{info_name}"] = mean_value
        evaluation_metrics = {key: np.mean(value) for key, value in evaluation_metrics.items()}
        combined_metrics = {**rollout_info_metrics, **evaluation_metrics, **env_info_metrics, **steps_metrics, **time_metrics, **optimization_metrics}
        for key, value in combined_metrics.items():
            self.log(f"{key}", value, global_step)
        self.end_logging()
        logging_end_time = time.time()
        self.logging_time_prev = logging_end_time - saving_end_time

    # ------------------------------------------------------------------------------------------ eval / test
    def _deterministic_action(self, state):
        """ref: policy.get_deterministic_action (policy.py:85-93)."""
        self._select_precision()
        self.kernels.forward(self.params.flat, state, self._eval_ws(state.shape[0]), act_low=self.env_as_low, act_high=self.env_as_high,
                             clip_rescale=self.action_clipping_and_rescaling, deterministic=True, env_action=self._eval_action(state.shape[0]))
        return self._eval_action(state.shape[0])

    def _eval_ws(self, n):
        if getattr(self, "_eval_ws_buf", None) is None or self._eval_ws_n < n:
            self._eval_ws_buf, self._eval_ws_n = self.kernels.forward_workspace(n, self.device), n
            self._eval_action_buf = torch.zeros(n, self.kernels.act_dim, dtype=torch.float32, device=self.device)
        return self._eval_ws_buf

    def _eval_action(self, n):
        return self._eval_action_buf[:n]

    def _obs_to_device(self, state):
        if torch.is_tensor(state):
            return state.to(self.device, torch.float32).contiguous()
        return torch.tensor(np.asarray(state), dtype=torch.float32).to(self.device)

    def _evaluate(self):
        """ref: ppo.py:319-345."""
        self.set_eval_mode()
        eval_state, _ = self.eval_env.reset()
        eval_nr_episodes = 0
        evaluation_metrics = {"eval/episode_return": [], "eval/episode_length": []}
        while True:
            action = self._deterministic_action(self._obs_to_device(eval_state))
            if not self.is_torch_data_interface:
                action = action.cpu().numpy()
            eval_state, eval_reward, eval_terminated, eval_truncated, eval_info = self.eval_env.step(action)
            eval_done = eval_terminated | eval_truncated
            for i, single_done in enumerate(eval_done):
                if single_done:
                    eval_nr_episodes += 1
                    evaluation_metrics["eval/episode_return"].append(self.eval_env.get_final_info_value_at_index(eval_info, "episode_return", i))
                    evaluation_metrics["eval/episode_length"].append(self.eval_env.get_final_info_value_at_index(eval_info, "episode_length", i))
                    if eval_nr_episodes == self.evaluation_episodes:
                        break
            if eval_nr_episodes == self.evaluation_episodes:
                break
        self.set_train_mode()
        return evaluation_metrics

    def test(self, episodes):
        """ref: ppo.py:454-472."""
        self.set_eval_mode()
        for i in range(episodes):
            done = False
            episode_return = 0
            state, _ = self.eval_env.reset()
            while not done:
                processed_action = self._deterministic_action(self._obs_to_device(state))
                if not self.is_torch_data_interface:
                    processed_action = processed_action.cpu().numpy()
                state, reward, terminated, truncated, info = self.eval_env.step(processed_action)
                done = terminated | truncated
                done = bool(done.any()) if hasattr(done, "any") else bool(done)
                episode_return += reward
            rlx_logger.info(f"Episode {i + 1} - Return: {episode_return}")

    # --------------------------------------------------------------------------------------------- logging
    def log(self, name, value, step):
        if self.rank != 0:
            return
        if self.track_wandb:
            self.wandb_log_cache[name] = value
        if self.track_tb:
            self.writer.add_scalar(name, value, step)
        if self.track_console:
            self.log_console(name, value)

    def log_console(self, name, value):
        value = np.format_float_positional(value, trim="-")
        rlx_logger.info(f"│ {name.ljust(30)}│ {str(value).ljust(14)[:14]} │")

    def start_logging(self, step):
        if self.rank != 0:
            return
        if self.track_wandb:
            self.wandb_log_cache = {"global_step": int(step)}
        if self.track_console:
            rlx_logger.info("┌" + "─" * 31 + "┬" + "─" * 16 + "┐")
        else:
            rlx_logger.info(f"Step: {step}")

    def end_logging(self, wandb_commit=True):
        if self.rank != 0:
            return
        if self.track_wandb:
            import wandb
            wandb.log(self.wandb_log_cache, commit=wandb_commit)
        if self.track_console:
            rlx_logger.info("└" + "─" * 31 + "┴" + "─" * 16 + "┘")

    # ------------------------------------------------------------------------------------- checkpointing
    def save(self):
        """ref: ppo.py:426-436.  Same dict keys, the reference modules' parameter names and order and the reference optimisers' parameter
        numbering, so that the reference's own load() (strict load_state_dict, ppo.py:439-451) accepts the file and vice versa."""
        file_path = self.save_path + "/best.model"
        pol, cri = self.params.state_dicts()
        step, lr = float(self.adam_step.item()), self.current_learning_rate()
        torch.save({
            "config_algorithm": self.config.algorithm,
            "policy_state_dict": pol,
            "critic_state_dict": cri,
            "policy_optimizer_state_dict": self.params.adam_state_dict(POLICY_PARAM_ORDER, nt.POLICY_KEYS, self.exp_avg, self.exp_avg_sq, step, lr),
            "critic_optimizer_state_dict": self.params.adam_state_dict(CRITIC_PARAM_ORDER, nt.CRITIC_KEYS, self.exp_avg, self.exp_avg_sq, step, lr),
        }, file_path)
        if self.track_wandb:
            import wandb
            wandb.save(file_path, base_path=os.path.dirname(file_path))

    @classmethod
    def load(cls, config, train_env, eval_env, run_path, writer, explicitly_set_algorithm_params):
        checkpoint = torch.load(config.runner.load_model, weights_only=False)
        loaded_algorithm_config = checkpoint["config_algorithm"]
        for key, value in loaded_algorithm_config.items():
            if f"algorithm.{key}" not in explicitly_set_algorithm_params and key in config.algorithm and key not in ("name", "device", "compile_mode"):
                config.algorithm[key] = value
        model = cls(config, train_env, eval_env, run_path, writer)
        named = {**checkpoint["policy_state_dict"], **checkpoint["critic_state_dict"]}
        model.params.load_named(named)
        step_p = model.params.load_adam_state(checkpoint["policy_optimizer_state_dict"], POLICY_PARAM_ORDER, nt.POLICY_KEYS, model.exp_avg, model.exp_avg_sq)
        step_c = model.params.load_adam_state(checkpoint["critic_optimizer_state_dict"], CRITIC_PARAM_ORDER, nt.CRITIC_KEYS, model.exp_avg, model.exp_avg_sq)
        model.adam_step.fill_(int(max(step_p, step_c)))
        return model

    def set_train_mode(self):
        self.training = True

    def set_eval_mode(self):
        self.training = False

    def general_properties():
        return GeneralProperties
