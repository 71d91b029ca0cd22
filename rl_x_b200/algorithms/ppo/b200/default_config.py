"""Same keys and defaults as rl_x/algorithms/ppo/pytorch/default_config.py:4-30.  Differences, all explicit:
    `bf16_mixed_precision_training` defaults to False (this build is the fp32 parity path), `compile_mode` is accepted and
    ignored (no tracing compiler here), and three B200-specific keys are appended."""
from rl_x_b200.config_dict import config_from_defaults

_DEFAULTS = (
    ('device', "gpu"),  # a CUDA device is mandatory: there is no CPU fallback
    ('compile_mode', "default"),
    ('bf16_mixed_precision_training', False),
    ('total_timesteps', 1e9),
    ('learning_rate', 3e-4),
    ('anneal_learning_rate', False),
    ('nr_steps', 2048),
    ('nr_epochs', 10),
    ('minibatch_size', 64),
    ('gamma', 0.99),
    ('gae_lambda', 0.95),
    ('clip_range', 0.2),
    ('entropy_coef', 0.0),
    ('critic_coef', 0.5),
    ('max_grad_norm', 0.5),
    ('std_dev', 1.0),
    ('action_clipping_and_rescaling', True),
    ('nr_hidden_units', 256),
    ('evaluation_frequency', -1),
    ('evaluation_episodes', 10),
    ('gemm_engine', "auto"),  # auto | simt (fp32 FFMA) | tcgen05 (3xTF32 tensor cores)
    ('exact_global_permutation', True),  # multi-GPU: reference-exact global shuffle (ppo.py:273-276) vs per-rank local shuffles
    ('gradient_exchange', "peer"),  # multi-GPU: peer (library all-reduce kernel over NVLink peer memory) | nccl (torch.distributed)
    ('peer_exchange_algorithm', "auto"),  # auto | one_shot: both select the one-shot peer all-reduce kernel, the only one there is
    ('device_episode_statistics', True),  # TORCH-interface envs: episode return / length tracked on the device, read back once per iteration
    ('ignore_process_group', False),      # build a single-GPU instance inside a multi-rank job (bench.py's sharded-vs-single parity check)
    ('rollout_noise', "philox"),  # philox (in-kernel counter-based normals) | torch (torch.randn on device, injected)
)


def get_config(algorithm_name):
    return config_from_defaults(algorithm_name, _DEFAULTS)
