"""One PPO minibatch update (config-2 shapes) in isolation, for `ncu --set full` captures of every kernel on the update path.

    ncu --set full --clock-control none --import-source on -k regex:rlx -s <11*warmup> -c 11 -o minibatch_prof python profiles/profile_minibatch.py [engine] [reps]
"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_x_b200 import _native as nt
from rl_x_b200.algorithms.ppo.b200.kernels import PpoKernels, make_hparams

engine = sys.argv[1] if len(sys.argv) > 1 else "tcgen05"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
nt.load().rlx_set_gemm_engine(1 if engine == "tcgen05" else 0)
obs, act, hidden, m = 376, 17, 256, 32768
k = PpoKernels(obs, act, hidden)
dev = "cuda"
g = torch.Generator(device=dev).manual_seed(0)
P = k.param_count
params = torch.randn(P, device=dev, generator=g) * 0.05
ldx = k.states_pitch()
states = torch.randn(m, ldx, device=dev, generator=g)
states[:, obs] = 1.0
states[:, obs + 1:] = 0.0
actions = torch.randn(m, act, device=dev, generator=g)
logp = -25.0 + torch.randn(m, device=dev, generator=g)
adv, ret = torch.randn(m, device=dev, generator=g), torch.randn(m, device=dev, generator=g)
stats = torch.empty(1, 2, device=dev)
k.advantage_stats(adv, m, m, stats)
ws = k.minibatch_workspace(m, dev)
args = k.minibatch_args(m=m, m_global=m, states=states, actions=actions, log_probs=logp, advantages=adv, returns=ret, adv_stats=stats, params=params,
                        grads=torch.zeros(P, device=dev), exp_avg=torch.zeros(P, device=dev), exp_avg_sq=torch.zeros(P, device=dev),
                        lr=torch.full((1,), 3e-4, device=dev), step_count=torch.zeros(1, dtype=torch.int64, device=dev),
                        hp=make_hparams(0.2, 0.0, 0.5, 0.5), metrics=torch.zeros(8, device=dev), workspace=ws, states_ld=ldx, states_ones_col=True)
for _ in range(reps):
    k.fwdbwd(args)
    k.clip_adam(args)
torch.cuda.synchronize()
nt.timing_begin()
for _ in range(5):
    k.fwdbwd(args)
    k.clip_adam(args)
for name, c in nt.timing_end().items():
    if c["launches"]:
        print(f"{name:14s} {c['ms'] / 5 * 1e3:9.1f} us/minibatch  launches={c['launches'] // 5}  {c['flops'] / max(c['ms'], 1e-9) / 1e9:8.1f} TFLOP/s  {c['bytes'] / max(c['ms'], 1e-9) / 1e6:8.1f} GB/s")
