"""Opt-in mma.sync formulation of the PPO loss head (rlx_set_head_engine(2), csrc/ppo_head_mma.cuh) inside rlx_ppo_minibatch_fwdbwd_f32:
gradients and metrics must equal the default fused SIMT head's."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _run_head_engine(lib, k, fp, engine, m, ldx, states, actions, logp, adv, ret, stats, hp):
    from rl_x_b200 import _native as nt
    P = k.param_count
    assert lib.rlx_set_head_engine(engine) == engine
    grads, metrics = torch.zeros(P, device=DEV), torch.zeros(nt.RLX_PPO_NMETRIC, device=DEV)
    args = k.minibatch_args(m=m, m_global=m, states=states, actions=actions, log_probs=logp, advantages=adv, returns=ret, adv_stats=stats,
                            params=fp.flat, grads=grads, exp_avg=torch.zeros(P, device=DEV), exp_avg_sq=torch.zeros(P, device=DEV),
                            lr=torch.full((1,), 3e-4, device=DEV), step_count=torch.zeros(1, dtype=torch.int64, device=DEV),
                            hp=hp, metrics=metrics, workspace=k.minibatch_workspace(m, DEV), states_ld=ldx, states_ones_col=True)
    k.fwdbwd(args)
    torch.cuda.synchronize()
    return grads, metrics.cpu().numpy()


@pytest.mark.parametrize("obs,act,hidden,m", [(376, 17, 256, 32768), (376, 17, 256, 4096), (24, 5, 128, 1000), (11, 3, 512, 777), (8, 23, 256, 130),
                                              (8, 31, 128, 16), (6, 7, 256, 17)])
def test_mma_head_matches_fused_head(obs, act, hidden, m):
    """rlx_set_head_engine(2), csrc/ppo_head_mma.cuh: every gradient segment and every metric of one minibatch equals the SIMT head's
    (3xTF32 products against fp32 FMAs: agreement at the 1e-6 level of each segment's norm); ragged row counts cover the partial
    16-row and 128-row tiles."""
    from rl_x_b200 import _native as nt
    from rl_x_b200.algorithms.ppo.b200.kernels import PpoKernels, make_hparams
    from oracle import ppo_oracle as O
    from rl_x_b200.algorithms.ppo.b200.ppo import FlatParameters
    lib = nt.load()
    k = PpoKernels(obs, act, hidden)
    pol, cri = O.init_params(obs, act, hidden, seed=3)
    fp = FlatParameters(k, DEV)
    fp.load_named({**pol, **cri})
    fp.view(fp.flat, nt.POLICY_KEYS["policy_logstd"]).copy_(torch.linspace(-0.4, 0.3, act).reshape(fp.shapes["logstd"]))  # distinct std per action
    g = torch.Generator().manual_seed(m)
    ldx = k.states_pitch()
    states = torch.zeros(m, ldx)
    states[:, :obs] = torch.randn(m, obs, generator=g)
    states[:, obs] = 1.0
    t = lambda x: x.to(DEV).contiguous()
    actions, logp, adv, ret = t(torch.randn(m, act, generator=g)), t(torch.randn(m, generator=g) * 0.3 - act), t(torch.randn(m, generator=g)), t(torch.randn(m, generator=g))
    stats = torch.tensor([float(adv.mean()), float(adv.std()) if m > 1 else 1.0], device=DEV)
    hp = make_hparams(0.2, 0.01, 0.5, 0.5)
    try:
        g0, m0 = _run_head_engine(lib, k, fp, 0, m, ldx, t(states), actions, logp, adv, ret, stats, hp)
        g2, m2 = _run_head_engine(lib, k, fp, 2, m, ldx, t(states), actions, logp, adv, ret, stats, hp)
    finally:
        lib.rlx_set_head_engine(0)
    report, worst = [], 0.0
    for seg in nt.SEGMENT_NAMES:
        a, b = fp.view(g0, seg).double(), fp.view(g2, seg).double()
        rel = float((b - a).norm() / max(float(a.norm()), 1e-30))
        report.append(f"{seg}: {rel:.2e} (norm {float(a.norm()):.2e})")
        worst = max(worst, rel)
    assert worst <= 2e-5, "\n".join(report) + f"\nmetrics fused {m0[:5]}\nmetrics mma   {m2[:5]}"
    np.testing.assert_allclose(m2[:5], m0[:5], rtol=2e-4, atol=2e-6)
