"""End-to-end GPU tests of the plugin class: PPO.train() through the reference-shaped API, replaying the environment
stream and action noise of the executed reference (golden fixtures) and comparing the resulting weights and logged metrics."""
import numpy as np
import pytest
import torch

from oracle import ppo_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["simt", "tcgen05"])
def gemm_engine(request):
    """Every test runs once per GEMM engine (shapes the tcgen05 engine does not cover fall back to the SIMT engine)."""
    from rl_x_b200 import _native as nt
    lib = nt.load()
    lib.rlx_set_gemm_engine(1 if request.param == "tcgen05" else 0)
    yield request.param
    lib.rlx_set_gemm_engine(0)
DEV = "cuda"


class _Space:
    def __init__(self, shape, low=None, high=None):
        self.shape, self.low, self.high = shape, low, high


def _props(interface):
    from rl_x_b200.environments.types import ActionSpaceType, ObservationSpaceType, DataInterfaceType

    class P:
        observation_space_type = ObservationSpaceType.FLAT_VALUES
        action_space_type = ActionSpaceType.CONTINUOUS
        data_interface_type = getattr(DataInterfaceType, interface)
    return P


class ReplayEnv:
    """Feeds back the exact observation / reward / termination stream the reference saw (captured in the golden file)."""

    def __init__(self, g, interface="TORCH"):
        self.g, self.numpy = g, interface == "NUMPY"
        self.general_properties = _props(interface)
        self.single_observation_space = _Space((g.obs,))
        self.single_action_space = _Space((g.act,), np.full(g.act, g.act_low, np.float32), np.full(g.act, g.act_high, np.float32))
        self.t = 0
        self.actions = []

    def _o(self, x, dtype=None):
        if self.numpy:
            return np.asarray(x)
        t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
        return t

    def reset(self):
        return self._o(self.g["iter0/states"][0]), {}

    def step(self, action):
        g = self.g
        self.actions.append(torch.as_tensor(action).detach().cpu().clone())
        it, s = divmod(self.t, g.T)
        self.t += 1
        nxt = g[f"iter{it}/next_states"][s]
        rew = g[f"iter{it}/rewards"][s]
        term = g[f"iter{it}/terminations"][s] > 0.5
        trunc = np.full(g.N, self.t % 11 == 0)
        self._last_next = nxt
        return self._o(nxt), self._o(rew), self._o(term), self._o(trunc), {}

    def get_logging_info_dict(self, info):
        return {}

    def get_final_observation_at_index(self, info, i):
        return self._last_next[i]  # the replayed stream already holds what the reference stored as next_states

    def get_final_info_value_at_index(self, info, key, i):
        return 0.0

    def close(self):
        pass


def _config(g, engine="simt", **algo):
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.ppo.b200.default_config import get_config
    a = get_config("ppo.b200")
    a.nr_steps, a.minibatch_size, a.nr_epochs, a.nr_hidden_units = g.T, g.mb, g.epochs, g.hidden
    a.total_timesteps = g.N * g.T * g.iterations
    a.std_dev, a.entropy_coef, a.anneal_learning_rate = g.std_dev, g.entropy_coef, g.anneal
    a.learning_rate, a.clip_range, a.critic_coef, a.max_grad_norm = g.lr, g.clip_range, g.critic_coef, g.max_grad_norm
    a.gamma, a.gae_lambda = g.gamma, g.gae_lambda
    a.gemm_engine = engine
    for k, v in algo.items():
        a[k] = v
    return ConfigDict(algorithm=a, environment=ConfigDict(seed=g.seed, nr_envs=g.N),
                      runner=ConfigDict(save_model=False, track_console=False, track_tb=False, track_wandb=False, load_model=""))


def _reference_noise(g):
    """eps such that mean + std * eps reproduces the reference's stored actions, from the weights the reference acted with."""
    out = []
    for it in range(g.iterations):
        pol, _ = g.params("init" if it == 0 else f"iter{it - 1}")
        pol = {k: torch.from_numpy(v) for k, v in pol.items()}
        states = torch.from_numpy(g[f"iter{it}/states"]).reshape(-1, g.obs)
        with torch.no_grad():
            mean = O.policy_mean(pol, states)
        eps = (torch.from_numpy(g[f"iter{it}/actions"]).reshape(-1, g.act) - mean) / torch.exp(pol["policy_logstd"])
        out.append(eps.reshape(g.T, g.N, g.act))
    return torch.cat(out).to(DEV).contiguous()


@pytest.mark.parametrize("interface", ["TORCH", "NUMPY"])
def test_train_reproduces_reference_run(golden, interface, gemm_engine):
    from rl_x_b200.algorithms.ppo.b200.ppo import PPO
    g = golden
    env = ReplayEnv(g, interface)
    model = PPO(_config(g, engine=gemm_engine), env, env, "/tmp/rlx_test_run", None)
    eps = _reference_noise(g)
    calls = {"n": 0}

    def draw(step):
        i = calls["n"]
        calls["n"] += 1
        return eps[i]

    model._draw_noise = draw
    logged = []
    model.log = lambda name, value, step: logged.append((name, float(value), int(step)))
    snaps = []
    orig = model.start_logging

    def start_logging(step):
        b = model.batch
        snaps.append(dict(adv=b.advantages.cpu().numpy().copy(), ret=b.returns.cpu().numpy().copy(), val=b.values.cpu().numpy().copy(),
                          lp=b.log_probs.cpu().numpy().copy(), sd=model.params.state_dicts()))
        orig(step)

    model.start_logging = start_logging
    model.train()
    assert calls["n"] == g.T * g.iterations and len(snaps) == g.iterations
    # the env received the clipped / rescaled actions the reference sent
    np.testing.assert_allclose(torch.stack(env.actions).numpy(), g["env_actions"], rtol=1e-4, atol=5e-6)
    # north_star: <= 1e-5 relative on losses / advantages.  The norm (SURVEY.md §7a): ||ours - ref||_2 <= 1e-5 * ||ref||_2 per tensor, in the
    # FIRST iteration, where both sides act with identical weights.  From the second iteration on the run follows its own weights, which
    # Adam's eps-regime components have moved ~1e-5 of their norm away from the reference's (see test_one_epoch_at_bench_shape_vs_oracle):
    # there the bound is 1e-4 of the norm.  The elementwise allclose is the coarse guard against single outliers.
    relnorm = lambda a, b: float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b.astype(np.float64)), 1e-30))
    for it, s in enumerate(snaps):
        bar = 1e-5 if it == 0 else 1e-4
        for key, name in (("val", "values"), ("lp", "log_probs"), ("adv", "advantages"), ("ret", "returns")):
            assert relnorm(s[key], g[f"iter{it}/{name}"]) <= bar, (it, name, relnorm(s[key], g[f"iter{it}/{name}"]))
        np.testing.assert_allclose(s["val"], g[f"iter{it}/values"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(s["lp"], g[f"iter{it}/log_probs"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(s["adv"], g[f"iter{it}/advantages"], rtol=1e-4, atol=2e-5)
        np.testing.assert_allclose(s["ret"], g[f"iter{it}/returns"], rtol=1e-4, atol=2e-5)
        pol_ref, cri_ref = g.params(f"iter{it}")
        pol, cri = s["sd"]
        for name, v in {**pol_ref, **cri_ref}.items():
            ours = (pol if name in pol else cri)[name].numpy()
            rel = float(np.linalg.norm(ours - v) / np.linalg.norm(v))
            assert rel <= 2e-5, (it, name, rel)
    names = {n for n, _, _ in logged}
    for n in ["loss/policy_gradient_loss", "loss/critic_loss", "loss/entropy_loss", "policy_ratio/clip_fraction", "policy_ratio/approx_kl",
              "gradients/policy_grad_norm", "gradients/critic_grad_norm", "lr/learning_rate", "v_value/explained_variance", "policy/std_dev",
              "steps/nr_env_steps", "steps/nr_updates", "steps/nr_episodes", "time/acting_time", "time/calc_adv_and_return_time",
              "time/optimizing_time", "time/evaluating_time", "time/saving_time"]:
        assert n in names, n
    for n in ["loss/critic_loss", "loss/entropy_loss", "gradients/policy_grad_norm", "gradients/critic_grad_norm", "lr/learning_rate",
              "v_value/explained_variance", "policy/std_dev", "steps/nr_env_steps", "steps/nr_updates", "steps/nr_episodes"]:
        ours = [v for m, v, _ in logged if m == n]
        ref = g[f"metric/{n}"]
        np.testing.assert_allclose(ours[:1], ref[:1], rtol=1e-5, atol=1e-7, err_msg=n + " (first iteration: identical weights on both sides)")
        np.testing.assert_allclose(ours, ref, rtol=2e-4, atol=1e-6, err_msg=n)
    # pg_loss is a mean of signed terms with near-zero mean: its scale is the summand scale E|A_hat| ~ 0.8, not its own value
    ours = [v for m, v, _ in logged if m == "loss/policy_gradient_loss"]
    np.testing.assert_allclose(ours[:1], g["metric/loss/policy_gradient_loss"][:1], rtol=0, atol=1e-5 * 0.8)
    np.testing.assert_allclose(ours, g["metric/loss/policy_gradient_loss"], rtol=0, atol=2e-5)


def test_runner_trains_on_synthetic_env_and_checkpoints(tmp_path, monkeypatch, gemm_engine):
    from rl_x_b200.runner.runner import Runner
    from rl_x_b200 import _native as nt
    monkeypatch.chdir(tmp_path)
    argv = ["--environment.nr_envs=64", "--environment.obs_dim=24", "--environment.act_dim=5", "--algorithm.nr_steps=16",
            "--algorithm.minibatch_size=256", "--algorithm.nr_epochs=2", "--algorithm.nr_hidden_units=64", "--algorithm.total_timesteps=3072",
            f"--algorithm.gemm_engine={gemm_engine}",
            "--runner.save_model=True", "--runner.run_name=t1", "--environment.termination_probability=0.05"]
    nt.load().rlx_reset_launch_count()
    r = Runner(argv=argv)
    r.run()
    assert not getattr(r, "failed", False)
    assert nt.load().rlx_launch_count() > 100
    model = r.model
    assert len(model.iteration_times) == 2
    # like the reference, "save best" needs episode returns from the env (ppo.py:353-357); the synthetic stream has none
    model.save()
    ckpt = tmp_path / "runs" / "placeholder" / "placeholder" / "t1" / "models" / "best.model"
    assert ckpt.exists()
    ck = torch.load(ckpt, weights_only=False)
    assert set(ck) == {"config_algorithm", "policy_state_dict", "critic_state_dict", "policy_optimizer_state_dict", "critic_optimizer_state_dict"}
    assert set(ck["policy_state_dict"]) == set(O.POLICY_KEYS) and set(ck["critic_state_dict"]) == set(O.CRITIC_KEYS)
    # the checkpoint drives plain torch modules shaped like the reference's (policy.py:45-52)
    pol = {k: v for k, v in ck["policy_state_dict"].items()}
    x = torch.randn(7, 24)
    mean = O.policy_mean(pol, x)
    assert mean.shape == (7, 5) and torch.isfinite(mean).all()
    # and loads back into the plugin, continuing with identical weights / moments
    r2 = Runner(argv=argv[:-3] + ["--runner.load_model=" + str(ckpt), "--runner.run_name=t2", "--runner.mode=test", "--runner.nr_test_episodes=1",
                                  "--environment.horizon=5"])
    m2, env, _ = r2._build_model(str(tmp_path / "x"), None)
    p1, c1 = ck["policy_state_dict"], ck["critic_state_dict"]
    p2, c2 = m2.params.state_dicts()
    for k in p1:
        assert torch.equal(p1[k], p2[k])
    for k in c1:
        assert torch.equal(c1[k], c2[k])
    assert int(m2.adam_step.item()) == int(float(ck["policy_optimizer_state_dict"]["state"][0]["step"]))
    m2.test(1)


def test_config1_pendulum_trains_evaluates_and_saves_best(tmp_path, monkeypatch):
    """BASELINE.json configs[0]: PPO on Pendulum-v1 with nr_envs=4 through the runner (NUMPY data interface, gym-style autoreset infos).
    Covers PPO._evaluate() (ppo.py:319-345 of the reference): deterministic actions until `evaluation_episodes` episodes finished."""
    from rl_x_b200.runner.runner import Runner
    monkeypatch.chdir(tmp_path)
    argv = ["--environment.name=synthetic.pendulum", "--algorithm.nr_steps=256", "--algorithm.minibatch_size=64", "--algorithm.nr_epochs=2",
            "--algorithm.nr_hidden_units=64", "--algorithm.total_timesteps=3072", "--algorithm.evaluation_frequency=1024",
            "--algorithm.evaluation_episodes=3", "--runner.save_model=True", "--runner.run_name=c1"]
    r = Runner(argv=argv)
    model, env, eval_env = r._build_model(str(tmp_path / "run"), None)
    assert model.nr_envs == 4 and not model.is_torch_data_interface
    logged = []
    model.log = lambda name, value, step: logged.append((name, float(value), int(step)))
    model.train()
    names = [n for n, _, _ in logged]
    for n in ("rollout/episode_return", "rollout/episode_length", "eval/episode_return", "eval/episode_length", "loss/critic_loss", "time/sps"):
        assert n in names, n
    ev = [v for n, v, _ in logged if n == "eval/episode_length"]
    assert len(ev) == 3 and all(v == 200.0 for v in ev)             # every evaluation: 3 episodes of TimeLimit(200)
    rets = [v for n, v, _ in logged if n == "rollout/episode_return"]
    assert all(-2000.0 < v < 0.0 for v in rets)                       # Pendulum-v1 returns: 200 steps of cost in [0, 16.3]
    assert [v for n, v, _ in logged if n == "rollout/episode_length"] == [200.0] * len(rets)
    assert (tmp_path / "run" / "models" / "best.model").exists()    # episodes finished -> save-best fired (ppo.py:353-357)
    assert model.nr_episodes == 4 * (3 * 256 // 200)


def test_device_episode_statistics_match_a_host_recomputation(gemm_engine):
    """SURVEY.md §8 f1: for TORCH-interface envs episode return / length are tracked on the device inside the rollout-store kernel and
    read back once per iteration.  Check against a host replay of the stored rewards / terminations / truncations with the semantics
    of the reference env + wrapper (warp_torch/environment.py:159-178, wrappers.py:15-33)."""
    from rl_x_b200.runner.runner import Runner
    N, T, horizon, iters = 64, 40, 13, 3
    argv = [f"--environment.nr_envs={N}", "--environment.obs_dim=24", "--environment.act_dim=5", f"--environment.horizon={horizon}",
            "--environment.termination_probability=0.03", f"--algorithm.nr_steps={T}", "--algorithm.minibatch_size=256", "--algorithm.nr_epochs=1",
            "--algorithm.nr_hidden_units=64", f"--algorithm.total_timesteps={iters * N * T}", f"--algorithm.gemm_engine={gemm_engine}"]
    r = Runner(argv=argv)
    model, env, _ = r._build_model("/tmp/rlx_epstats", None)
    assert model.is_torch_data_interface
    logged, per_iter = [], []
    model.log = lambda name, value, step: logged.append((name, float(value), int(step)))
    orig = model.start_logging

    def start_logging(step):
        b = model.batch
        per_iter.append((b.rewards.cpu().numpy().copy(), b.terminations.cpu().numpy().copy()))
        orig(step)

    model.start_logging = start_logging
    model.train()
    ep_ret, ep_len, t_global = np.zeros(N, np.float32), np.zeros(N, np.float32), 0
    want_ret, want_len, episodes = [], [], 0
    for rew, term in per_iter:
        rets, lens = [], []
        for t in range(T):
            t_global += 1
            done = (term[t] > 0.5) | (t_global % horizon == 0)  # the synthetic env truncates every `horizon` steps
            ep_ret += rew[t]
            ep_len += 1
            rets += ep_ret[done].tolist()
            lens += ep_len[done].tolist()
            ep_ret[done], ep_len[done] = 0, 0
        episodes += len(rets)
        want_ret.append(np.mean(rets))
        want_len.append(np.mean(lens))
    got_ret = [v for n, v, _ in logged if n == "rollout/episode_return"]
    got_len = [v for n, v, _ in logged if n == "rollout/episode_length"]
    np.testing.assert_allclose(got_ret, want_ret, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(got_len, want_len, rtol=1e-7)
    assert [v for n, v, _ in logged if n == "steps/nr_episodes"][-1] == episodes
    assert len(model.saving_return_buffer) == episodes


def test_load_checkpoint_written_by_the_reference(tmp_path, monkeypatch):
    """PPO.load() on a best.model written by the executed reference's own save() (tests/golden/make_golden_ppo_ckpt.py): weights and both
    Adam states arrive where the reference had them (its optimizer numbers policy_logstd as parameter 0), training continues from it, and
    the file save() writes afterwards has the reference's layout again."""
    import os
    from rl_x_b200 import _native as nt
    from rl_x_b200.runner.runner import Runner
    monkeypatch.chdir(tmp_path)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ex = np.load(os.path.join(root, "tests", "golden", "ppo_ref_checkpoint_expect.npz"))
    N, T, obs, act, hid, mb, E = (int(x) for x in ex["meta"])
    argv = [f"--environment.nr_envs={N}", f"--environment.obs_dim={obs}", f"--environment.act_dim={act}", "--runner.save_model=True",
            "--runner.run_name=fromref", "--runner.load_model=" + os.path.join(root, "tests", "golden", "ppo_ref_checkpoint.model"),
            f"--algorithm.total_timesteps={2 * N * T}"]
    r = Runner(argv=argv)
    model, env, _ = r._build_model(str(tmp_path / "run"), None)
    assert (model.nr_steps, model.nr_epochs, model.minibatch_size, model.nr_hidden_units) == (T, E, mb, hid)  # taken from the checkpoint's config
    for tag, keys in (("policy", nt.POLICY_KEYS), ("critic", nt.CRITIC_KEYS)):
        for name, seg in keys.items():
            assert np.array_equal(model.params.view(model.params.flat, seg).cpu().numpy(), ex[f"{tag}/{name}/param"]), name
            assert np.array_equal(model.params.view(model.exp_avg, seg).cpu().numpy(), ex[f"{tag}/{name}/exp_avg"]), name
            assert np.array_equal(model.params.view(model.exp_avg_sq, seg).cpu().numpy(), ex[f"{tag}/{name}/exp_avg_sq"]), name
    assert int(model.adam_step.item()) == int(ex["policy/policy_logstd/step"])
    model.train()
    assert int(model.adam_step.item()) > int(ex["policy/policy_logstd/step"])
    model.save()
    ck = torch.load(str(tmp_path / "run" / "models" / "best.model"), weights_only=False)
    assert list(ck["policy_state_dict"])[0] == "policy_logstd" and tuple(ck["policy_optimizer_state_dict"]["state"][0]["exp_avg"].shape) == (1, act)


@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_gpu_sharded_run_equals_single_gpu_run(tmp_path, gemm_engine, exchange):
    """Env-sharded data parallelism over 2 GPUs reproduces the 1-GPU run on the same global batch, with the gradient carried by
    the library's peer-memory all-reduce kernel ("peer") or by NCCL ("nccl")."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = os.path.join(root, "tests", "dist_check_ppo.py")
    w1, w2 = str(tmp_path / "w1.pt"), str(tmp_path / "w2.pt")
    subprocess.run([sys.executable, script, "--out", w1, "--engine", gemm_engine], check=True, timeout=600)
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                    "--master-port", "29631", script, "--out", w2, "--engine", gemm_engine, "--exchange", exchange], check=True, timeout=600)
    subprocess.run([sys.executable, script, "--compare", w1, w2], check=True, timeout=120)


def test_peer_allreduce_kernel_all_ranks_bit_identical(tmp_path):
    """rlx_comm_allreduce_sum_f32 over every visible GPU: exact integer-valued sums, identical bits on every rank, 2000 back-to-back
    calls (exercises the double-buffered slots and the flag protocol)."""
    import os
    import subprocess
    import sys
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = os.path.join(root, "tests", "dist_check_comm.py")
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(n, 8)), "--master-addr", "127.0.0.1",
                    "--master-port", "29633", script], check=True, timeout=600)
