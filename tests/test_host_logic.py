"""CPU-side tests: C-ABI surface, numpy-exact host RNG, reference-identical initialisation, config/runner plumbing,
shard index arithmetic (incl. a world_size-2 gloo run).  No CUDA compute is invoked here."""
import os
import re
import sys

import numpy as np
import pytest
import torch

from conftest import load_like_the_reference, reference_enums, reference_interfaces, reference_module, reference_optimizer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from rl_x_b200 import _native as nt
    import ctypes
    lib = nt.load()
    header = open(os.path.join(ROOT, "include", "rlx_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(rlx_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 25
    raw = ctypes.CDLL(nt.library_path())
    for name in sorted(declared):
        assert hasattr(raw, name), f"{name} declared in include/rlx_b200.h but not exported"
    assert declared == set(nt.exported_symbols()), declared ^ set(nt.exported_symbols())
    assert lib.rlx_version() == 1
    assert isinstance(nt.last_error(), str)


def test_param_layout_matches_reference_shapes():
    from rl_x_b200 import _native as nt
    off, crit = nt.ppo_layout(376, 17, 256)
    assert off[-1] == 329251  # SURVEY §8: 166 690 + 162 561
    shapes = nt.segment_shapes(376, 17, 256)
    for i, name in enumerate(nt.SEGMENT_NAMES):
        assert off[i + 1] - off[i] == int(np.prod(shapes[name]))
    assert sum(off[i + 1] - off[i] for i in range(13) if crit[i]) == 162561


@pytest.mark.parametrize("seed", [0, 1, 3, 12345, 2**40 + 17])
def test_pcg64_stream_is_numpy_exact(seed):
    from rl_x_b200 import _native as nt
    g, r = nt.Pcg64Generator(seed), np.random.default_rng(seed)
    st = r.bit_generator.state["state"]
    assert (g.state.s[0] << 64 | g.state.s[1], g.state.s[2] << 64 | g.state.s[3]) == (st["state"], st["inc"])
    for n in [0, 1, 2, 3, 10, 1000, 65536]:
        a, b = np.arange(n), np.arange(n)
        for _ in range(2):  # in-place re-shuffle continues the stream, like the epochs of ppo.py:274-276
            g.shuffle(a)
            r.shuffle(b)
            assert np.array_equal(a, b)
    for high in [1, 2, 4, 977, 10**6, 2**32 - 1, 2**32, 2**32 + 5, 2**40]:
        assert np.array_equal(g.integers(high, 1001), r.integers(high, size=1001))
    assert g.next_uint64() == int(r.bit_generator.random_raw())


@pytest.mark.parametrize("seed", [0, 7, 123456789])
def test_pcg64_choice_without_replacement_is_numpy_exact(seed):
    """Generator.choice(pop, size, replace=False) (espo.py:256): both of numpy's branches (Floyd + hash set, tail shuffle), interleaved
    with shuffles on the same stream, and the stream position afterwards."""
    from rl_x_b200 import _native as nt
    g, r = nt.Pcg64Generator(seed), np.random.default_rng(seed)
    for pop, size in [(10, 3), (10, 10), (1, 1), (5, 0), (2048, 64), (2048, 2048), (10001, 100), (10001, 201), (20000, 400), (20000, 401),
                      (32768, 4096), (131072, 64)]:
        for _ in range(2):
            assert np.array_equal(g.choice(pop, size), r.choice(pop, size=size, replace=False)), (pop, size)
        a, b = np.arange(17), np.arange(17)
        g.shuffle(a)
        r.shuffle(b)
        assert np.array_equal(a, b)
    assert g.next_uint64() == int(r.bit_generator.random_raw())
    with pytest.raises(RuntimeError):
        g.choice(4, 5)


def test_pcg64_matches_golden_permutations(golden):
    from rl_x_b200 import _native as nt
    g = nt.Pcg64Generator(golden.seed)
    k = 0
    for it in range(golden.iterations):
        idx = np.arange(golden.B)
        for _ in range(golden.epochs):
            g.shuffle(idx)
            assert np.array_equal(idx, golden[f"perm/{k}"])
            k += 1


def test_pcg64_rejects_bad_arrays():
    from rl_x_b200 import _native as nt
    g = nt.Pcg64Generator(1)
    with pytest.raises(TypeError):
        g.shuffle(np.arange(10, dtype=np.int32))
    with pytest.raises(RuntimeError):
        g.integers(0, 5)


def test_initial_parameters_identical_to_reference(golden):
    from rl_x_b200.algorithms.ppo.b200.ppo import init_reference_parameters
    nthreads = torch.get_num_threads()
    torch.set_num_threads(1)  # the fixture was generated single-threaded; LAPACK's QR rounds differently per thread count / CPU
    try:
        named = init_reference_parameters(golden.obs, golden.act, golden.hidden, golden.std_dev, golden.seed)
    finally:
        torch.set_num_threads(nthreads)
    pol, cri = golden.params("init")
    for k, v in {**pol, **cri}.items():
        # same RNG stream and same call order; the QR inside orthogonal_ is LAPACK and differs by an ulp with the thread count
        np.testing.assert_allclose(named[k].numpy(), v, rtol=1e-5, atol=1e-5, err_msg=k)


def test_config_overrides_and_runner_show_config():
    from rl_x_b200.runner.runner import Runner
    r = Runner(argv=["--runner.mode=show_config", "--algorithm.nr_steps=128", "--environment.nr_envs=64",
                     "--algorithm.anneal_learning_rate=True", "--algorithm.learning_rate=1e-3"])
    c = r._config
    assert c.algorithm.nr_steps == 128 and c.environment.nr_envs == 64 and c.algorithm.anneal_learning_rate is True
    assert c.algorithm.learning_rate == 1e-3 and c.algorithm.name == "ppo.b200" and c.environment.name == "synthetic.box"
    assert sorted(r._explicitly_set) == ["algorithm.anneal_learning_rate", "algorithm.learning_rate", "algorithm.nr_steps", "environment.nr_envs"]
    with pytest.raises(KeyError):
        Runner(argv=["--algorithm.no_such_key=1"])
    with pytest.raises(ModuleNotFoundError):
        Runner(argv=["--algorithm.name=does.not.exist"])


def test_default_config_keys_cover_reference_keys():
    from rl_x_b200.algorithms.ppo.b200.default_config import get_config
    ref_keys = ["name", "device", "compile_mode", "bf16_mixed_precision_training", "total_timesteps", "learning_rate", "anneal_learning_rate",
                "nr_steps", "nr_epochs", "minibatch_size", "gamma", "gae_lambda", "clip_range", "entropy_coef", "critic_coef", "max_grad_norm",
                "std_dev", "action_clipping_and_rescaling", "nr_hidden_units", "evaluation_frequency", "evaluation_episodes"]
    c = get_config("ppo.b200")
    for k in ref_keys:  # rl_x/algorithms/ppo/pytorch/default_config.py:4-30
        assert k in c, k
    assert (c.nr_steps, c.nr_epochs, c.minibatch_size, c.gamma, c.gae_lambda, c.clip_range) == (2048, 10, 64, 0.99, 0.95, 0.2)


def test_espo_plugin_registers_with_reference_keys():
    """espo.b200 registers like the reference's espo.pytorch (espo/pytorch/__init__.py) and its default config carries every key of
    rl_x/algorithms/espo/pytorch/default_config.py:4-30."""
    import rl_x_b200.algorithms.espo.b200  # noqa: F401  (registers)
    from rl_x_b200.algorithms.algorithm_manager import get_algorithm_config, get_algorithm_model_class
    cfg = get_algorithm_config("espo.b200")
    for key in ["name", "device", "compile_mode", "bf16_mixed_precision_training", "total_timesteps", "learning_rate", "anneal_learning_rate",
                "nr_steps", "max_epochs", "minibatch_size", "gamma", "gae_lambda", "max_ratio_delta", "delta_calc_operator", "entropy_coef",
                "critic_coef", "max_grad_norm", "std_dev", "action_clipping_and_rescaling", "nr_hidden_units", "evaluation_frequency",
                "evaluation_episodes"]:
        assert key in cfg, key
    assert (cfg.max_epochs, cfg.max_ratio_delta, cfg.delta_calc_operator) == (300, 0.25, "mean")
    assert get_algorithm_model_class("espo.b200").__name__ == "ESPO"


def test_ppo_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from rl_x_b200.runner.runner import Runner
    r = Runner(argv=["--environment.nr_envs=8", "--algorithm.nr_steps=4", "--algorithm.minibatch_size=8"])
    from rl_x_b200.algorithms.ppo.b200.ppo import PPO
    train_env, eval_env = r._create_train_and_eval_env(r._config)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PPO(r._config, train_env, eval_env, "/tmp/x", None)


def test_ppo_rejects_unknown_peer_exchange_algorithm():
    """algorithm.peer_exchange_algorithm accepts auto | one_shot (the one-shot kernel is the only peer all-reduce); anything else is
    refused before anything runs."""
    from rl_x_b200.runner.runner import Runner
    from rl_x_b200.algorithms.ppo.b200.ppo import PPO
    r = Runner(argv=["--environment.nr_envs=8", "--algorithm.nr_steps=4", "--algorithm.minibatch_size=8", "--algorithm.peer_exchange_algorithm=ring"])
    train_env, eval_env = r._create_train_and_eval_env(r._config)
    with pytest.raises(ValueError, match="peer_exchange_algorithm must be 'auto' or 'one_shot'"):
        PPO(r._config, train_env, eval_env, "/tmp/x", None)


@pytest.mark.parametrize("algo", ["sac.b200", "fastsac.b200", "ppo_lstm.b200"])
def test_non_identity_observation_indices_are_rejected_not_ignored(algo):
    """SURVEY §8 a20: the reference index-selects the network inputs with env.policy_observation_indices / critic_observation_indices
    (sac/pytorch/policy.py:13,46, q_network.py:10,37 and the same lines in fastsac / ppo_lstm).  The kernels here read whole rows, so an
    env that asks for a subset must be refused before anything runs (PPO / ESPO check the same thing after their device check)."""
    from rl_x_b200.runner.runner import Runner
    from rl_x_b200.algorithms.algorithm_manager import get_algorithm_model_class
    r = Runner(argv=[f"--algorithm.name={algo}", "--environment.nr_envs=8"])
    env, eval_env = r._create_train_and_eval_env(r._config)
    cls = get_algorithm_model_class(algo)
    obs = env.single_observation_space.shape[0]
    env.policy_observation_indices = np.arange(obs)            # identity: accepted (the next check is the device one)
    expected = RuntimeError if not torch.cuda.is_available() else None
    if expected:
        with pytest.raises(expected, match="no CPU fallback"):
            cls(r._config, env, eval_env, "/tmp/x", None)
    env.critic_observation_indices = np.arange(obs - 1)        # the critic sees a subset: refused
    with pytest.raises(ValueError, match="non-identity critic_observation_indices"):
        cls(r._config, env, eval_env, "/tmp/x", None)


def test_synthetic_env_contract():
    from rl_x_b200.runner.runner import Runner
    r = Runner(argv=["--environment.nr_envs=8", "--environment.device=cpu", "--algorithm.device=cpu", "--environment.horizon=3"])
    env, eval_env = r._create_train_and_eval_env(r._config)
    assert env is eval_env
    obs, info = env.reset()
    assert obs.shape == (8, 376) and info == {}
    for t in range(1, 4):
        o, rew, term, trunc, info = env.step(torch.zeros(8, 17))
        assert o.shape == (8, 376) and rew.shape == (8,) and term.dtype == torch.bool and trunc.dtype == torch.bool
        assert bool(trunc.all()) == (t % 3 == 0)
    assert env.get_logging_info_dict(info) == {}
    assert env.single_action_space.low.shape == (17,) and env.general_properties.data_interface_type.name == "TORCH"


# ------------------------------------------------------------------------------------------------------- sharding
def test_local_rows_partition_the_permutation():
    from rl_x_b200.algorithms.ppo.b200 import sharding
    T, Ng, W, mb = 7, 12, 4, 10
    Nl = Ng // W
    perm = np.random.default_rng(0).permutation(T * Ng)
    gsizes = sharding.global_minibatch_sizes(T * Ng, mb)
    assert gsizes.sum() == T * Ng and gsizes[-1] == (T * Ng) % mb
    total = np.zeros(len(gsizes), dtype=np.int64)
    seen = []
    for rank in range(W):
        idx, counts = sharding.local_rows_of_permutation(perm, mb, Ng, Nl, rank)
        assert idx.shape[0] == T * Nl and sorted(idx.tolist()) == list(range(T * Nl))
        total += counts
        # map local rows back to global flat indices and check order within each minibatch
        t, e = np.divmod(idx, Nl)
        glob = t * Ng + e + rank * Nl
        off = np.concatenate([[0], np.cumsum(counts)])
        for k in range(len(counts)):
            mine = [p for p in perm[k * mb:(k + 1) * mb] if (p % Ng) // Nl == rank]
            assert glob[off[k]:off[k + 1]].tolist() == mine
        seen.extend(glob.tolist())
    assert np.array_equal(total, gsizes) and sorted(seen) == list(range(T * Ng))


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from oracle import ppo_oracle as O
    from rl_x_b200.algorithms.ppo.b200 import sharding
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    T, Ng, obs, act, H, mb = 6, 8, 5, 2, 16, 16
    Nl = Ng // world
    g = torch.Generator().manual_seed(0)
    states = torch.randn(T, Ng, obs, generator=g)
    actions = torch.randn(T, Ng, act, generator=g)
    logp = torch.randn(T, Ng, generator=g) * 0.1 - 2.0
    adv = torch.randn(T, Ng, generator=g)
    ret = torch.randn(T, Ng, generator=g)
    pol, cri = O.init_params(obs, act, H, seed=5)
    perm = np.random.default_rng(3).permutation(T * Ng)
    full = O.Learner(pol, cri)
    flat = lambda x: x.reshape((-1,) + x.shape[2:])
    idx0 = torch.as_tensor(perm[:mb])
    gp_full, gc_full, m_full = full.grads(flat(states)[idx0], flat(actions)[idx0], flat(logp)[idx0], flat(adv)[idx0], flat(ret)[idx0])

    # sharded: this rank's rows of minibatch 0, global advantage statistics, gradient SUM / global size
    sl = sharding.shard_env_slice(Ng, world, rank)
    loc = lambda x: x[:, sl].reshape((-1,) + x.shape[2:])
    lidx, counts = sharding.local_rows_of_permutation(perm, mb, Ng, Nl, rank)
    rows = torch.as_tensor(lidx[:counts[0]])
    a_loc = loc(adv)[rows]
    s = torch.stack([a_loc.sum(), torch.tensor(float(len(rows)))])
    dist.all_reduce(s)
    mean = s[0] / s[1]
    ssq = ((a_loc - mean) ** 2).sum()
    dist.all_reduce(ssq)
    std = torch.sqrt(ssq / (s[1] - 1))
    L = O.Learner(pol, cri)
    new_logp, _ = O.get_logprob_entropy(L.pol, loc(states)[rows], loc(actions)[rows])
    ratio = (new_logp - loc(logp)[rows]).exp()
    A = (a_loc - mean) / (std + 1e-8)
    pg = torch.maximum(-A * ratio, -A * torch.clamp(ratio, 0.8, 1.2)).sum() / mb
    closs = 0.5 * (0.5 * (O.critic_value(L.cri, loc(states)[rows]).reshape(-1) - loc(ret)[rows]) ** 2).sum() / mb
    (pg + closs).backward()
    err = 0.0
    for k in O.POLICY_KEYS:
        gsum = L.pol[k].grad.clone()
        dist.all_reduce(gsum)
        err = max(err, float((gsum - gp_full[k]).abs().max()))
    for k in O.CRITIC_KEYS:
        gsum = L.cri[k].grad.clone()
        dist.all_reduce(gsum)
        err = max(err, float((gsum - gc_full[k]).abs().max()))
    dist.destroy_process_group()
    q.put((rank, err))


def test_sharded_gradient_equals_single_process_gloo_world2():
    """The data-parallel recipe (global permutation, owner-computes rows, global advantage statistics, gradient sums
    divided by the global minibatch size, all-reduce(sum)) reproduces the unsharded minibatch gradient."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, err in results:
        assert err < 5e-7, (rank, err)


# ------------------------------------------------------------------------------------------- checkpoint interoperability
def _ckpt_fixture():
    from rl_x_b200.algorithms.ppo.b200.kernels import PpoKernels
    from rl_x_b200.algorithms.ppo.b200.ppo import FlatParameters
    ck = torch.load(os.path.join(ROOT, "tests", "golden", "ppo_ref_checkpoint.model"), weights_only=False)
    ex = np.load(os.path.join(ROOT, "tests", "golden", "ppo_ref_checkpoint_expect.npz"))
    N, T, obs, act, hid, mb, E = (int(x) for x in ex["meta"])
    k = PpoKernels(obs, act, hid)
    return ck, ex, k, FlatParameters(k, "cpu")


def test_checkpoint_written_by_the_reference_maps_onto_the_flat_layout():
    """tests/golden/ppo_ref_checkpoint.model was written by the executed reference's own PPO.save() (make_golden_ppo_ckpt.py).  Its
    optimizer states are numbered in nn.Module.parameters() order - policy_logstd FIRST - and must land on the right segments."""
    from rl_x_b200 import _native as nt
    from rl_x_b200.algorithms.ppo.b200.ppo import CRITIC_PARAM_ORDER, POLICY_PARAM_ORDER
    ck, ex, k, fp = _ckpt_fixture()
    assert list(ck["policy_state_dict"]) == list(POLICY_PARAM_ORDER) and list(ck["critic_state_dict"]) == list(CRITIC_PARAM_ORDER)
    fp.load_named({**ck["policy_state_dict"], **ck["critic_state_dict"]})
    m1, m2 = torch.zeros(k.param_count), torch.zeros(k.param_count)
    sp = fp.load_adam_state(ck["policy_optimizer_state_dict"], POLICY_PARAM_ORDER, nt.POLICY_KEYS, m1, m2)
    sc = fp.load_adam_state(ck["critic_optimizer_state_dict"], CRITIC_PARAM_ORDER, nt.CRITIC_KEYS, m1, m2)
    for tag, keys in (("policy", nt.POLICY_KEYS), ("critic", nt.CRITIC_KEYS)):
        for name, seg in keys.items():
            assert np.array_equal(fp.view(fp.flat, seg).numpy(), ex[f"{tag}/{name}/param"]), name
            assert np.array_equal(fp.view(m1, seg).numpy(), ex[f"{tag}/{name}/exp_avg"]), name
            assert np.array_equal(fp.view(m2, seg).numpy(), ex[f"{tag}/{name}/exp_avg_sq"]), name
            assert float(ex[f"{tag}/{name}/step"]) == sp == sc
    # and back: what save() writes is, tensor for tensor and index for index, what the reference wrote
    pol, cri = fp.state_dicts()
    assert list(pol) == list(ck["policy_state_dict"]) and all(torch.equal(pol[n], ck["policy_state_dict"][n]) for n in pol)
    assert list(cri) == list(ck["critic_state_dict"]) and all(torch.equal(cri[n], ck["critic_state_dict"][n]) for n in cri)
    for key, order, keys in (("policy_optimizer_state_dict", POLICY_PARAM_ORDER, nt.POLICY_KEYS), ("critic_optimizer_state_dict", CRITIC_PARAM_ORDER, nt.CRITIC_KEYS)):
        ours, ref = fp.adam_state_dict(order, keys, m1, m2, sp, 3e-4), ck[key]
        assert ours["param_groups"][0]["params"] == ref["param_groups"][0]["params"]
        assert set(ours["param_groups"][0]) == set(ref["param_groups"][0])
        for i in ref["state"]:
            for f in ("exp_avg", "exp_avg_sq"):
                assert torch.equal(ours["state"][i][f], ref["state"][i][f]), (key, i, f)
            assert float(ours["state"][i]["step"]) == float(ref["state"][i]["step"])
    # a permuted optimizer state (the round-1 bug: logstd last) is rejected instead of being mis-assigned
    bad = {"state": {i: ck["policy_optimizer_state_dict"]["state"][(i + 1) % 7] for i in range(7)}}
    with pytest.raises(ValueError, match="expected"):
        fp.load_adam_state(bad, POLICY_PARAM_ORDER, nt.POLICY_KEYS, m1, m2)
    # torch builds that keep the compile wrapper's prefix in state_dict()
    fp2 = fp.__class__(k, "cpu")
    fp2.load_named({"_orig_mod." + n: v for n, v in {**ck["policy_state_dict"], **ck["critic_state_dict"]}.items()})
    assert torch.equal(fp2.flat, fp.flat)


def test_checkpoint_written_here_loads_into_the_reference_modules():
    """The other direction: strict load_state_dict + optimizer.load_state_dict as in the reference's load() (ppo.py:447-450), into modules
    and Adam optimizers laid out as the reference's (parameter names, shapes, order, optimizer numbering and settings captured from the
    executed reference in tests/golden/reference_interfaces.json)."""
    from rl_x_b200 import _native as nt
    from rl_x_b200.algorithms.ppo.b200.kernels import PpoKernels
    from rl_x_b200.algorithms.ppo.b200.ppo import CRITIC_PARAM_ORDER, FlatParameters, POLICY_PARAM_ORDER
    ref = reference_interfaces()["checkpoints"]["ppo"]
    meta = ref["meta"]
    k = PpoKernels(meta["obs"], meta["act"], meta["hidden"])
    fp = FlatParameters(k, "cpu")
    g = torch.Generator().manual_seed(0)
    fp.flat.copy_(torch.randn(k.param_count, generator=g))
    m1, m2 = torch.randn(k.param_count, generator=g), torch.rand(k.param_count, generator=g)
    pol, cri = fp.state_dicts()
    policy, critic = reference_module(ref["modules"]["policy"]), reference_module(ref["modules"]["critic"])
    policy.load_state_dict(pol)
    critic.load_state_dict(cri)
    popt = reference_optimizer(ref["optimizers"]["policy_optimizer"], {"": policy})
    copt = reference_optimizer(ref["optimizers"]["critic_optimizer"], {"": critic})
    popt.load_state_dict(fp.adam_state_dict(POLICY_PARAM_ORDER, nt.POLICY_KEYS, m1, m2, 5, 3e-4))
    copt.load_state_dict(fp.adam_state_dict(CRITIC_PARAM_ORDER, nt.CRITIC_KEYS, m1, m2, 5, 3e-4))
    for net, opt, keys in ((policy, popt, nt.POLICY_KEYS), (critic, copt, nt.CRITIC_KEYS)):
        for name, p in net.named_parameters():
            seg = keys[name]
            assert torch.equal(p.detach(), fp.view(fp.flat, seg)), name
            assert torch.equal(opt.state[p]["exp_avg"], fp.view(m1, seg)) and torch.equal(opt.state[p]["exp_avg_sq"], fp.view(m2, seg)), name
            assert float(opt.state[p]["step"]) == 5.0


# ------------------------------------------------------------------------------------------------- config 1: Pendulum-v1
def test_pendulum_restates_the_published_dynamics_and_the_autoreset_convention():
    """BASELINE.json configs[0].  Known answers computed by hand from the published Pendulum-v1 update rule (see environment.py), plus the
    gymnasium-0.29 vector autoreset convention the reference's wrapper reads (gym/mujoco/humanoid_v4/wrappers.py:9-32)."""
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.environments.synthetic.pendulum import create_train_and_eval_env, get_config
    from rl_x_b200.environments.synthetic.pendulum.environment import angle_normalize
    cfg = ConfigDict(environment=get_config("synthetic.pendulum"))
    env, eval_env = create_train_and_eval_env(cfg)
    assert env is eval_env and env.nr_envs == 4 and env.general_properties.data_interface_type.name == "NUMPY"
    assert env.single_observation_space.shape == (3,) and env.single_action_space.shape == (1,)
    assert float(env.single_action_space.low[0]) == -2.0 and float(env.single_action_space.high[0]) == 2.0
    assert abs(angle_normalize(3 * np.pi / 2) + np.pi / 2) < 1e-12 and abs(angle_normalize(-np.pi) + np.pi) < 1e-12
    obs, info = env.reset(seed=5)
    rng = np.random.default_rng(5)  # sub-env 0 owns default_rng(seed + 0)
    th, thdot = rng.uniform(low=[-np.pi, -1.0], high=[np.pi, 1.0])
    np.testing.assert_allclose(obs[0], [np.cos(th), np.sin(th), thdot], rtol=1e-6)
    u = 3.5  # clipped to max_torque 2
    obs1, rew, term, trunc, info = env.step(np.full((4, 1), u))
    cost = angle_normalize(th) ** 2 + 0.1 * thdot ** 2 + 0.001 * 2.0 ** 2
    thdot1 = np.clip(thdot + (15.0 * np.sin(th) + 3.0 * 2.0) * 0.05, -8, 8)
    th1 = th + thdot1 * 0.05
    assert abs(rew[0] + cost) < 1e-12 and not term.any() and not trunc.any() and info == {}
    np.testing.assert_allclose(obs1[0], [np.cos(th1), np.sin(th1), thdot1], rtol=1e-6)
    total = rew.copy()
    for t in range(2, 201):
        obs_t, rew, term, trunc, info = env.step(np.zeros((4, 1)))
        total += rew
        if t < 200:
            assert not trunc.any() and info == {}
    assert trunc.all() and not term.any()  # TimeLimit(200)
    log = env.get_logging_info_dict(info)
    np.testing.assert_allclose(log["episode_return"], total, rtol=1e-12)
    assert log["episode_length"] == [200.0] * 4
    final0 = env.get_final_observation_at_index(info, 0)
    assert final0.shape == (3,) and not np.array_equal(final0, obs_t[0])  # obs_t is already the next episode's first observation
    assert env.get_final_info_value_at_index(info, "episode_return", 2) == log["episode_return"][2]
    assert abs(np.hypot(obs_t[:, 0], obs_t[:, 1]) - 1).max() < 1e-6 and np.abs(obs_t[:, 2]).max() <= 1.0  # fresh reset states


def test_tanh_fast_error_model():
    """csrc/common.cuh::tanh_fast (the tensor-engine epilogues' tanh) restated in fp32 numpy arithmetic with the MUFU approximations at their
    documented worst (ex2.approx 2 ulp, rcp.approx 1 ulp, both signs): max relative error < 6e-7 over a dense sample incl. the branch point at
    |x| = 0.25 and the saturation region, rms < 1e-7 - the accuracy class of the 3xTF32 products feeding it, far inside the 1e-5 parity bar.
    (The kernel itself is covered on the GPU by every forward / gradient parity test.)"""
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.normal(0, 1.5, 400_000), rng.uniform(-0.4, 0.4, 200_000), np.linspace(-9, 9, 40_001),
                        [0.0, 0.25, -0.25, np.nextafter(np.float32(0.25), 0), 15.0, 20.0, -30.0]]).astype(np.float32)
    ref = np.tanh(x.astype(np.float64))

    def tanh_fast(x, worst):
        f = np.float32
        x2 = x * x
        p = x2 * f(62 / 2835) + f(-17 / 315)
        p = p * x2 + f(2 / 15)
        p = p * x2 + f(-1 / 3)
        p = p * x2 + f(1.0)
        small = (x * p).astype(np.float32)
        ax = np.minimum(np.abs(x), f(15.0))
        e = np.exp2((ax * f(2.885390081777927)).astype(np.float32).astype(np.float64)).astype(np.float32)
        e = (e * f(1 + worst * 2 * 2.0 ** -23)).astype(np.float32)
        r = (f(1) / (e + f(1))).astype(np.float32)
        r = (r * f(1 + worst * 2.0 ** -23)).astype(np.float32)
        big = np.copysign((f(1) - f(2) * r).astype(np.float32), x)
        return np.where(np.abs(x) < f(0.25), small, big)

    for worst in (0, 1, -1):
        y = tanh_fast(x, worst).astype(np.float64)
        rel = np.abs(y - ref) / np.maximum(np.abs(ref), 1e-30)
        rel[ref == 0] = np.abs(y[ref == 0])
        assert rel.max() < 6e-7, (worst, rel.max())
        assert np.sqrt(np.mean(rel ** 2)) < 1e-7


def test_build_digest_does_not_depend_on_the_checkout_path(tmp_path, monkeypatch):
    """The freshness stamp travels with the prebuilt .so to a box where the tree lives under another path; there the library must still count
    as fresh, or every rank of a torchrun job would start recompiling it at the same time."""
    import shutil
    from rl_x_b200 import build as b
    here = b._digest()
    other = tmp_path / "elsewhere"
    shutil.copytree(b.CSRC, other / "csrc")
    shutil.copytree(b.INCLUDE, other / "include")
    monkeypatch.setattr(b, "CSRC", str(other / "csrc"))
    monkeypatch.setattr(b, "INCLUDE", str(other / "include"))
    assert b._digest() == here
    with open(other / "csrc" / "gae.cu", "a") as fh:
        fh.write("\n// changed\n")
    assert b._digest() != here


def _last_json_line(path):
    import json
    with open(path) as fh:
        lines = [ln for ln in fh.read().splitlines() if ln.startswith("{")]
    return json.loads(lines[-1])


def test_committed_bench_records_carry_the_contract_keys():
    """The bench lines committed under profiles/ (the last hardware runs of `python bench.py` and `bench.py --impl reference`) against the
    key list of the measurement contract: a renamed or dropped key would otherwise only be noticed by the driver."""
    import os
    prof = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles")
    line = _last_json_line(os.path.join(prof, "r02_bench_1gpu.json"))
    for key in ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "gpu_launches", "clocks", "roofline", "cpu_baseline", "e2e"]:
        assert key in line, key
    assert line["n_gpus"] == 1 and line["warmup"] >= 3 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["dtype"] == "f32" and line["data"] == "synthetic" and "workload" in line["config"] and "model" not in line["config"]
    assert abs(line["value"] - 4096 * 128 / (line["ms_per_step"] * 1e-3)) <= 1e-6 * line["value"]       # value and ms_per_step tell one story
    roof = line["roofline"]
    assert set(["bound", "achieved", "peak", "unit", "frac", "traffic"]) <= set(roof) and roof["bound"] in ("hbm", "tensor")
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) <= 1e-9
    assert set(["value", "unit", "cores", "kind", "sample"]) <= set(line["cpu_baseline"]) and line["cpu_baseline"]["kind"] in ("reference", "port")
    e2e = line["e2e"]
    assert set(["value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"]) <= set(e2e) and e2e["h2d_bytes_per_step"] > 0 < e2e["d2h_bytes_per_step"]
    assert e2e["value"] < line["value"]                              # host copies inside the timed region cannot be free
    assert set(["sm_mhz", "sm_max_mhz", "reasons"]) <= set(line["clocks"]) and line["gpu_launches"] > 0
    assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    ref = _last_json_line(os.path.join(prof, "r02_reference_arm.json"))
    assert ref["impl"] == "reference" and ref["metric"] == line["metric"] and ref["unit"] == line["unit"] and ref["config"]["workload"] == line["config"]["workload"]
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 == ref["e2e"]["d2h_bytes_per_step"] and ref["e2e"]["value"] == ref["value"]
    assert ref["cpu_baseline"]["kind"] == "reference" and ref["cpu_baseline"]["value"] == ref["value"]


def test_sac_checkpoint_written_by_the_reference_maps_onto_the_flat_layout():
    """tests/golden/sac_ref_checkpoint.model was written by the executed reference's own SAC.save() (make_golden_sac_ckpt.py).  Module keys,
    the parameter numbering inside the three Adam state dicts (policy; q1 then q2; log_alpha - sac.py:75-77) and the param_group keys
    must be what rl_x_b200's SAC.load() / save() assume: every tensor lands on its segment of the flat buffers, and the dicts save()
    builds from those buffers equal the reference's entry for entry."""
    from rl_x_b200.algorithms.sac.b200 import sac as S
    ck = torch.load(os.path.join(ROOT, "tests", "golden", "sac_ref_checkpoint.model"), weights_only=False)
    ex = np.load(os.path.join(ROOT, "tests", "golden", "sac_ref_checkpoint_expect.npz"))
    N, obs, act, hid, batch = (int(x) for x in ex["meta"])
    k = S.SacKernels(obs, act, hid, -5.0, 2.0)
    strip = lambda d: {key.replace("_orig_mod.", ""): v for key, v in d.items()}
    assert list(strip(ck["policy_state_dict"])) == list(S.POLICY_PARAM_ORDER)
    for net in ("q1", "q2", "q1_target", "q2_target"):
        assert list(strip(ck[f"{net}_state_dict"])) == list(S.Q_PARAM_ORDER)
    # parameters: what load_named() does, on CPU flats
    policy, q = torch.zeros(k.Pp), torch.zeros(4 * k.Pq)
    pv, qv = k.policy_views(policy), k.q_views(q)
    for key, v in strip(ck["policy_state_dict"]).items():
        pv[key].copy_(v.detach().reshape(pv[key].shape))
        assert np.array_equal(pv[key].numpy(), ex[f"policy/{key}/param"]), key
    for net in S.Q_NETS:
        for key, v in strip(ck[f"{net}_state_dict"]).items():
            qv[net][key].copy_(v.detach().reshape(qv[net][key].shape))
            assert np.array_equal(qv[net][key].numpy(), ex[f"{net}/{key}/param"]), (net, key)
    assert np.array_equal(torch.as_tensor(ck["log_alpha"]).detach().numpy().reshape(-1), ex["log_alpha/param"].reshape(-1))
    # optimizer states: the views SAC._optimizer_views() hands to _load_adam_state, rebuilt here on CPU flats
    m_p, v_p, m_q, v_q, m_a, v_a = torch.zeros(k.Pp), torch.zeros(k.Pp), torch.zeros(2 * k.Pq), torch.zeros(2 * k.Pq), torch.zeros(1), torch.zeros(1)
    pol_views = lambda flat: [k.policy_views(flat)[name] for name in S.POLICY_PARAM_ORDER]

    def q_views(flat):  # q1's six tensors, then q2's
        both = k.q_views(torch.cat([flat, torch.zeros(2 * k.Pq)]))   # q_views expects the four-net buffer; only q1 / q2 are looked at
        return [both[net][name] for net in ("q1", "q2") for name in S.Q_PARAM_ORDER]

    steps = S._load_adam_state(ck["policy_optimizer_state_dict"], pol_views(m_p), pol_views(v_p), "policy")
    for name, m, v in zip(S.POLICY_PARAM_ORDER, pol_views(m_p), pol_views(v_p)):
        assert np.array_equal(m.numpy(), ex[f"policy/{name}/exp_avg"]) and np.array_equal(v.numpy(), ex[f"policy/{name}/exp_avg_sq"]), name
        assert float(ex[f"policy/{name}/step"]) == steps
    qm, qvv = [torch.zeros_like(t) for t in q_views(m_q)], [torch.zeros_like(t) for t in q_views(v_q)]
    q_steps = S._load_adam_state(ck["q_optimizer_state_dict"], qm, qvv, "q")
    names = [(net, name) for net in ("q1", "q2") for name in S.Q_PARAM_ORDER]
    for (net, name), m, v in zip(names, qm, qvv):
        assert np.array_equal(m.numpy(), ex[f"{net}/{name}/exp_avg"]) and np.array_equal(v.numpy(), ex[f"{net}/{name}/exp_avg_sq"]), (net, name)
        assert float(ex[f"{net}/{name}/step"]) == q_steps
    a_steps = S._load_adam_state(ck["entropy_optimizer_state_dict"], [m_a], [v_a], "entropy")
    assert np.array_equal(m_a.numpy(), ex["log_alpha/exp_avg"].reshape(-1)) and float(ex["log_alpha/step"]) == a_steps
    # and back: the state dicts save() builds are, key for key and tensor for tensor, what the reference wrote
    for key, (ms, vs, st) in (("policy_optimizer_state_dict", (pol_views(m_p), pol_views(v_p), steps)), ("q_optimizer_state_dict", (qm, qvv, q_steps)),
                             ("entropy_optimizer_state_dict", ([m_a], [v_a], a_steps))):
        ours, ref = S._adam_state_dict(ms, vs, st, ck[key]["param_groups"][0]["lr"]), ck[key]
        assert ours["param_groups"][0]["params"] == ref["param_groups"][0]["params"]
        assert set(ours["param_groups"][0]) == set(ref["param_groups"][0]), set(ours["param_groups"][0]) ^ set(ref["param_groups"][0])
        assert set(ours["state"]) == set(ref["state"])
        for i in ref["state"]:
            for f in ("exp_avg", "exp_avg_sq"):
                assert torch.equal(ours["state"][i][f].reshape(ref["state"][i][f].shape), ref["state"][i][f]), (key, i, f)
            assert float(ours["state"][i]["step"]) == float(ref["state"][i]["step"])
    # a state of the wrong shape (e.g. a permuted numbering) is refused, not mis-assigned
    bad = {"state": {0: ck["policy_optimizer_state_dict"]["state"][1]}}
    with pytest.raises(ValueError, match="expected"):
        S._load_adam_state(bad, pol_views(m_p), pol_views(v_p), "policy")


def test_sac_checkpoint_written_here_loads_into_the_reference_modules(tmp_path):
    """The other direction for SAC: the state dicts SAC.save() builds from the flat buffers go through strict load_state_dict /
    optimizer.load_state_dict exactly as the reference's load() does (sac.py:398-416), into modules and optimizers laid out as the
    reference's (tests/golden/reference_interfaces.json), and every parameter / Adam moment ends up where its name says."""
    from rl_x_b200.algorithms.sac.b200 import sac as S
    from rl_x_b200.algorithms.sac.b200.default_config import get_config
    ref = reference_interfaces()["checkpoints"]["sac"]
    obs, act, hid = ref["meta"]["obs"], ref["meta"]["act"], ref["meta"]["hidden"]
    a = get_config("sac.b200")
    a.nr_hidden_units = hid
    k = S.SacKernels(obs, act, hid, float(a.log_std_min), float(a.log_std_max))
    g = torch.Generator().manual_seed(1)
    policy, q = torch.randn(k.Pp, generator=g), torch.randn(4 * k.Pq, generator=g)
    m_p, v_p, m_q, v_q = torch.randn(k.Pp, generator=g), torch.rand(k.Pp, generator=g), torch.randn(4 * k.Pq, generator=g), torch.rand(4 * k.Pq, generator=g)
    pv, qv = k.policy_views(policy), k.q_views(q)
    pm, pvv = k.policy_views(m_p), k.policy_views(v_p)
    qm, qvv = k.q_views(m_q), k.q_views(v_q)
    # the whole file, as save() assembles it (checkpoint_dict), through the reference's load(): its assignment of checkpoint["log_alpha"]
    # to a registered parameter only accepts an nn.Parameter
    views = {"policy": ([pm[n] for n in S.POLICY_PARAM_ORDER], [pvv[n] for n in S.POLICY_PARAM_ORDER]),
             "q": ([qm[net][n] for net in ("q1", "q2") for n in S.Q_PARAM_ORDER], [qvv[net][n] for net in ("q1", "q2") for n in S.Q_PARAM_ORDER]),
             "entropy": ([torch.tensor([0.25])], [torch.tensor([0.5])])}
    path = str(tmp_path / "best.model")
    torch.save(S.checkpoint_dict(a, {n: pv[n].clone() for n in pv}, {net: {n: t.clone() for n, t in d.items()} for net, d in qv.items()},
                                 torch.tensor([-0.7]), views, [7, 7, 7], 3e-4), path)
    mods, opts, ent = load_like_the_reference(path, ref)
    assert isinstance(ent.log_alpha, torch.nn.Parameter) and float(ent.log_alpha.detach()) == pytest.approx(-0.7)
    for name, p in mods["policy"].named_parameters():
        st = opts["policy_optimizer"].state[p]
        assert torch.equal(p.detach(), pv[name]) and torch.equal(st["exp_avg"], pm[name]) and torch.equal(st["exp_avg_sq"], pvv[name]), name
        assert float(st["step"]) == 7.0
    for net in ("q1", "q2", "q1_target", "q2_target"):
        for name, p in mods[net].named_parameters():
            assert torch.equal(p.detach(), qv[net][name]), (net, name)
            if net in ("q1", "q2"):
                st = opts["q_optimizer"].state[p]
                assert torch.equal(st["exp_avg"], qm[net][name]) and torch.equal(st["exp_avg_sq"], qvv[net][name]), (net, name)
    st = next(iter(opts["entropy_optimizer"].state.values()))
    assert float(st["exp_avg"]) == 0.25 and float(st["exp_avg_sq"]) == 0.5 and float(st["step"]) == 7.0


def test_plugins_pass_the_reference_runners_compatibility_check():
    """Drop-in at the plugin level (INTEGRATION.md 1): this package's plugins put through the expressions of the reference's runner
    (rl_x/runner/runner.py:86-101) with the reference's enum members on the environment side.  Those expressions use `in` / `==` on Enum
    members of two different packages, which only holds because this package's enums equal same-named members of same-named foreign enums
    (environments/types.py: NamedEnum)."""
    import importlib
    from rl_x_b200.algorithms.algorithm_manager import get_algorithm_config, get_algorithm_general_properties, get_algorithm_model_class
    E = reference_enums()
    RefAction, RefObservation, RefInterface = E["ActionSpaceType"], E["ObservationSpaceType"], E["DataInterfaceType"]
    RefSimulation, RefFramework = E["SimulationType"], E["DeepLearningFrameworkType"]
    for algo, cls in (("ppo.b200", "PPO"), ("espo.b200", "ESPO"), ("sac.b200", "SAC"), ("fastsac.b200", "FastSAC"), ("ppo_lstm.b200", "PPO_LSTM")):
        importlib.import_module("rl_x_b200.algorithms." + algo)
        props = get_algorithm_general_properties(algo)
        assert get_algorithm_model_class(algo).__name__ == cls and get_algorithm_config(algo).name == algo

        class EnvProps:   # what a reference environment plugin states (e.g. custom_mujoco/ant/warp_torch/general_properties.py)
            action_space_type, observation_space_type = RefAction.CONTINUOUS, RefObservation.FLAT_VALUES
            data_interface_type, simulation_type = RefInterface.TORCH, RefSimulation.WARP

        # runner.py:86-91, verbatim conditions
        assert not (EnvProps.action_space_type not in props.action_space_types)
        assert not (EnvProps.observation_space_type not in props.observation_space_types)
        if algo not in ("sac.b200",):   # SAC takes NUMPY environments only, like the reference's sac.pytorch
            assert not (EnvProps.data_interface_type not in props.data_interface_types)
        # what the check must still reject: discrete actions and image observations (SURVEY 8 a20)
        assert RefAction.DISCRETE not in props.action_space_types and RefObservation.IMAGES not in props.observation_space_types
        # runner.py:100-101
        assert (RefFramework.TORCH == props.deep_learning_framework_type) and not (RefFramework.JAX == props.deep_learning_framework_type)
    # and this package's synthetic environment under the reference runner's simulation-type tests (runner.py:102-103)
    from rl_x_b200.environments.synthetic.box.general_properties import GeneralProperties as BoxProps
    assert not (RefSimulation.JAX_BASED == BoxProps.simulation_type)
    assert BoxProps.action_space_type in [RefAction.CONTINUOUS, RefAction.DISCRETE] and BoxProps.data_interface_type in [RefInterface.NUMPY, RefInterface.TORCH]
    # every member of the reference's enums exists here under the same name and value
    from rl_x_b200.algorithms import deep_learning_framework_type as fw
    from rl_x_b200.environments import types as env_types
    for name, ref_enum in E.items():
        ours = getattr(fw if name == "DeepLearningFrameworkType" else env_types, name)
        assert {m.name: m.value for m in ours} == {m.name: m.value for m in ref_enum}, name


def test_default_configs_are_ml_collections_config_dicts_where_available(monkeypatch):
    """The reference's runner passes every plugin's default config to ml_collections' config_flags.DEFINE_config_dict (runner.py:179-181), which
    accepts ml_collections.config_dict.ConfigDict instances only.  ml_collections is absent from this image, so a stand-in module proves the
    selection: with it importable, every get_config() of this package returns an instance of ITS ConfigDict; without it, the local class."""
    import sys
    import types
    from rl_x_b200 import config_dict as local

    class FakeMlConfigDict(dict):   # the part of the real class's surface the default_config modules use
        __getattr__, __setattr__ = dict.__getitem__, dict.__setitem__

    fake, fake_cd = types.ModuleType("ml_collections"), types.ModuleType("ml_collections.config_dict")
    fake_cd.ConfigDict, fake.config_dict = FakeMlConfigDict, fake_cd
    getters = []
    for algo in ("ppo", "espo", "sac", "fastsac", "ppo_lstm"):
        mod = __import__(f"rl_x_b200.algorithms.{algo}.b200.default_config", fromlist=["get_config"])
        getters.append((mod.get_config, f"{algo}.b200"))
    for env in ("box", "pendulum"):
        mod = __import__(f"rl_x_b200.environments.synthetic.{env}.default_config", fromlist=["get_config"])
        getters.append((mod.get_config, f"synthetic.{env}"))
    from rl_x_b200.runner.default_config import get_config as runner_config
    monkeypatch.setitem(sys.modules, "ml_collections", None)             # "not installed" (other tests of this session stage a stub of their own)
    monkeypatch.setitem(sys.modules, "ml_collections.config_dict", None)
    assert all(type(get(name)) is local.ConfigDict for get, name in getters)
    monkeypatch.setitem(sys.modules, "ml_collections", fake)
    monkeypatch.setitem(sys.modules, "ml_collections.config_dict", fake_cd)
    for get, name in getters:
        cfg = get(name)
        assert type(cfg) is FakeMlConfigDict and cfg.name == name, name
    assert type(runner_config("train")) is FakeMlConfigDict


def test_importing_a_plugin_package_registers_it_with_the_reference_too(tmp_path, monkeypatch):
    """No bridge package: the reference's runner does importlib.import_module(f"{package}.algorithms.{name}") for each implementation
    package and then asks rl_x's OWN managers for the plugin (runner.py:232-247, 86-96).  With rl_x importable (here: a stand-in whose
    register functions take the reference's parameters, tests/golden/reference_interfaces.json), importing rl_x_b200's plugin packages must
    therefore leave them in rl_x's registries as well as in this package's."""
    import importlib
    registry = reference_interfaces()["registry"]
    pkg = tmp_path / "rl_x"
    for kind in ("algorithms", "environments"):
        (pkg / kind).mkdir(parents=True)
        (pkg / kind / "__init__.py").write_text("")
        params = registry[f"register_{kind[:-1]}"]
        (pkg / kind / f"{kind[:-1]}_manager.py").write_text(
            f"_{kind} = {{}}\n\n\ndef register_{kind[:-1]}({', '.join(params)}):\n    _{kind}[name] = dict({', '.join(f'{p}={p}' for p in params)})\n")
    (pkg / "__init__.py").write_text("")
    monkeypatch.syspath_prepend(str(tmp_path))
    is_rl_x = lambda m: m == "rl_x" or m.startswith("rl_x.")
    for mod in [m for m in sys.modules if is_rl_x(m)]:
        monkeypatch.delitem(sys.modules, mod)
    try:
        from rl_x.algorithms import algorithm_manager as ref_algorithms
        from rl_x.environments import environment_manager as ref_environments
        for name in ("ppo.b200", "espo.b200", "sac.b200", "fastsac.b200", "ppo_lstm.b200"):
            importlib.reload(importlib.import_module(f"rl_x_b200.algorithms.{name}"))       # what runner.import_algorithm does
            entry = ref_algorithms._algorithms[name]
            assert entry["get_model_class"].__module__.startswith("rl_x_b200.algorithms." + name)
            assert entry["get_default_config"](name).name == name
            assert entry["general_properties"].deep_learning_framework_type.name == "TORCH"
        for name in ("synthetic.box", "synthetic.pendulum"):
            importlib.reload(importlib.import_module(f"rl_x_b200.environments.{name}"))
            entry = ref_environments._environments[name]
            assert callable(entry["create_train_and_eval_env"])
            assert entry["get_default_config"](name).name == name
            assert entry["general_properties"].action_space_type.name == "CONTINUOUS"
    finally:
        for mod in [m for m in sys.modules if is_rl_x(m)]:      # the stand-in leaves with this test
            del sys.modules[mod]


def test_default_configs_carry_every_reference_key_with_the_reference_value():
    """Every key of the reference's default_config.py of the five algorithms is present with the SAME default, except the one documented
    difference (bf16_mixed_precision_training: this build's default is the fp32 parity path); keys this build adds are not reference keys.
    The reference's defaults: tests/golden/reference_interfaces.json."""
    import importlib
    configs = reference_interfaces()["default_configs"]
    assert sorted(configs) == ["espo", "fastsac", "ppo", "ppo_lstm", "sac"]
    for algo, ref in configs.items():
        ours = importlib.import_module(f"rl_x_b200.algorithms.{algo}.b200.default_config").get_config("x")
        assert [k for k in ref if k not in ours] == [], algo
        different = {k: (ref[k], ours[k]) for k in ref if k != "name" and ref[k] != ours[k]}
        assert set(different) <= {"bf16_mixed_precision_training"}, (algo, different)


def test_model_classes_have_the_reference_classes_methods_and_signatures():
    """Duck typing is the boundary (SURVEY 8 b): every method of the reference's model class exists on this package's class with the same
    parameter names (`load` may be a classmethod: the runner calls it on the class either way, runner.py:334-337).  Read from the sources;
    the reference's side is tests/golden/reference_interfaces.json."""
    import ast

    def methods(path, cls):
        for node in ast.walk(ast.parse(open(path).read())):
            if isinstance(node, ast.ClassDef) and node.name == cls:
                return {f.name: [a.arg for a in f.args.args if a.arg != "cls"] for f in node.body if isinstance(f, ast.FunctionDef)}
        raise AssertionError(f"no class {cls} in {path}")

    pkg = os.path.join(ROOT, "rl_x_b200", "algorithms")
    reference = reference_interfaces()["methods"]
    cases = [("PPO", [f"{pkg}/ppo/b200/ppo.py"]), ("SAC", [f"{pkg}/sac/b200/sac.py"]), ("FastSAC", [f"{pkg}/fastsac/b200/fastsac.py"]),
             ("ESPO", [f"{pkg}/ppo/b200/ppo.py", f"{pkg}/espo/b200/espo.py"]), ("PPO_LSTM", [f"{pkg}/ppo_lstm/b200/ppo_lstm.py"])]
    assert sorted(reference) == sorted(c for c, _ in cases)
    for cls, our_paths in cases:
        ref, ours = reference[cls], {}
        for p, c in zip(our_paths, ["PPO", cls] if len(our_paths) == 2 else [cls]):   # ESPO inherits PPO here
            ours.update(methods(p, c))
        assert [m for m in ref if m not in ours] == [], cls
        assert {m: (ref[m], ours[m]) for m in ref if ref[m] != ours[m]} == {}, cls
