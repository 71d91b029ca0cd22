"""FastSAC update (rl_x_b200/csrc/fastsac.cu) checked WITHOUT a GPU: the source is compiled with g++ -DRLX_EMU (see csrc/dual_build.cuh) and
driven through the batches and normal draws of the executed reference run (tests/golden/fastsac_update.npz), side by side with
oracle/fastsac_oracle.py, which is itself pinned to that run.  After every critic / policy update the emulated library's parameters,
optimiser moments, target networks and metrics must match the oracle's; at the end they must match the reference's logged metrics."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import emu_build_cmd

from oracle import fastsac_oracle as FS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("obs_dim", "act_dim", "nr_atoms")]


class HP(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("gamma", "tau", "v_min", "v_max", "target_entropy", "log_std_min", "log_std_max", "weight_decay",
                                         "adam_beta1", "adam_beta2", "adam_eps", "max_grad_norm", "clipped_double_q")]


class Args(C.Structure):
    _fields_ = ([("dims", Dims), ("n", C.c_int64)] +
                [(k, C.c_void_p) for k in ("states", "next_states", "actions", "rewards", "dones", "truncations", "effective_n_steps", "noise",
                                           "action_scale", "policy_params", "policy_grads", "policy_m", "policy_v", "q_params", "q_grads", "q_m", "q_v",
                                           "q_target_params", "log_alpha", "alpha_state", "lr", "steps")] +
                [("hp", HP), ("metrics", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)])


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = tmp_path_factory.mktemp("fastsac_emu") / "libfastsac_emu.so"
    subprocess.run(emu_build_cmd(out, os.path.join(ROOT, "rl_x_b200", "csrc", "fastsac.cu")), check=True)
    lib = C.CDLL(str(out))
    lib.rlx_fastsac_workspace_bytes.restype = C.c_size_t
    lib.rlx_fastsac_workspace_bytes.argtypes = [C.POINTER(Dims), C.c_int64]
    return lib


def flat(net):
    return np.concatenate([t.detach().numpy().reshape(-1) for t in FS._leaves(net)]).astype(np.float32)


@pytest.mark.parametrize("tag", ["update", "update_clipped"])
def test_emulated_fastsac_updates_track_the_pinned_oracle(emu, tag):
    z = np.load(os.path.join(ROOT, "tests", "golden", f"fastsac_{tag}.npz"))
    N, obs, act, batch, n_steps, nopt, seed, ncu, npu, atoms, stride = (int(x) for x in z["meta"])
    gamma, tau, lr, lsmin, lsmax, tgt_ent, vmin, vmax, wd, b1, b2, alpha0, low, high, scale, clipped, max_gn = (float(x) for x in z["meta_f"])
    torch.set_num_threads(1)
    pol, q1, q2 = FS.reference_init(obs, act, atoms, seed)
    center = (low + high) / 2
    action_scale = torch.full((act,), max(abs(low - center), abs(high - center)) / scale)
    L = FS.Learner(pol, q1, q2, action_scale, lr, wd, (b1, b2), gamma, tau, vmin, vmax, atoms, tgt_ent, alpha0, lsmin, lsmax,
                   clipped_double_q=bool(clipped), max_grad_norm=max_gn)
    nrm = FS.Normalizer(obs)

    d = Dims(obs, act, atoms)
    poff, qoff = (C.c_int64 * 17)(), (C.c_int64 * 15)()
    assert emu.rlx_fastsac_param_layout(C.byref(d), poff, qoff) == 0
    P, Q = flat(L.pol), np.concatenate([flat(L.q1), flat(L.q2)])
    assert poff[16] == P.size and 2 * qoff[14] == Q.size
    QT = Q.copy()
    gP, mP, vP = np.zeros_like(P), np.zeros_like(P), np.zeros_like(P)
    gQ, mQ, vQ = np.zeros_like(Q), np.zeros_like(Q), np.zeros_like(Q)
    la, astate = np.array([np.log(alpha0)], np.float32), np.zeros(3, np.float32)
    lr_a, steps = np.array([lr], np.float32), np.zeros(3, np.int64)
    sc = action_scale.numpy().astype(np.float32)
    nbytes = emu.rlx_fastsac_workspace_bytes(C.byref(d), batch)
    ws = np.full(nbytes // 4, np.nan, np.float32)   # exact size (ASan build) and NaN-filled (a read of workspace nothing wrote in this call poisons the outputs)
    hp = HP(gamma, tau, vmin, vmax, tgt_ent, lsmin, lsmax, wd, b1, b2, 1e-8, max_gn, clipped)
    nmean, nvar, nstd, ncount = np.zeros(obs, np.float32), np.ones(obs, np.float32), np.ones(obs, np.float32), np.zeros(1, np.int64)
    emu.rlx_fastsac_normalize_f32.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                              C.c_void_p, C.c_void_p, C.c_void_p]

    def call(fn, s, ns, a_, r, dn, tr, eff, noise, metrics):
        arrs = [np.ascontiguousarray(t.numpy() if torch.is_tensor(t) else t, dtype=np.float32) if t is not None else None
                for t in (s, ns, a_, r, dn, tr, eff, noise)]
        a = Args()
        a.dims, a.n = d, batch
        for name, arr in zip(("states", "next_states", "actions", "rewards", "dones", "truncations", "effective_n_steps", "noise"), arrs):
            setattr(a, name, arr.ctypes.data if arr is not None else None)
        a.action_scale = sc.ctypes.data
        a.policy_params, a.policy_grads, a.policy_m, a.policy_v = P.ctypes.data, gP.ctypes.data, mP.ctypes.data, vP.ctypes.data
        a.q_params, a.q_grads, a.q_m, a.q_v, a.q_target_params = Q.ctypes.data, gQ.ctypes.data, mQ.ctypes.data, vQ.ctypes.data, QT.ctypes.data
        a.log_alpha, a.alpha_state, a.lr, a.steps = la.ctypes.data, astate.ctypes.data, lr_a.ctypes.data, steps.ctypes.data
        a.hp, a.metrics, a.workspace, a.workspace_bytes = hp, metrics.ctypes.data, ws.ctypes.data, nbytes
        state = dict(P=P, gP=gP, mP=mP, vP=vP, Q=Q, gQ=gQ, mQ=mQ, vQ=vQ, QT=QT, log_alpha=la, alpha_state=astate, steps=steps, metrics=metrics)
        before = {k_: v_.copy() for k_, v_ in state.items()} if race_check[0] else None
        rc = fn(C.byref(a), None)
        assert rc == 0, rc
        if race_check[0]:
            # Race check (csrc/dual_build.cuh): the same update from the same state with the emulated threads of every launch run in
            # DESCENDING order must produce the same bits; a thread reading another thread's output of the same launch would not.
            first = {k_: v_.copy() for k_, v_ in state.items()}
            for k_, v_ in state.items():
                v_[...] = before[k_]
            ws[:] = np.nan
            emu.rlx_emu_set_thread_order(1)
            try:
                assert fn(C.byref(a), None) == 0
            finally:
                emu.rlx_emu_set_thread_order(0)
            for k_, v_ in state.items():
                assert np.array_equal(v_, first[k_]), f"{fn.__name__}: {k_} depends on the thread order"

    def close(ours, ref, what, rtol=3e-4, atol=3e-6):
        np.testing.assert_allclose(ours, ref, rtol=rtol, atol=atol, err_msg=what)

    def close_params(ours, ref, what):
        """parameters after AdamW steps: Adam divides by sqrt(v), which turns fp32 rounding of a near-zero gradient entry into a difference
        of a fraction of lr in that entry (more entries are in that regime when clip_grad_norm_ scales the gradient down) — bound single
        entries by one full step (lr) and the tensor as a whole by its relative norm."""
        np.testing.assert_allclose(ours, ref, rtol=3e-4, atol=lr, err_msg=what)
        rel = float(np.linalg.norm(ours - ref) / np.linalg.norm(ref))
        assert rel <= 2e-5, (what, rel)

    logged = {}
    race_check = [True]   # on for the first optimisation step (it doubles the work)
    for u in range(nopt):
        race_check[0] = (u == 0)
        b = {k: z[f"step{u}/{k}"] for k in ["states", "next_states", "actions", "rewards", "dones", "truncations", "effective_n_steps"]}
        total = b["states"].shape[0]
        wsn = np.zeros(4 * obs * (total // 256 + 2), np.float32)
        s_emu, ns_emu = np.zeros_like(b["states"]), np.zeros_like(b["next_states"])
        for src, dst in ((b["states"], s_emu), (b["next_states"], ns_emu)):
            src = np.ascontiguousarray(src)
            assert emu.rlx_fastsac_normalize_f32(src.ctypes.data, total, obs, nmean.ctypes.data, nvar.ctypes.data, nstd.ctypes.data, ncount.ctypes.data, 1,
                                                 1e-8, dst.ctypes.data, wsn.ctypes.data, None) == 0
        s = nrm.normalize(torch.from_numpy(b["states"]), update=True)
        ns = nrm.normalize(torch.from_numpy(b["next_states"]), update=True)
        close(s_emu, s.numpy(), "normalised states", 1e-5, 1e-5)
        close(ns_emu, ns.numpy(), "normalised next states", 1e-5, 1e-5)
        close(nmean, nrm.mean.numpy().reshape(-1), "running mean", 1e-5, 1e-6)
        close(nvar, nrm.var.numpy().reshape(-1), "running var", 1e-5, 1e-6)
        assert int(ncount[0]) == nrm.count
        view = lambda t: torch.as_tensor(t).view(npu, ncu, batch, *t.shape[1:])
        s, ns = view(s), view(ns)
        a_, r, dn, tr, eff = (view(b[k]) for k in ["actions", "rewards", "dones", "truncations", "effective_n_steps"])
        normals = torch.from_numpy(z[f"step{u}/normals"])
        k, step_metrics = 0, []
        for i in range(npu):
            for j in range(ncu):
                m = L.critic_and_entropy_step(s[i, j], ns[i, j], a_[i, j], r[i, j], dn[i, j], tr[i, j], eff[i, j], normals[k])
                mc = np.zeros(8, np.float32)
                call(emu.rlx_fastsac_critic_update_f32, s[i, j], ns[i, j], a_[i, j], r[i, j], dn[i, j], tr[i, j], eff[i, j], normals[k], mc)
                k += 1
                for idx, name in enumerate(["loss/q_loss", "loss/entropy_loss", "q/q_min", "q/q_max", "entropy/entropy", "gradients/critic_grad_norm",
                                            "gradients/entropy_grad_norm"]):
                    assert abs(float(mc[idx]) - m[name]) <= 3e-4 * max(1.0, abs(m[name])), (u, i, j, name, mc[idx], m[name])
                close_params(Q, np.concatenate([flat(L.q1), flat(L.q2)]), f"q params after critic update {u}.{i}.{j}")
                close_params(QT, np.concatenate([flat(L.q1t), flat(L.q2t)]), "target params")
                close(la, L.log_alpha.detach().numpy(), "log_alpha", 1e-5, 1e-7)
            mo = L.policy_step(s[i, -1], normals[k])
            mp = np.zeros(8, np.float32)
            call(emu.rlx_fastsac_policy_update_f32, s[i, -1], None, None, None, None, None, None, normals[k], mp)
            k += 1
            for idx, name in enumerate(["loss/policy_loss", "entropy/alpha", "gradients/policy_grad_norm"]):
                assert abs(float(mp[idx]) - mo[name]) <= 3e-4 * max(1.0, abs(mo[name])), (u, i, name, mp[idx], mo[name])
            close_params(P, flat(L.pol), f"policy params after policy update {u}.{i}")
            m = dict(m)
            m.update(mo)
            step_metrics.append({**m, **{"emu/" + nm: float(v) for nm, v in zip(["loss/q_loss", "loss/policy_loss"], [mc[0], mp[0]])}})
        for name in ("emu/loss/q_loss", "emu/loss/policy_loss"):
            logged.setdefault(name, []).append(float(np.mean([sm[name] for sm in step_metrics])))
    # the emulated library's own losses against what the executed reference logged
    np.testing.assert_allclose(logged["emu/loss/q_loss"], z["metric/loss/q_loss"], rtol=3e-4)
    np.testing.assert_allclose(logged["emu/loss/policy_loss"], z["metric/loss/policy_loss"], rtol=3e-4, atol=2e-5)  # a difference of O(1) terms
    assert list(steps) == [nopt * npu * ncu, nopt * npu * ncu, nopt * npu]


@pytest.mark.parametrize("tag", ["update", "update_clipped"])
def test_plugin_class_reproduces_the_reference_run_under_emulation(tmp_path, tag):
    """The whole plugin (rl_x_b200/algorithms/fastsac/b200: FastSAC class + n-step ReplayBuffer) on CPU: the two modules are loaded with
    their device hooks rewritten (device -> cpu, stream -> NULL, library -> host emulation builds of fastsac.cu and replay_nstep.cu; the
    shipped modules raise without CUDA).  With the golden run's seed and environment the torch generator is consumed in the reference's
    order (module init, acting noise, torch.randint sampling, update noise), so the run must reproduce the metrics the executed
    reference logged at every step."""
    import types
    from rl_x_b200 import _native as nt
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.fastsac.b200.default_config import get_config
    from rl_x_b200.environments.types import ActionSpaceType, ObservationSpaceType, DataInterfaceType
    emus = []
    for name in ("fastsac", "replay_nstep"):
        out = tmp_path / f"lib{name}_emu.so"
        subprocess.run(emu_build_cmd(out, os.path.join(ROOT, "rl_x_b200", "csrc", f"{name}.cu")), check=True)
        emus.append(C.CDLL(str(out)))
    real = nt.load()

    class Lib:
        def __getattr__(self, name):
            for e in emus:
                try:
                    f = getattr(e, name)
                except AttributeError:
                    continue
                f.argtypes, f.restype = getattr(real, name).argtypes, getattr(real, name).restype
                return f
            raise AttributeError(name)

    lib = Lib()

    def load_patched(relpath, modname, drop_import=None, extra=None):
        src = open(os.path.join(ROOT, *relpath)).read()
        if drop_import:
            assert drop_import in src
            src = src.replace(drop_import, "")
        for old, new in [('torch.device("cuda", torch.cuda.current_device())', 'torch.device("cpu")'),
                         ('if a.device != "gpu" or not torch.cuda.is_available():', 'if False:'), ('if not torch.cuda.is_available():', 'if False:'),
                         ("return C.c_void_p(torch.cuda.current_stream().cuda_stream)", "return None"),
                         ("C.c_void_p(torch.cuda.current_stream().cuda_stream)", "None"), ("self.lib = nt.load()", "self.lib = LIB")]:
            src = src.replace(old, new)
        mod = types.ModuleType(modname)
        mod.LIB = lib
        mod.__dict__.update(extra or {})
        exec(compile(src, modname, "exec"), mod.__dict__)
        return mod

    rb = load_patched(("rl_x_b200", "algorithms", "fastsac", "b200", "replay_buffer.py"), "fastsac_replay_emulated")
    fs = load_patched(("rl_x_b200", "algorithms", "fastsac", "b200", "fastsac.py"), "fastsac_emulated",
                      drop_import="from rl_x_b200.algorithms.fastsac.b200.replay_buffer import ReplayBuffer", extra={"ReplayBuffer": rb.ReplayBuffer})
    z = np.load(os.path.join(ROOT, "tests", "golden", f"fastsac_{tag}.npz"))
    N, obs, act, batch, n_steps, nopt, seed, ncu, npu, atoms, stride = (int(x) for x in z["meta"])
    clipped, max_gn = bool(z["meta_f"][15]), float(z["meta_f"][16])

    class Sp:
        def __init__(self, shape, **kw):
            self.shape = shape
            self.__dict__.update(kw)

    class Props:
        observation_space_type, action_space_type, data_interface_type = ObservationSpaceType.FLAT_VALUES, ActionSpaceType.CONTINUOUS, DataInterfaceType.TORCH

    class Env:  # the environment of tests/golden/make_golden_fastsac.py
        general_properties, horizon = Props, 5

        def __init__(self):
            self.g = torch.Generator().manual_seed(seed + 100)
            self.single_observation_space = Sp((obs,))
            low, high = np.full(act, -1.5, np.float32), np.full(act, 0.5, np.float32)
            self.single_action_space = Sp((act,), low=low, high=high, center=(low + high) / 2, scale=np.full(act, 0.8, np.float32))
            self.t = 0

        def reset(self):
            return torch.randn(N, obs, generator=self.g) * 2 + 1, {}

        def step(self, action):
            self.t += 1
            return (torch.randn(N, obs, generator=self.g) * 2 + 1, torch.randn(N, generator=self.g), torch.rand(N, generator=self.g) < 0.2,
                    torch.full((N,), self.t % 4 == 0), {})

        def get_logging_info_dict(self, info):
            return {}

        def close(self):
            pass

    a = get_config("fastsac.b200")
    a.batch_size, a.buffer_size_per_env, a.learning_starts, a.total_timesteps, a.n_steps = batch, 8, 3, N * 9, n_steps
    a.nr_critic_updates_per_policy_update, a.nr_policy_updates_per_step, a.logging_frequency, a.save_frequency = ncu, npu, N, -1
    a.learning_rate, a.target_entropy, a.clipped_double_q_learning, a.max_grad_norm = 1e-3, -float(act), clipped, max_gn
    cfg = ConfigDict(algorithm=a, environment=ConfigDict(seed=seed, nr_envs=N),
                     runner=ConfigDict(save_model=False, track_console=False, track_tb=False, track_wandb=False, load_model=""))
    torch.set_num_threads(1)
    env = Env()
    model = fs.FastSAC(cfg, env, env, str(tmp_path), None)
    logged = []
    model.log = lambda name, value, step: logged.append((name, float(value)))
    model.train()
    checked = 0
    for key in z.files:
        if not key.startswith("metric/"):
            continue
        name = key[len("metric/"):]
        ours = [v for nme, v in logged if nme == name]
        np.testing.assert_allclose(ours, z[key], rtol=5e-4, atol=5e-6, err_msg=name)
        checked += 1
    assert checked >= 15


def test_plugin_checkpoint_has_the_reference_layout(tmp_path):
    """FastSAC.save() writes the reference's file (fastsac.py:463-478): the state dicts load with strict=True into torch modules shaped like
    the reference's Policy / QNetwork and its three AdamW optimisers accept the optimiser states; FastSAC.load() restores the flat
    buffers exactly.  (Run on CPU with the same source rewrites as above.)"""
    import types
    from rl_x_b200 import _native as nt
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.fastsac.b200.default_config import get_config
    from rl_x_b200.environments.types import ActionSpaceType, ObservationSpaceType, DataInterfaceType
    src = open(os.path.join(ROOT, "rl_x_b200", "algorithms", "fastsac", "b200", "fastsac.py")).read()
    src = src.replace("from rl_x_b200.algorithms.fastsac.b200.replay_buffer import ReplayBuffer", "ReplayBuffer = None")
    for old, new in [('torch.device("cuda", torch.cuda.current_device())', 'torch.device("cpu")'),
                     ('if a.device != "gpu" or not torch.cuda.is_available():', 'if False:'), ("self.lib = nt.load()", "self.lib = nt.load()")]:
        assert old in src
        src = src.replace(old, new)
    mod = types.ModuleType("fastsac_ckpt")
    exec(compile(src, "fastsac_ckpt", "exec"), mod.__dict__)   # only the layout query of the real library is used here (host function)
    obs, act, atoms = 9, 4, 21

    class Sp:
        def __init__(self, shape, **kw):
            self.shape = shape
            self.__dict__.update(kw)

    class Props:
        observation_space_type, action_space_type, data_interface_type = ObservationSpaceType.FLAT_VALUES, ActionSpaceType.CONTINUOUS, DataInterfaceType.TORCH

    class Env:
        general_properties, horizon = Props, 3
        single_observation_space = Sp((obs,))
        single_action_space = Sp((act,), low=np.full(act, -1.0, np.float32), high=np.full(act, 1.0, np.float32), center=np.zeros(act, np.float32),
                                 scale=np.ones(act, np.float32))

    a = get_config("fastsac.b200")
    a.nr_atoms = atoms
    cfg = ConfigDict(algorithm=a, environment=ConfigDict(seed=8, nr_envs=4),
                     runner=ConfigDict(save_model=True, track_console=False, track_tb=False, track_wandb=False, load_model=""))
    model = mod.FastSAC(cfg, Env(), Env(), str(tmp_path / "run"), None)
    g = torch.Generator().manual_seed(0)
    for t in (model.policy_m, model.policy_v, model.q_m, model.q_v, model.q_target_params, model.alpha_state, model.norm_mean):
        t.copy_(torch.rand(t.shape, generator=g))
    model.steps.copy_(torch.tensor([12, 12, 3]))
    model.norm_count.fill_(77)
    model.save()
    path = tmp_path / "run" / "models" / "latest.model"
    ck = torch.load(path, weights_only=False)
    assert set(ck) == {"config_algorithm", "policy_state_dict", "q1_state_dict", "q2_state_dict", "q1_target_state_dict", "q2_target_state_dict", "log_alpha",
                       "policy_optimizer_state_dict", "q_optimizer_state_dict", "entropy_optimizer_state_dict", "observation_normalizer_state_dict"}

    def torso(inp, widths):
        layers, last = [], inp
        for w in widths:
            layers += [torch.nn.Linear(last, w), torch.nn.LayerNorm(w), torch.nn.SiLU()]
            last = w
        return layers

    class Policy(torch.nn.Module):       # module structure of rl_x/algorithms/fastsac/pytorch/policy.py:36-48
        def __init__(self):
            super().__init__()
            self.torso = torch.nn.Sequential(*torso(obs, (512, 256, 128)))
            self.mean, self.log_std = torch.nn.Linear(128, act), torch.nn.Linear(128, act)

    class QNetwork(torch.nn.Module):     # q_network.py:24-35
        def __init__(self):
            super().__init__()
            self.critic = torch.nn.Sequential(*torso(obs + act, (768, 384, 192)), torch.nn.Linear(192, atoms))

    pol, q1, q2 = Policy(), QNetwork(), QNetwork()
    pol.load_state_dict(ck["policy_state_dict"], strict=True)
    q1.load_state_dict(ck["q1_state_dict"], strict=True)
    q2.load_state_dict(ck["q2_state_dict"], strict=True)
    QNetwork().load_state_dict(ck["q1_target_state_dict"], strict=True)
    torch.optim.AdamW(pol.parameters(), lr=1e-3).load_state_dict(ck["policy_optimizer_state_dict"])
    torch.optim.AdamW(list(q1.parameters()) + list(q2.parameters()), lr=1e-3).load_state_dict(ck["q_optimizer_state_dict"])
    torch.optim.AdamW([torch.nn.Parameter(torch.zeros(1))], lr=1e-3).load_state_dict(ck["entropy_optimizer_state_dict"])
    # the module built from the checkpoint computes what the oracle computes from the plugin's flat parameters
    x = torch.randn(5, obs)
    with torch.no_grad():
        latent = pol.torso(x)
        opol = {"torso": [(l.weight, l.bias) for l in pol.torso if not isinstance(l, torch.nn.SiLU)], "mean": (pol.mean.weight, pol.mean.bias),
                "log_std": (pol.log_std.weight, pol.log_std.bias)}
        assert torch.allclose(latent, FS.torso_forward(opol, x), atol=1e-6)
        assert torch.equal(torch.cat([t.reshape(-1) for t in FS._leaves(opol)]), model.policy_params)
    # round trip
    cfg.runner.load_model = str(path)
    cfg.runner.save_model = False
    again = mod.FastSAC.load(cfg, Env(), Env(), str(tmp_path / "run2"), None, [])
    for name in ("policy_params", "q_params", "q_target_params", "log_alpha", "policy_m", "policy_v", "q_m", "q_v", "alpha_state", "norm_mean", "norm_var",
                 "norm_std", "norm_count", "steps"):
        a_, b_ = getattr(model, name), getattr(again, name)
        if name == "alpha_state":
            a_, b_ = a_[1:], b_[1:]   # element 0 is the transient gradient
        assert torch.equal(a_, b_), name


def test_checkpoints_move_between_the_plugin_and_the_reference_classes(tmp_path):
    """f2 for FastSAC against the reference's checkpoint layout (tests/golden/reference_interfaces.json, captured from the executed
    reference's FastSAC: file keys, module keys / shapes / dtypes, AdamW numbering and settings): (1) a `latest.model` laid out as the
    reference's FastSAC.save() writes it (fastsac.py:463-478), after AdamW steps on every parameter, is read by the plugin's load() and every
    tensor - parameters, targets, both AdamW moments, step counts, log_alpha, normaliser statistics - lands on the segment its name says;
    (2) the file the plugin's save() writes goes through the reference's load() sequence (strict load_state_dict + optimizer
    load_state_dict, :481-500) and arrives tensor for tensor.  The plugin runs on CPU with the source rewrites of the tests above."""
    import types
    from conftest import load_like_the_reference, reference_interfaces, reference_module, reference_optimizers
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.fastsac.b200.default_config import get_config
    from rl_x_b200.environments.types import ActionSpaceType, ObservationSpaceType, DataInterfaceType
    interfaces = reference_interfaces()
    layout = interfaces["checkpoints"]["fastsac"]
    obs, act, atoms, N = (layout["meta"][k] for k in ("obs", "act", "nr_atoms", "nr_envs"))

    class Sp:
        def __init__(self, shape, **kw):
            self.shape = shape
            self.__dict__.update(kw)

    class Props:
        observation_space_type, action_space_type, data_interface_type = ObservationSpaceType.FLAT_VALUES, ActionSpaceType.CONTINUOUS, DataInterfaceType.TORCH

    class Env:
        general_properties, horizon = Props, 3
        single_observation_space = Sp((obs,))
        single_action_space = Sp((act,), low=np.full(act, -1.0, np.float32), high=np.full(act, 1.0, np.float32), center=np.zeros(act, np.float32),
                                 scale=np.ones(act, np.float32))

    # ---- a file laid out as the reference's save() writes it, with optimiser state on every parameter
    g = torch.Generator().manual_seed(0)
    ref = {name: reference_module(m) for name, m in layout["modules"].items()}
    ent = torch.nn.Module()
    ent.log_alpha = torch.nn.Parameter(torch.full(layout["log_alpha"]["shape"], -0.3))
    with torch.no_grad():
        for name, m in ref.items():
            for p in m.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    opts = reference_optimizers(layout, ref, ent)
    for opt in opts.values():
        for _ in range(3):
            for group in opt.param_groups:
                for p in group["params"]:
                    p.grad = torch.randn(p.shape, generator=g) * 0.1
            opt.step()
    with torch.no_grad():
        for tgt, src in (("q1_target", "q1"), ("q2_target", "q2")):
            for p, q in zip(ref[tgt].parameters(), ref[src].parameters()):
                p.copy_(q + torch.randn(p.shape, generator=g) * 0.01)
        nrm = ref["observation_normalizer"]
        nrm.running_mean.copy_(torch.randn(nrm.running_mean.shape, generator=g))                       # non-trivial running statistics
        nrm.running_var.copy_(torch.rand(nrm.running_var.shape, generator=g) + 0.5)
        nrm.running_std_dev.copy_(nrm.running_var.sqrt())
        nrm.count.fill_(32)
    ra = ConfigDict(dict(interfaces["default_configs"]["fastsac"]))
    ra.name, ra.device, ra.bf16_mixed_precision_training, ra.compile_mode, ra.nr_atoms = "fastsac.pytorch", "cpu", False, "default", atoms
    ref_file = str(tmp_path / "latest.model")
    torch.save({"config_algorithm": ra, **{f"{name}_state_dict": m.state_dict() for name, m in ref.items()}, "log_alpha": ent.log_alpha,
                **{f"{name}_state_dict": opt.state_dict() for name, opt in opts.items()}}, ref_file)
    assert set(torch.load(ref_file, weights_only=False)) == set(layout["keys"])

    # ---- the plugin class on CPU (device hooks rewritten; only host functions of the library are used)
    src = open(os.path.join(ROOT, "rl_x_b200", "algorithms", "fastsac", "b200", "fastsac.py")).read()
    src = src.replace("from rl_x_b200.algorithms.fastsac.b200.replay_buffer import ReplayBuffer", "ReplayBuffer = None")
    for old, new in [('torch.device("cuda", torch.cuda.current_device())', 'torch.device("cpu")'),
                     ('if a.device != "gpu" or not torch.cuda.is_available():', 'if False:')]:
        assert old in src
        src = src.replace(old, new)
    mod = types.ModuleType("fastsac_interop")
    exec(compile(src, "fastsac_interop", "exec"), mod.__dict__)
    a = get_config("fastsac.b200")
    cfg = ConfigDict(algorithm=a, environment=ConfigDict(seed=8, nr_envs=N),
                     runner=ConfigDict(save_model=True, track_console=False, track_tb=False, track_wandb=False, load_model=ref_file))
    ours = mod.FastSAC.load(cfg, Env(), Env(), str(tmp_path / "our_run"), None, [])
    assert int(ours.dims.nr_atoms) == atoms     # taken from the file's config_algorithm
    nq = ours.q_offsets[-1]

    def check(module, opt, flat, m, v, net, step_index):
        named, nm, nv = ours._named(flat, net), ours._named(m, net) if m is not None else None, ours._named(v, net) if v is not None else None
        for name, p in module.named_parameters():
            assert torch.equal(named[name], p.detach()), (net, name)
            if opt is not None:
                st = opt.state[p]
                assert torch.equal(nm[name], st["exp_avg"]) and torch.equal(nv[name], st["exp_avg_sq"]), (net, name)
                assert int(ours.steps[step_index]) == int(float(st["step"])) == 3

    def check_all(ref, opts):
        check(ref["policy"], opts["policy_optimizer"], ours.policy_params, ours.policy_m, ours.policy_v, "policy", 2)
        check(ref["q1"], opts["q_optimizer"], ours.q_params[:nq], ours.q_m[:nq], ours.q_v[:nq], "q", 0)
        check(ref["q2"], opts["q_optimizer"], ours.q_params[nq:], ours.q_m[nq:], ours.q_v[nq:], "q", 0)
        check(ref["q1_target"], None, ours.q_target_params[:nq], None, None, "q", 0)
        check(ref["q2_target"], None, ours.q_target_params[nq:], None, None, "q", 0)

    check_all(ref, opts)
    assert torch.equal(ours.log_alpha.reshape(-1), ent.log_alpha.detach().reshape(-1))
    st = opts["entropy_optimizer"].state[ent.log_alpha]
    assert float(ours.alpha_state[1]) == float(st["exp_avg"]) and float(ours.alpha_state[2]) == float(st["exp_avg_sq"]) and int(ours.steps[1]) == 3
    nsd = ref["observation_normalizer"].state_dict()
    assert torch.equal(ours.norm_mean.reshape(-1), nsd["running_mean"].reshape(-1)) and torch.equal(ours.norm_var.reshape(-1), nsd["running_var"].reshape(-1))
    assert int(ours.norm_count[0]) == int(nsd["count"])

    # ---- and back: what the plugin writes, through the reference's load() sequence
    for t in (ours.policy_params, ours.q_params, ours.q_target_params, ours.policy_m, ours.q_m):
        t.add_(torch.randn(t.shape, generator=g) * 0.01)          # not the tensors that came in
    ours.save()
    back, back_opts, back_ent = load_like_the_reference(os.path.join(str(tmp_path / "our_run"), "models", "latest.model"), layout)
    check_all(back, back_opts)
    assert torch.equal(ours.log_alpha.reshape(-1), back_ent.log_alpha.detach().reshape(-1))
    bsd = back["observation_normalizer"].state_dict()
    assert torch.equal(ours.norm_mean.reshape(-1), bsd["running_mean"].reshape(-1)) and int(ours.norm_count[0]) == int(bsd["count"])
