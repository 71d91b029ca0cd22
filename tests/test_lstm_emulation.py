"""PPO+LSTM update path (rl_x_b200/csrc/lstm.cu) checked WITHOUT a GPU: the same source is compiled with g++ -DRLX_EMU (kernel launches
become loops over threads, GEMMs an interpreter of the GemmP contract) and its outputs are compared with oracle/ppo_lstm_oracle.py's
autograd.  This validates indexing, strides, the carry-reset rule, BPTT and every hand-derived gradient; what it cannot validate is
anything specific to the device (the real SIMT GEMM kernels are covered by the PPO parity tests).  The emulation library is built
into a temporary directory and is never loaded by the product."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import emu_build_cmd

from oracle import ppo_lstm_oracle as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("obs_dim", "act_dim", "hidden", "enc_dim", "lstm_dim", "options")]


OPT_FILM, OPT_SHARED = 1, 2   # RLX_LSTM_OPT_* (include/rlx_b200.h)


class Args(C.Structure):
    _fields_ = ([("dims", Dims), ("T", C.c_int64), ("n_env", C.c_int64)] +
                [(n, C.c_void_p) for n in ("states", "actions", "log_probs", "advantages", "returns", "dones", "init_c", "init_h", "adv_stats",
                                           "policy_params", "critic_params", "policy_grads", "critic_grads")] +
                [(n, C.c_float) for n in ("clip_range", "entropy_coef", "critic_coef", "reserved")] +
                [("metrics", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)])


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = tmp_path_factory.mktemp("lstm_emu") / "liblstm_emu.so"
    src = os.path.join(ROOT, "rl_x_b200", "csrc", "lstm.cu")
    subprocess.run(emu_build_cmd(out, src), check=True)
    lib = C.CDLL(str(out))
    lib.rlx_lstm_minibatch_workspace_bytes.restype = C.c_size_t
    lib.rlx_lstm_minibatch_workspace_bytes.argtypes = [C.POINTER(Dims), C.c_int64, C.c_int64]
    return lib


POLICY_SEGS = ["lstm_obs_encoder_dense.kernel", "lstm_obs_encoder_dense.bias", "lstm_obs_encoder_ln.scale", "lstm_obs_encoder_ln.bias",
               "obs_encoder_dense.kernel", "obs_encoder_dense.bias", "obs_encoder_ln.scale", "obs_encoder_ln.bias", "Wi", "Wh", "bh",
               "lstm_ln.scale", "lstm_ln.bias", "torso_dense1.kernel", "torso_dense1.bias", "torso_dense2.kernel", "torso_dense2.bias",
               "mean_head.kernel", "mean_head.bias", "policy_logstd", "Wf", "bf"]
CRITIC_SEGS = ["Dense_0.kernel", "Dense_0.bias", "Dense_1.kernel", "Dense_1.bias", "Dense_2.kernel", "Dense_2.bias"]


def _get(tree, dotted):
    for k in dotted.split("."):
        tree = tree[k]
    return tree


def flatten_policy(pol):
    """oracle tree -> the flat layout of include/rlx_b200.h (gate blocks i|f|g|o side by side)."""
    parts = []
    for name in POLICY_SEGS:
        if name == "Wi":
            parts.append(torch.cat([pol["lstm"]["i" + k]["kernel"] for k in L.GATES], dim=1))
        elif name == "Wh":
            parts.append(torch.cat([pol["lstm"]["h" + k]["kernel"] for k in L.GATES], dim=1))
        elif name == "bh":
            parts.append(torch.cat([pol["lstm"]["h" + k]["bias"] for k in L.GATES]))
        elif name in ("Wf", "bf"):   # FiLM blocks gamma | beta side by side; empty for "concat"
            leaf = "kernel" if name == "Wf" else "bias"
            parts.append(torch.cat([pol["lstm_film_gamma"][leaf], pol["lstm_film_beta"][leaf]], dim=-1) if "lstm_film_gamma" in pol else torch.zeros(0))
        elif name.startswith("obs_encoder") and "obs_encoder_dense" not in pol:
            parts.append(torch.zeros(0))   # shared encoder: no obs_encoder segments
        else:
            parts.append(_get(pol, name))
    return [p.detach().reshape(-1) for p in parts]


def flatten_critic(cri):
    return [_get(cri, n).detach().reshape(-1) for n in CRITIC_SEGS]


def _np(t):
    return np.ascontiguousarray(t.detach().numpy(), dtype=np.float32)


@pytest.mark.parametrize("options", [0, OPT_FILM, OPT_SHARED, OPT_FILM | OPT_SHARED])
@pytest.mark.parametrize("T,n,obs,act,hid,enc,lstm", [
    (7, 5, 6, 2, 12, 8, 4), (5, 3, 9, 3, 16, 12, 8), (33, 40, 5, 2, 8, 8, 4),
    # BASELINE config 5's minibatch (128 steps x 256 envs, reference widths): ~2 min per option set with RLX_EMU_CXXFLAGS=-O2, so on request
    # only.  Last run (round 2, all four option sets): worst entry at 0.3 % of the GPU test's tolerance.
    pytest.param(128, 256, 64, 8, 256, 128, 64, marks=pytest.mark.skipif(os.environ.get("RLX_SLOW_TESTS") != "1", reason="slow: RLX_SLOW_TESTS=1"))])
def test_emulated_lstm_fwdbwd_matches_oracle_autograd(emu, T, n, obs, act, hid, enc, lstm, options):
    torch.manual_seed(T * 100 + n)
    pol, cri = L.init_params(obs, act, hidden=hid, enc=enc, lstm=lstm, std_dev=0.8, seed=T, share_encoder=bool(options & OPT_SHARED),
                             combine="film" if options & OPT_FILM else "concat")
    # non-trivial LayerNorm parameters and biases so that every gradient path is exercised
    for tree in (pol, cri):
        for name, v in L.tree_leaves(tree):
            if name.endswith("bias") or name.endswith("scale"):
                v.add_(0.1 * torch.randn_like(v))
    states, actions = torch.randn(T, n, obs), torch.randn(T, n, act)
    log_probs = torch.randn(T, n) * 0.1 - 2.5
    adv, ret = torch.randn(T, n), torch.randn(T, n)
    dones = (torch.rand(T, n) < 0.2).float()
    init = (torch.randn(n, lstm) * 0.5, torch.randn(n, lstm) * 0.5)
    clip, ent, cc = 0.2, 0.01, 0.5

    learner = L.Learner(pol, cri, clip_range=clip, entropy_coef=ent, critic_coef=cc)
    mb = dict(states=states, actions=actions, log_probs=log_probs, returns=ret, advantages=adv, dones=dones, init_carry=init)
    gp_ref, gc_ref, metrics_ref = learner.grads(mb)
    # oracle gradients are per leaf of its (sorted) tree; bring them into the flat layout
    gp_tree = dict(zip([nm for nm, _ in L.tree_leaves(learner.pol)], gp_ref))
    gc_tree = dict(zip([nm for nm, _ in L.tree_leaves(learner.cri)], gc_ref))

    def grad_seg(name):
        if name == "Wi":
            return torch.cat([gp_tree[f"lstm.i{k}.kernel"] for k in L.GATES], dim=1)
        if name == "Wh":
            return torch.cat([gp_tree[f"lstm.h{k}.kernel"] for k in L.GATES], dim=1)
        if name == "bh":
            return torch.cat([gp_tree[f"lstm.h{k}.bias"] for k in L.GATES])
        if name in ("Wf", "bf"):
            leaf = "kernel" if name == "Wf" else "bias"
            return (torch.cat([gp_tree[f"lstm_film_gamma.{leaf}"], gp_tree[f"lstm_film_beta.{leaf}"]], dim=-1) if options & OPT_FILM
                    else torch.zeros(0))
        return gp_tree.get(name, torch.zeros(0))   # obs_encoder.* are absent with a shared encoder

    d = Dims(obs, act, hid, enc, lstm, options)
    P = np.concatenate([_np(x) for x in flatten_policy(pol)])
    Cc = np.concatenate([_np(x) for x in flatten_critic(cri)])
    poff, coff = (C.c_int64 * (len(POLICY_SEGS) + 1))(), (C.c_int64 * 7)()
    assert emu.rlx_lstm_param_layout(C.byref(d), poff, coff) == 0
    assert poff[len(POLICY_SEGS)] == P.size and coff[6] == Cc.size
    gP, gC = np.full_like(P, np.nan), np.full_like(Cc, np.nan)
    stats = np.array([float(adv.mean()), float(adv.std(unbiased=False))], dtype=np.float32)
    metrics = np.zeros(8, np.float32)
    nbytes = emu.rlx_lstm_minibatch_workspace_bytes(C.byref(d), T, n)
    # exact size: an AddressSanitizer run (conftest.emu_build_cmd) sees any overrun; NaN-filled: a kernel that reads workspace before
    # something wrote it in THIS call (stale data from the previous minibatch on the device) poisons the outputs
    ws = np.full(nbytes // 4, np.nan, np.float32)
    arrs = dict(states=_np(states), actions=_np(actions), log_probs=_np(log_probs), advantages=_np(adv), returns=_np(ret), dones=_np(dones),
                init_c=_np(init[0]), init_h=_np(init[1]))
    a = Args()
    a.dims, a.T, a.n_env = d, T, n
    for k, v in arrs.items():
        setattr(a, k, v.ctypes.data)
    a.adv_stats, a.policy_params, a.critic_params = stats.ctypes.data, P.ctypes.data, Cc.ctypes.data
    a.policy_grads, a.critic_grads, a.metrics = gP.ctypes.data, gC.ctypes.data, metrics.ctypes.data
    a.clip_range, a.entropy_coef, a.critic_coef = clip, ent, cc
    a.workspace, a.workspace_bytes = ws.ctypes.data, nbytes
    assert emu.rlx_lstm_ppo_minibatch_fwdbwd_f32(C.byref(a), None) == 0
    assert np.isfinite(gP).all() and np.isfinite(gC).all()

    scale = max(float(np.abs(np.concatenate([_np(grad_seg(nm)).reshape(-1) for nm in POLICY_SEGS])).max()), 1e-6)
    for i, name in enumerate(POLICY_SEGS):
        ours, ref = gP[poff[i]:poff[i + 1]], _np(grad_seg(name)).reshape(-1)
        np.testing.assert_allclose(ours, ref, rtol=2e-4, atol=2e-6 * max(scale, 1.0), err_msg=name)
    for i, name in enumerate(CRITIC_SEGS):
        ours, ref = gC[coff[i]:coff[i + 1]], _np(gc_tree[name]).reshape(-1)
        np.testing.assert_allclose(ours, ref, rtol=2e-4, atol=2e-6, err_msg=name)
    for j, key in enumerate(["loss/policy_gradient_loss", "loss/critic_loss", "loss/entropy_loss", "policy_ratio/approx_kl", "policy_ratio/clip_fraction"]):
        assert abs(float(metrics[j]) - metrics_ref[key]) <= 2e-5 * max(1.0, abs(metrics_ref[key])), (key, metrics[j], metrics_ref[key])
    assert metrics[7] == T * n
    # Race check: the same call with the emulated threads of every launch run in DESCENDING order must give the same bits.  A thread that
    # reads what another thread of the same launch writes (a data race on the device) would make the result depend on the order.
    gP2, gC2, metrics2 = np.full_like(P, np.nan), np.full_like(Cc, np.nan), np.zeros(8, np.float32)
    ws[:] = np.nan
    a.policy_grads, a.critic_grads, a.metrics = gP2.ctypes.data, gC2.ctypes.data, metrics2.ctypes.data
    emu.rlx_emu_set_thread_order(1)
    try:
        assert emu.rlx_lstm_ppo_minibatch_fwdbwd_f32(C.byref(a), None) == 0
    finally:
        emu.rlx_emu_set_thread_order(0)
    assert np.array_equal(gP, gP2) and np.array_equal(gC, gC2) and np.array_equal(metrics, metrics2)
    # The recurrence as ONE block-cooperative launch per direction (rlx_set_lstm_persistent: recurrent kernel and the envs' hidden state in
    # shared memory, a barrier per step; emulated with one OS thread per CUDA thread): same arithmetic in the same order, so the same bits.
    gP3, gC3, metrics3 = np.full_like(P, np.nan), np.full_like(Cc, np.nan), np.zeros(8, np.float32)
    ws[:] = np.nan
    a.policy_grads, a.critic_grads, a.metrics = gP3.ctypes.data, gC3.ctypes.data, metrics3.ctypes.data
    emu.rlx_lstm_persistent_launch_count.restype = C.c_uint64
    launches = emu.rlx_lstm_persistent_launch_count()
    assert emu.rlx_set_lstm_persistent(1) == 1
    try:
        assert emu.rlx_lstm_ppo_minibatch_fwdbwd_f32(C.byref(a), None) == 0
    finally:
        emu.rlx_set_lstm_persistent(0)
    assert emu.rlx_lstm_persistent_launch_count() == launches + 2   # forward and backward
    assert np.array_equal(gP, gP3) and np.array_equal(gC, gC3) and np.array_equal(metrics, metrics3)


def test_emulated_optax_step_and_env_gather(emu):
    n = 5000
    g0 = torch.Generator().manual_seed(3)
    p = torch.randn(n, generator=g0)
    ref_p = [p.clone().requires_grad_(True)]
    opt = L.OptaxAdam(ref_p, 1e-2, max_norm=0.5)
    ours = _np(p).copy()
    mu, nu = np.zeros(n, np.float32), np.zeros(n, np.float32)
    lr, step, norm, ws = np.array([1e-2], np.float32), np.zeros(1, np.int64), np.zeros(1, np.float32), np.zeros(64, np.float32)
    emu.rlx_optax_clip_adam_f32.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_void_p, C.c_void_p] + [C.c_float] * 4 + [C.c_void_p] * 3
    for s in range(4):
        g = torch.randn(n, generator=g0) * (0.001 if s == 2 else 1.0)   # step 2 stays below the clip threshold
        ref_norm = opt.step([g.clone()])
        gg = _np(g)
        assert emu.rlx_optax_clip_adam_f32(ours.ctypes.data, gg.ctypes.data, mu.ctypes.data, nu.ctypes.data, n, lr.ctypes.data, step.ctypes.data,
                                           0.5, 0.9, 0.999, 1e-8, norm.ctypes.data, ws.ctypes.data, None) == 0
        assert abs(float(norm[0]) - ref_norm) <= 1e-5 * ref_norm
        np.testing.assert_allclose(ours, _np(ref_p[0]), rtol=1e-5, atol=1e-6)
    assert int(step[0]) == 4
    T, N, w = 3, 7, 4
    src = np.arange(T * N * w, dtype=np.float32).reshape(T, N, w)
    idx = np.array([5, 0, 5, 2], dtype=np.int64)
    out = np.zeros((T, 4, w), np.float32)
    emu.rlx_gather_env_columns_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
    assert emu.rlx_gather_env_columns_f32(src.ctypes.data, idx.ctypes.data, T, N, 4, w, out.ctypes.data, None) == 0
    assert np.array_equal(out, src[:, idx])


class StepArgs(C.Structure):
    _fields_ = ([("dims", Dims), ("n", C.c_int64)] +
                [(k, C.c_void_p) for k in ("obs", "c", "h", "noise", "policy_params", "critic_params", "act_low", "act_high")] +
                [("clip_rescale", C.c_int32), ("reserved", C.c_int32)] +
                [(k, C.c_void_p) for k in ("action", "env_action", "logp", "value", "workspace")] + [("workspace_bytes", C.c_size_t)])


@pytest.mark.parametrize("options", [0, OPT_FILM, OPT_SHARED, OPT_FILM | OPT_SHARED])
def test_emulated_rollout_step_matches_oracle(emu, options):
    """rlx_lstm_step_f32 == get_action_and_value (ppo_lstm.py:107-118) over a few consecutive steps with the carry threaded through and
    reset by rlx_lstm_mask_carry_f32; plus the critic-only forward and the population-std helper."""
    obs_d, act, hid, enc, lstm, n = 7, 3, 16, 12, 8, 6
    torch.manual_seed(4)
    pol, cri = L.init_params(obs_d, act, hidden=hid, enc=enc, lstm=lstm, std_dev=0.6, seed=9, share_encoder=bool(options & OPT_SHARED),
                             combine="film" if options & OPT_FILM else "concat")
    for tree in (pol, cri):
        for name, v in L.tree_leaves(tree):
            if name.endswith("bias") or name.endswith("scale"):
                v.add_(0.1 * torch.randn_like(v))
    d = Dims(obs_d, act, hid, enc, lstm, options)
    P = np.concatenate([_np(x) for x in flatten_policy(pol)])
    Cc = np.concatenate([_np(x) for x in flatten_critic(cri)])
    low, high = np.full(act, -2.0, np.float32), np.full(act, 0.5, np.float32)
    nbytes = emu.rlx_lstm_minibatch_workspace_bytes(C.byref(d), 1, n)
    # exact size: an AddressSanitizer run (conftest.emu_build_cmd) sees any overrun; NaN-filled: a kernel that reads workspace before
    # something wrote it in THIS call (stale data from the previous minibatch on the device) poisons the outputs
    ws = np.full(nbytes // 4, np.nan, np.float32)
    c, h = np.zeros((n, lstm), np.float32), np.zeros((n, lstm), np.float32)
    carry = (torch.zeros(n, lstm), torch.zeros(n, lstm))
    emu.rlx_lstm_mask_carry_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
    for step in range(4):
        obs, noise = torch.randn(n, obs_d), torch.randn(n, act)
        with torch.no_grad():
            proc, action, value, logp, carry = L.get_action_and_value(pol, cri, obs, carry, noise, torch.from_numpy(low), torch.from_numpy(high))
        o, nz = _np(obs), _np(noise)
        out_a, out_e, out_lp, out_v = (np.zeros((n, act), np.float32), np.zeros((n, act), np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32))
        a = StepArgs()
        a.dims, a.n = d, n
        a.obs, a.c, a.h, a.noise = o.ctypes.data, c.ctypes.data, h.ctypes.data, nz.ctypes.data
        a.policy_params, a.critic_params, a.act_low, a.act_high = P.ctypes.data, Cc.ctypes.data, low.ctypes.data, high.ctypes.data
        a.clip_rescale = 1
        a.action, a.env_action, a.logp, a.value = out_a.ctypes.data, out_e.ctypes.data, out_lp.ctypes.data, out_v.ctypes.data
        a.workspace, a.workspace_bytes = ws.ctypes.data, nbytes
        c_in, h_in = c.copy(), h.copy()
        assert emu.rlx_lstm_step_f32(C.byref(a), None) == 0
        # race check (see the fwd/bwd test): descending thread order from the same inputs, same bits (the carry is updated in place)
        first = [x.copy() for x in (out_a, out_e, out_lp, out_v, c, h)]
        c[:], h[:] = c_in, h_in
        emu.rlx_emu_set_thread_order(1)
        try:
            assert emu.rlx_lstm_step_f32(C.byref(a), None) == 0
        finally:
            emu.rlx_emu_set_thread_order(0)
        assert all(np.array_equal(x, y) for x, y in zip(first, (out_a, out_e, out_lp, out_v, c, h)))
        np.testing.assert_allclose(out_a, _np(action), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(out_e, _np(proc), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(out_lp, _np(logp), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(out_v, _np(value), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(c, _np(carry[0]), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(h, _np(carry[1]), rtol=1e-5, atol=1e-6)
        done = (torch.rand(n) < 0.4).float()
        carry = (carry[0] * (1 - done)[:, None], carry[1] * (1 - done)[:, None])   # ppo_lstm.py:283
        dn = _np(done)
        assert emu.rlx_lstm_mask_carry_f32(c.ctypes.data, h.ctypes.data, dn.ctypes.data, n, lstm, None) == 0
        np.testing.assert_allclose(c, _np(carry[0]), rtol=1e-5, atol=1e-6)
    # deterministic mode (noise == NULL): action = mean
    a.noise, a.logp, a.value, a.critic_params = None, None, None, None
    obs = torch.randn(n, obs_d)
    o = _np(obs)
    a.obs = o.ctypes.data
    with torch.no_grad():
        mean, _, _ = L.apply_one_step(pol, obs, carry)
    assert emu.rlx_lstm_step_f32(C.byref(a), None) == 0
    np.testing.assert_allclose(out_a, _np(mean), rtol=1e-5, atol=1e-6)
    # critic-only forward over many rows, population std
    rows = 300
    x = torch.randn(rows, obs_d)
    xv, outv = _np(x), np.zeros(rows, np.float32)
    nb = emu.rlx_lstm_minibatch_workspace_bytes(C.byref(d), 1, rows)
    ws2 = np.full(nb // 4, np.nan, np.float32)
    emu.rlx_lstm_critic_forward_f32.argtypes = [C.POINTER(Dims), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    assert emu.rlx_lstm_critic_forward_f32(C.byref(d), Cc.ctypes.data, xv.ctypes.data, rows, outv.ctypes.data, ws2.ctypes.data, nb, None) == 0
    with torch.no_grad():
        np.testing.assert_allclose(outv, _np(L.critic_value(cri, x).reshape(-1)), rtol=1e-5, atol=1e-6)
    y = (torch.randn(1000) * 2 + 3)
    yv, st2, wsp = _np(y), np.zeros(2, np.float32), np.zeros(1000 + 2 * 4 + 8, np.float32)
    emu.rlx_mean_popstd_f32.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    assert emu.rlx_mean_popstd_f32(yv.ctypes.data, 1000, st2.ctypes.data, wsp.ctypes.data, None) == 0
    assert abs(st2[0] - float(y.mean())) < 1e-5 and abs(st2[1] - float(y.std(unbiased=False))) < 1e-5


def test_plugin_class_runs_under_emulation(emu, tmp_path):
    """Host logic of rl_x_b200/algorithms/ppo_lstm/b200/ppo_lstm.py (rollout bookkeeping, env-column minibatches, schedules, logging,
    evaluation) exercised on CPU: the module source is loaded with its three device hooks rewritten (device -> cpu, stream -> NULL,
    library -> the emulation build + an oracle GAE), which the shipped module never does — it raises without CUDA."""
    import types
    from oracle import ppo_oracle as O
    from rl_x_b200 import _native as nt
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.ppo_lstm.b200.default_config import get_config
    from rl_x_b200.environments.types import ActionSpaceType, ObservationSpaceType, DataInterfaceType
    real = nt.load()

    class Lib:
        """The emulation build behind the plugin's `self.lib`, plus a stand-in for CUDA-graph capture: while `capturing`, calls are
        recorded instead of executed (as stream capture does), and FakeGraph.replay() issues the recorded calls."""
        capturing, recorded, launches = False, None, 0

        def __getattr__(self, name):
            if name == "rlx_launch_count":
                return lambda: Lib.launches
            if name == "rlx_add_launch_count":
                def add(n):
                    Lib.launches += int(n)
                return add
            if name == "rlx_gae_f32":
                def gae(r, term, v, nv, last, T, N, gamma, lam, adv, ret, stream):
                    t = lambda ptr: torch.from_numpy(np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_float)), shape=(T, N)))
                    a, rr = O.gae(t(r), t(term), t(v), t(nv), gamma, lam)
                    t(adv).copy_(a)
                    t(ret).copy_(rr)
                    return 0
                return gae
            f = getattr(emu, name)
            f.argtypes, f.restype = getattr(real, name).argtypes, getattr(real, name).restype

            def call(*args):
                Lib.launches += 1
                if Lib.capturing:
                    Lib.recorded.append((f, args))
                    return 0
                return f(*args)
            return call

    class FakeGraph:
        def replay(self):
            for f, args in self.calls:
                assert f(*args) == 0

    class FakeGraphContext:
        def __init__(self, g, capture_error_mode="global"):
            self.g = g

        def __enter__(self):
            Lib.capturing, Lib.recorded = True, []

        def __exit__(self, *exc):
            Lib.capturing, self.g.calls = False, Lib.recorded

    class TorchWithFakeGraphs:
        """`torch` as the plugin module sees it on this CPU-only box: everything real except torch.cuda.CUDAGraph / torch.cuda.graph."""
        class cuda:
            CUDAGraph, graph = FakeGraph, FakeGraphContext

        def __getattr__(self, name):
            return getattr(torch, name)

    path = os.path.join(ROOT, "rl_x_b200", "algorithms", "ppo_lstm", "b200", "ppo_lstm.py")
    src = open(path).read()
    for old, new in [('torch.device("cuda", torch.cuda.current_device())', 'torch.device("cpu")'),
                     ('if a.device != "gpu" or not torch.cuda.is_available():', 'if False:'),
                     ("return C.c_void_p(torch.cuda.current_stream().cuda_stream)", "return None"), ("self.lib = nt.load()", "self.lib = LIB")]:
        assert old in src
        src = src.replace(old, new)
    mod = types.ModuleType("ppo_lstm_emulated")
    mod.LIB = Lib()
    exec(compile(src, "ppo_lstm_emulated", "exec"), mod.__dict__)
    mod.torch = TorchWithFakeGraphs()
    N, T, obs, act = 8, 16, 12, 3

    class Sp:
        def __init__(self, shape, low=None, high=None):
            self.shape, self.low, self.high = shape, low, high

    results = {}
    for iface, combine, share, graph in (("TORCH", "concat", False, False), ("NUMPY", "concat", False, False), ("TORCH", "film", False, False),
                                         ("TORCH", "concat", True, False), ("NUMPY", "film", True, False), ("TORCH", "concat", False, True),
                                         ("NUMPY", "film", True, True)):
        class P:
            observation_space_type, action_space_type = ObservationSpaceType.FLAT_VALUES, ActionSpaceType.CONTINUOUS
            data_interface_type = getattr(DataInterfaceType, iface)

        class Env:
            general_properties = P
            single_observation_space = Sp((obs,))
            single_action_space = Sp((act,), np.full(act, -1.0, np.float32), np.full(act, 1.0, np.float32))

            def __init__(self):
                self.g = torch.Generator().manual_seed(3)

            def _o(self, x):
                return x if iface == "TORCH" else x.numpy()

            def reset(self):
                return self._o(torch.randn(N, obs, generator=self.g)), {}

            def step(self, action):
                assert tuple(action.shape) == (N, act)
                self.last = torch.randn(N, obs, generator=self.g)
                return (self._o(self.last), self._o(torch.randn(N, generator=self.g)), self._o(torch.rand(N, generator=self.g) < 0.1),
                        self._o(torch.zeros(N, dtype=torch.bool)), {})

            def get_logging_info_dict(self, info):
                return {}

            def get_final_observation_at_index(self, info, i):
                return self.last[i].numpy()

            def get_final_info_value_at_index(self, info, key, i):
                return 1.0

            def close(self):
                pass

        a = get_config("ppo_lstm.b200")
        a.nr_steps, a.minibatch_size, a.nr_epochs, a.total_timesteps = T, 4 * T, 2, 3 * N * T
        a.nr_hidden_units, a.obs_encoding_dim, a.lstm_hidden_dim, a.learning_rate, a.anneal_learning_rate = 32, 16, 8, 1e-3, True
        a.evaluation_frequency, a.evaluation_episodes = N * T, 2
        a.lstm_obs_combine_method, a.share_lstm_obs_encoder, a.use_cuda_graph = combine, share, graph
        cfg = ConfigDict(algorithm=a, environment=ConfigDict(seed=5, nr_envs=N),
                         runner=ConfigDict(save_model=False, track_console=False, track_tb=False, track_wandb=False, load_model=""))
        env = Env()
        model = mod.PPO_LSTM(cfg, env, env, str(tmp_path), None)
        before = model.policy_params.clone()
        logged = []
        model.log = lambda name, value, step: logged.append((name, float(value)))
        model.train()
        assert all(np.isfinite(v) for nme, v in logged if not nme.startswith("time/"))
        names = {nme for nme, _ in logged}
        for nme in ["loss/policy_gradient_loss", "loss/critic_loss", "loss/entropy_loss", "policy_ratio/approx_kl", "policy_ratio/clip_fraction",
                    "gradients/policy_grad_norm", "gradients/critic_grad_norm", "lr/learning_rate", "v_value/explained_variance", "policy/std_dev",
                    "steps/nr_env_steps", "steps/nr_updates", "steps/nr_episodes", "eval/episode_return"]:
            assert nme in names, nme
        # linear schedule (ppo_lstm.py:78-81): the rate of the last optimiser step of each of the 3 iterations
        np.testing.assert_allclose([v for nme, v in logged if nme == "lr/learning_rate"], [1e-3, 1e-3 * 2 / 3, 1e-3 / 3], rtol=1e-6)
        assert [v for nme, v in logged if nme == "steps/nr_updates"] == [4.0, 8.0, 12.0]
        assert float((model.policy_params - before).abs().max()) > 1e-4
        results[(iface, combine, share, graph)] = ([(nme, v) for nme, v in logged if nme.split("/")[0] in ("loss", "gradients", "policy_ratio", "lr", "steps")],
                                                   model.policy_params.clone(), model.critic_params.clone())
        assert (model._graph is not None) == graph and (not graph or len(model._graph.calls) == 12)   # 8 gathers, stats, fwd+bwd, 2 x Adam
        pol_named, _ = model.named_parameters()
        assert pol_named["Wf"].numel() == (8 * 2 * 16 if combine == "film" else 0) and pol_named["We2"].numel() == (0 if share else obs * 16)
    # the two data interfaces drive the same computation
    assert results[("TORCH", "concat", False, False)][0] == results[("NUMPY", "concat", False, False)][0]
    # the captured-and-replayed update (use_cuda_graph) issues the same calls on the same buffers as the eager loop: identical numbers
    for key in (("TORCH", "concat", False), ("NUMPY", "film", True)):
        eager, replayed = results[key + (False,)], results[key + (True,)]
        assert eager[0] == replayed[0] and torch.equal(eager[1], replayed[1]) and torch.equal(eager[2], replayed[2])


def test_emulated_nstep_replay_matches_reference_golden(tmp_path):
    """rl_x_b200/csrc/replay_nstep.cu (FastSAC n-step sampling) compiled for the host and run on the golden rings of the executed reference:
    gathers, flags and effective lengths bit-exact; the n-step reward equals the oracle's step-ordered float32 sum bit for bit and the
    reference's torch.sum to one rounding."""
    from conftest import GOLDEN_DIR
    from oracle import fastsac_replay_oracle as F
    out = tmp_path / "libnstep_emu.so"
    subprocess.run(emu_build_cmd(out, os.path.join(ROOT, "rl_x_b200", "csrc", "replay_nstep.cu")), check=True)
    lib = C.CDLL(str(out))
    lib.rlx_replay_sample_nstep_f32.argtypes = ([C.c_void_p, C.c_void_p] + [C.c_int64] * 5 + [C.c_int32, C.c_void_p, C.c_int64, C.c_int64] +
                                                [C.c_void_p] * 15)
    z = np.load(os.path.join(GOLDEN_DIR, "fastsac_replay.npz"))
    names = ["states", "next_states", "actions", "rewards", "dones", "truncations", "effective_n_steps"]
    for tag in [str(c) for c in z["cases"]]:
        cap, nr_envs, obs, act, n_steps, size, pos, ns = (int(x) for x in z[f"{tag}/meta"])
        ring = {k: np.ascontiguousarray(z[f"{tag}/ring/{k}"]) for k in names[:6]}
        idx_t, idx_e = np.ascontiguousarray(z[f"{tag}/idx_t"]), np.ascontiguousarray(z[f"{tag}/idx_e"])
        disc = np.ascontiguousarray(z[f"{tag}/discounts"])
        n = len(idx_t)
        outs = [np.zeros((n, obs), np.float32), np.zeros((n, obs), np.float32), np.zeros((n, act), np.float32)] + [np.zeros(n, np.float32) for _ in range(4)]
        scratch = np.zeros(n, np.int64)
        rc = lib.rlx_replay_sample_nstep_f32(idx_t.ctypes.data, idx_e.ctypes.data, n, cap, nr_envs, obs, act, n_steps, disc.ctypes.data, size, pos,
                                             *[ring[k].ctypes.data for k in names[:6]], *[o.ctypes.data for o in outs], scratch.ctypes.data, None)
        assert rc == 0
        # race check (csrc/dual_build.cuh): descending thread order, same bits
        outs2 = [np.zeros_like(o) for o in outs]
        lib.rlx_emu_set_thread_order(1)
        try:
            assert lib.rlx_replay_sample_nstep_f32(idx_t.ctypes.data, idx_e.ctypes.data, n, cap, nr_envs, obs, act, n_steps, disc.ctypes.data, size, pos,
                                                   *[ring[k].ctypes.data for k in names[:6]], *[o.ctypes.data for o in outs2],
                                                   np.zeros(n, np.int64).ctypes.data, None) == 0
        finally:
            lib.rlx_emu_set_thread_order(0)
        assert all(np.array_equal(x, y) for x, y in zip(outs, outs2)), tag
        want = F.sample(ring, idx_t, idx_e, n_steps, disc, size, pos)
        for name, got, w in zip(names, outs, want):
            assert np.array_equal(got, w), f"{tag}/{name} vs oracle"
            ref = z[f"{tag}/out/{name}"]
            if name == "rewards":
                np.testing.assert_allclose(got, ref, rtol=3e-7, atol=3e-7, err_msg=f"{tag}/{name}")
            else:
                assert np.array_equal(got, ref), f"{tag}/{name} vs reference"


def test_persistent_recurrence_is_race_free_under_tsan(tmp_path):
    """The one-launch-per-direction recurrence kernels (lstm_seq_fwd_kernel / lstm_seq_bwd_kernel: shared memory + one barrier per step) under
    ThreadSanitizer: the emulation runs each CUDA thread of a block as an OS thread and __syncthreads as a real barrier, so a barrier missing
    between a shared-memory write and another thread's read is a reported data race (dropping the per-step barrier of the forward kernel
    was tried: TSan flags it at the shared-memory read).  The driver also demands bit-identity with the per-step path."""
    exe = tmp_path / "emu_tsan_lstm"
    build = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=thread", "-pthread", "-DRLX_EMU", "-x", "c++",
                            os.path.join(ROOT, "rl_x_b200", "csrc", "lstm.cu"), os.path.join(ROOT, "tests", "emu_tsan_lstm.cpp"), "-o", str(exe)],
                           capture_output=True, text=True)
    if build.returncode != 0 and "tsan" in (build.stderr or "").lower():
        pytest.skip("this toolchain has no ThreadSanitizer runtime")
    assert build.returncode == 0, build.stderr[-2000:]
    run = subprocess.run([str(exe)], env=dict(os.environ, TSAN_OPTIONS="exitcode=66"), capture_output=True, text=True, timeout=600)
    assert run.returncode == 0 and run.stdout.strip().endswith("ok"), (run.returncode, (run.stdout + run.stderr)[-3000:])
