import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box: pytest -m gpu)")


def pytest_sessionfinish(session, exitstatus):
    """RLX_AUX_ENGINE_REPORT=<file>: leave "<tensor GEMMs> <persistent recurrence launches>" of this process - the FastSAC / PPO+LSTM GEMMs
    that ran on the tcgen05 engine and the one-launch-per-direction LSTM recurrences (the subprocess runs of run_suite_with_switches below read
    it back: a green suite that never took the path it was asked to take proves nothing)."""
    path = os.environ.get("RLX_AUX_ENGINE_REPORT")
    if path:
        try:
            from rl_x_b200 import _native as nt
            lib = nt.load()
            text = f"{int(lib.rlx_aux_tc_gemm_count())} {int(lib.rlx_lstm_persistent_launch_count())}"
        except Exception as exc:  # noqa: BLE001 - the report is best effort, the exit status carries the verdict
            text = f"unavailable: {exc}"
        with open(path, "w") as fh:
            fh.write(text)


def run_suite_with_switches(test_file, tmp_path, tensor_engine=False, persistent=False, timeout=900):
    """Run the GPU parity tests of `test_file` again in a SUBPROCESS with the opt-in paths on: RLX_AUX_GEMM_ENGINE=1 (dense layers on the tcgen05
    3xTF32 engine where it covers the product) and / or RLX_LSTM_PERSISTENT=1 (LSTM recurrence as one block-cooperative launch per direction).
    A subprocess because a kernel that traps or faults takes the CUDA context with it: here that costs one test, not the rest of the
    session.  Returns (returncode, output tail, tensor GEMM count, persistent launch count); the counts are -1 when no report came back."""
    import subprocess
    report = os.path.join(str(tmp_path), "aux_paths.txt")
    env = dict(os.environ, RLX_AUX_GEMM_ENGINE="1" if tensor_engine else "0", RLX_LSTM_PERSISTENT="1" if persistent else "0", RLX_AUX_ENGINE_REPORT=report)
    proc = subprocess.run([sys.executable, "-m", "pytest", test_file, "-x", "-q", "-m", "gpu", "-k", "not subprocess", "-p", "no:cacheprovider"],
                          env=env, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    counts = open(report).read().split() if os.path.exists(report) else []
    tc, pers = (int(counts[0]), int(counts[1])) if len(counts) == 2 and all(x.isdigit() for x in counts) else (-1, -1)
    return proc.returncode, (proc.stdout + proc.stderr)[-3000:], tc, pers


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class Golden:
    """Golden vectors captured from the executed reference (tests/golden/make_golden_ppo.py)."""

    def __init__(self, tag):
        self.z = np.load(os.path.join(GOLDEN_DIR, f"ppo_{tag}.npz"))
        m = self.z["meta"]
        self.N, self.T, self.obs, self.act, self.hidden, self.mb, self.epochs, self.iterations, self.seed = (int(x) for x in m)
        f = self.z["meta_f"]
        (self.gamma, self.gae_lambda, self.clip_range, self.entropy_coef, self.critic_coef, self.max_grad_norm, self.lr,
         self.std_dev, self.act_low, self.act_high) = (float(x) for x in f[:10])
        self.anneal = bool(f[10])
        self.B = self.N * self.T

    def __getitem__(self, k):
        return self.z[k]

    def params(self, prefix):
        """(policy dict, critic dict) of numpy arrays under e.g. 'init' or 'iter0'."""
        pol = {k.split("/", 2)[2]: self.z[k] for k in self.z.files if k.startswith(f"{prefix}/policy/")}
        cri = {k.split("/", 2)[2]: self.z[k] for k in self.z.files if k.startswith(f"{prefix}/critic/")}
        return pol, cri

    def perms(self, iteration):
        return [self.z[f"perm/{iteration * self.epochs + e}"] for e in range(self.epochs)]

    def lr_at(self, iteration):
        # LinearLR(start 1 -> end 0 over total_iters = iterations), stepped once per iteration (ppo.py:87-88,302-304)
        if not self.anneal:
            return self.lr
        return self.lr * (1.0 - iteration / self.iterations)


class GoldenEspo(Golden):
    """Golden vectors of the executed ESPO reference (tests/golden/make_golden_espo.py); same layout as the PPO files except that
    `epochs` is max_epochs, the third float is max_ratio_delta and the index arrays are `choice/<k>`."""

    def __init__(self, tag):
        self.z = np.load(os.path.join(GOLDEN_DIR, f"espo_{tag}.npz"))
        m = self.z["meta"]
        self.N, self.T, self.obs, self.act, self.hidden, self.mb, self.max_epochs, self.iterations, self.seed = (int(x) for x in m)
        self.epochs = self.max_epochs
        f = self.z["meta_f"]
        (self.gamma, self.gae_lambda, self.max_ratio_delta, self.entropy_coef, self.critic_coef, self.max_grad_norm, self.lr,
         self.std_dev, self.act_low, self.act_high) = (float(x) for x in f[:10])
        self.clip_range = float("inf")
        self.anneal = bool(f[10])
        self.B = self.N * self.T


@pytest.fixture(scope="session")
def golden_espo():
    return GoldenEspo("small")


@pytest.fixture(scope="session", params=["small", "humanoid"])
def golden(request):
    return Golden(request.param)


@pytest.fixture(scope="session")
def golden_small():
    return Golden("small")


@pytest.fixture(scope="session")
def golden_humanoid():
    return Golden("humanoid")


def emu_build_cmd(out, src):
    """g++ command of the host-emulation builds (tests/test_*_emulation.py).  RLX_EMU_CXXFLAGS adds flags, e.g. an AddressSanitizer pass
    over the emulated kernels:  RLX_EMU_CXXFLAGS="-g -fsanitize=address" LD_PRELOAD=$(gcc -print-file-name=libasan.so)
    ASAN_OPTIONS=detect_leaks=0 python -m pytest tests/test_lstm_emulation.py tests/test_fastsac_emulation.py"""
    import os
    import shlex
    return (["g++", "-x", "c++", "-std=c++17", "-O1", "-fPIC", "-shared", "-pthread", "-DRLX_EMU"] + shlex.split(os.environ.get("RLX_EMU_CXXFLAGS", ""))
            + ["-o", str(out), str(src)])


def reference_interfaces():
    """tests/golden/reference_interfaces.json, captured from the executed reference (tests/golden/make_golden_reference_interfaces.py)."""
    import json
    with open(os.path.join(GOLDEN_DIR, "reference_interfaces.json")) as fh:
        return json.load(fh)


class _Node(torch.nn.Module):
    pass


def reference_module(layout):
    """A module with the reference module's parameters and buffers: same names (torch.compile's "_orig_mod." prefix removed), shapes, dtypes
    and named_parameters() order, so that strict load_state_dict accepts exactly what the reference module accepts."""
    root = _Node()
    params = {n for n, _ in layout["parameters"]}
    for name, shape, dtype in layout["state_dict"]:
        *path, leaf = name.split(".")
        node = root
        for part in path:
            if not hasattr(node, part):
                node.add_module(part, _Node())
            node = getattr(node, part)
        if name in params:
            node.register_parameter(leaf, torch.nn.Parameter(torch.zeros(shape, dtype=getattr(torch, dtype))))
        else:
            node.register_buffer(leaf, torch.zeros(shape, dtype=getattr(torch, dtype)))
    assert [[n, list(p.shape)] for n, p in root.named_parameters()] == layout["parameters"]
    assert [[n, list(t.shape), str(t.dtype).replace("torch.", "")] for n, t in root.state_dict().items()] == layout["state_dict"]
    return root


def reference_optimizer(layout, modules):
    """The reference's optimizer over the stand-in modules: same class, same param_group settings, parameters in the reference's numbering.
    `modules`: prefix -> module, the prefixes the captured parameter names carry ("" for an optimizer over one module)."""
    named = {(f"{prefix}.{n}" if prefix else n): p for prefix, m in modules.items() for n, p in m.named_parameters()}
    groups = [dict(g["settings"], params=[named[n] for n in g["param_names"]]) for g in layout["param_groups"]]
    for g in groups:
        g["betas"] = tuple(g["betas"])
    return getattr(torch.optim, layout["class"])(groups)


def reference_optimizers(ref, mods, ent):
    """The three optimizers of the reference's SAC / FastSAC over stand-in modules (policy; q1 then q2; the entropy module's log_alpha)."""
    return {"policy_optimizer": reference_optimizer(ref["optimizers"]["policy_optimizer"], {"": mods["policy"]}),
            "q_optimizer": reference_optimizer(ref["optimizers"]["q_optimizer"], {"q1": mods["q1"], "q2": mods["q2"]}),
            "entropy_optimizer": reference_optimizer(ref["optimizers"]["entropy_optimizer"], {"": ent})}


def load_like_the_reference(path, ref):
    """What the reference's SAC / FastSAC load() does with a checkpoint file (sac.py:400-416, fastsac.py:483-500), on stand-in modules and
    optimizers laid out as the reference's (`ref`: one entry of reference_interfaces.json "checkpoints").  Returns the modules, the
    optimizers and the entropy module whose log_alpha the file replaced."""
    ck = torch.load(path, weights_only=False)
    assert hasattr(ck["config_algorithm"], "items")
    mods = {name: reference_module(layout) for name, layout in ref["modules"].items()}
    ent = _Node()
    ent.log_alpha = torch.nn.Parameter(torch.zeros(ref["log_alpha"]["shape"]))
    opts = reference_optimizers(ref, mods, ent)
    for name, mod in mods.items():
        mod.load_state_dict(ck[f"{name}_state_dict"])
    ent.log_alpha = ck["log_alpha"]          # a registered parameter: torch accepts only an nn.Parameter here
    for name, opt in opts.items():
        opt.load_state_dict(ck[f"{name}_state_dict"])
    assert set(ck) == set(ref["keys"]) and type(ck["log_alpha"]).__name__ == ref["keys"]["log_alpha"]
    return mods, opts, ent


def reference_enums():
    """The reference's enum classes as foreign classes: same class names, member names and values (captured from the reference in
    tests/golden/reference_interfaces.json), defined outside this package."""
    from enum import Enum
    return {name: Enum(name, members) for name, members in reference_interfaces()["enums"].items()}
