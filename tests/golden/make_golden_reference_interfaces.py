#!/usr/bin/env python
"""Generate tests/golden/reference_interfaces.json: the parts of the reference's interface that this package must match, captured from the
EXECUTED reference (the staged copy oracle/_ref, plus the ESPO and PPO+LSTM modules of the reference tree itself):

  enums            member name -> value of the environment / framework enums the reference's runner compares across packages
  registry         parameter names of register_algorithm / register_environment
  default_configs  every algorithm's default_config.get_config() as a plain dict
  methods          method name -> parameter names of the five model classes (read from the sources)
  checkpoints      for PPO, SAC and FastSAC: the keys save() writes and their types, each module's parameters and state_dict entries
                   (names without the torch.compile wrapper's "_orig_mod." prefix, shapes, dtypes) and each optimizer's class, param_group
                   settings and parameter names in the optimizer's numbering

    python oracle/make_ref.py [REFERENCE_ROOT]
    python tests/golden/make_golden_reference_interfaces.py [REFERENCE_ROOT]
"""
import ast
import json
import os
import runpy
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
os.environ["TORCHDYNAMO_DISABLE"] = "1"

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import make_ref, ref_arm  # noqa: E402

OBS, ACT, N, HID, ATOMS = 5, 3, 2, 16, 21


def strip(name):
    return name.replace("_orig_mod.", "")


def module_layout(mod):
    return {"parameters": [[strip(n), list(p.shape)] for n, p in mod.named_parameters()],
            "state_dict": [[strip(n), list(t.shape), str(t.dtype).replace("torch.", "")] for n, t in mod.state_dict().items()]}


def optimizer_layout(opt, names):
    """names: parameter object id -> name.  Group settings are kept when JSON can hold them (betas as a list)."""
    groups = []
    for g in opt.param_groups:
        settings = {k: (list(v) if isinstance(v, tuple) else v) for k, v in g.items() if k != "params"}
        settings = {k: v for k, v in settings.items() if v is None or isinstance(v, (bool, int, float, str, list))}
        groups.append({"settings": settings, "param_names": [names[id(p)] for p in g["params"]]})
    return {"class": type(opt).__name__, "param_groups": groups}


def checkpoint_keys(path):
    ck = torch.load(path, weights_only=False)
    return {k: type(v).__name__ for k, v in ck.items()}


def methods(path, cls):
    for node in ast.walk(ast.parse(open(path).read())):
        if isinstance(node, ast.ClassDef) and node.name == cls:
            return {f.name: [a.arg for a in f.args.args if a.arg != "cls"] for f in node.body if isinstance(f, ast.FunctionDef)}
    raise AssertionError(f"no class {cls} in {path}")


def cfg(algorithm, save_model=True):
    C = ref_arm._ConfigDict
    return C(algorithm=algorithm, environment=C(seed=0, nr_envs=N),
             runner=C(save_model=save_model, track_console=False, track_tb=False, track_wandb=False))


def names_of(**modules):
    return {id(p): f"{prefix}.{strip(n)}" if prefix else strip(n) for prefix, m in modules.items() for n, p in m.named_parameters()}


def main():
    ref_root = sys.argv[1] if len(sys.argv) > 1 else make_ref.REF_ROOT
    refppo = ref_arm.import_reference()
    import rl_x.algorithms.sac.pytorch.sac as refsac
    import rl_x.algorithms.fastsac.pytorch.fastsac as reffs
    from rl_x.algorithms import algorithm_manager, deep_learning_framework_type
    from rl_x.environments import action_space_type, data_interface_type, environment_manager, observation_space_type, simulation_type
    out = {"enums": {}, "registry": {}, "default_configs": {}, "methods": {}, "checkpoints": {}}
    for mod, cls in ((action_space_type, "ActionSpaceType"), (observation_space_type, "ObservationSpaceType"), (data_interface_type, "DataInterfaceType"),
                     (simulation_type, "SimulationType"), (deep_learning_framework_type, "DeepLearningFrameworkType")):
        out["enums"][cls] = {m.name: m.value for m in getattr(mod, cls)}
    for mod, fn in ((algorithm_manager, "register_algorithm"), (environment_manager, "register_environment")):
        f = getattr(mod, fn)
        out["registry"][fn] = list(f.__code__.co_varnames[:f.__code__.co_argcount])

    staged = os.path.join(make_ref.DST, "rl_x", "algorithms")
    tree = os.path.join(ref_root, "rl_x", "algorithms")
    sources = {"ppo": (f"{staged}/ppo/pytorch", "ppo.py", "PPO"), "sac": (f"{staged}/sac/pytorch", "sac.py", "SAC"),
               "fastsac": (f"{staged}/fastsac/pytorch", "fastsac.py", "FastSAC"), "espo": (f"{tree}/espo/pytorch", "espo.py", "ESPO"),
               "ppo_lstm": (f"{tree}/ppo_lstm/flax", "ppo_lstm.py", "PPO_LSTM")}
    for algo, (d, src, cls) in sources.items():
        out["default_configs"][algo] = dict(runpy.run_path(os.path.join(d, "default_config.py"))["get_config"]("x"))
        out["methods"][cls] = methods(os.path.join(d, src), cls)

    torch.manual_seed(0)
    run = tempfile.mkdtemp(prefix="rlx_golden_interfaces_")
    from rl_x.algorithms.ppo.pytorch.default_config import get_config as ppo_config
    a = ppo_config("ppo.pytorch")
    a.device, a.bf16_mixed_precision_training, a.nr_steps, a.nr_epochs, a.minibatch_size, a.nr_hidden_units = "cpu", False, 4, 1, 8, HID
    env = ref_arm.SyntheticTorchEnv(N, OBS, ACT)
    m = refppo.PPO(cfg(a), env, env, os.path.join(run, "ppo"), None)
    os.makedirs(m.save_path, exist_ok=True)
    m.save()
    out["checkpoints"]["ppo"] = {
        "keys": checkpoint_keys(os.path.join(m.save_path, "best.model")),
        "modules": {"policy": module_layout(m.policy), "critic": module_layout(m.critic)},
        "optimizers": {"policy_optimizer": optimizer_layout(m.policy_optimizer, names_of(**{"": m.policy})),
                       "critic_optimizer": optimizer_layout(m.critic_optimizer, names_of(**{"": m.critic}))}}

    from rl_x.algorithms.sac.pytorch.default_config import get_config as sac_config
    from rl_x.environments.action_space_type import ActionSpaceType
    from rl_x.environments.data_interface_type import DataInterfaceType
    from rl_x.environments.observation_space_type import ObservationSpaceType

    class Props:
        observation_space_type, action_space_type, data_interface_type = ObservationSpaceType.FLAT_VALUES, ActionSpaceType.CONTINUOUS, DataInterfaceType.NUMPY

    class Env:
        general_properties, horizon = Props, 3
        single_observation_space = ref_arm._Space((OBS,))
        single_action_space = ref_arm._Space((ACT,), np.full(ACT, -1.0, np.float32), np.full(ACT, 1.0, np.float32))
        single_action_space.center, single_action_space.scale = np.zeros(ACT, np.float32), np.ones(ACT, np.float32)

    a = sac_config("sac.pytorch")
    a.device, a.bf16_mixed_precision_training, a.nr_hidden_units = "cpu", False, HID
    m = refsac.SAC(cfg(a), Env(), Env(), os.path.join(run, "sac"), None)
    os.makedirs(m.save_path, exist_ok=True)
    m.save()
    c = m.critic
    out["checkpoints"]["sac"] = {
        "keys": checkpoint_keys(os.path.join(m.save_path, "best.model")),
        "log_alpha": {"class": type(m.entropy_coefficient.log_alpha).__name__, "shape": list(m.entropy_coefficient.log_alpha.shape)},
        "modules": {"policy": module_layout(m.policy), "q1": module_layout(c.q1), "q2": module_layout(c.q2), "q1_target": module_layout(c.q1_target),
                    "q2_target": module_layout(c.q2_target)},
        "optimizers": {"policy_optimizer": optimizer_layout(m.policy_optimizer, names_of(**{"": m.policy})),
                       "q_optimizer": optimizer_layout(m.q_optimizer, names_of(q1=c.q1, q2=c.q2)),
                       "entropy_optimizer": optimizer_layout(m.entropy_optimizer, {id(m.entropy_coefficient.log_alpha): "log_alpha"})}}

    from rl_x.algorithms.fastsac.pytorch.default_config import get_config as fastsac_config
    a = fastsac_config("fastsac.pytorch")
    a.device, a.bf16_mixed_precision_training, a.compile_mode, a.nr_atoms = "cpu", False, "default", ATOMS
    Props.data_interface_type = DataInterfaceType.TORCH
    m = reffs.FastSAC(cfg(a), Env(), Env(), os.path.join(run, "fastsac"), None)
    os.makedirs(m.save_path, exist_ok=True)
    m.save()
    c = m.critic
    out["checkpoints"]["fastsac"] = {
        "keys": checkpoint_keys(os.path.join(m.save_path, "latest.model")),
        "log_alpha": {"class": type(m.entropy_coefficient.log_alpha).__name__, "shape": list(m.entropy_coefficient.log_alpha.shape)},
        "modules": {"policy": module_layout(m.policy), "q1": module_layout(c.q1), "q2": module_layout(c.q2), "q1_target": module_layout(c.q1_target),
                    "q2_target": module_layout(c.q2_target), "observation_normalizer": module_layout(m.observation_normalizer)},
        "optimizers": {"policy_optimizer": optimizer_layout(m.policy_optimizer, names_of(**{"": m.policy})),
                       "q_optimizer": optimizer_layout(m.q_optimizer, names_of(q1=c.q1, q2=c.q2)),
                       "entropy_optimizer": optimizer_layout(m.entropy_optimizer, {id(m.entropy_coefficient.log_alpha): "log_alpha"})},
        "meta": {"obs": OBS, "act": ACT, "nr_envs": N, "nr_atoms": ATOMS}}
    out["checkpoints"]["ppo"]["meta"] = {"obs": OBS, "act": ACT, "nr_envs": N, "hidden": HID}
    out["checkpoints"]["sac"]["meta"] = {"obs": OBS, "act": ACT, "nr_envs": N, "hidden": HID}
    with open(os.path.join(HERE, "reference_interfaces.json"), "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")


if __name__ == "__main__":
    main()
