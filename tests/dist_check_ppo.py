"""Sharded-vs-single PPO parity check (run as a script; under torchrun for world_size > 1).

Every rank serves its slice of the SAME global table environment (observations / rewards / terminations keyed by global env
index) and the same global action-noise table, so a world_size-W run must reproduce the world_size-1 run: identical global
permutation, owner-computes rows, one gradient all-reduce per minibatch (SURVEY.md §8 e).

    python tests/dist_check_ppo.py --out /tmp/w1.pt                                   # single process
    torchrun --nproc-per-node 2 --master-addr 127.0.0.1 tests/dist_check_ppo.py --out /tmp/w2.pt
    python tests/dist_check_ppo.py --compare /tmp/w1.pt /tmp/w2.pt
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NG, T, OBS, ACT, HID, MB, EPOCHS, ITERS = 64, 16, 376, 17, 256, 192, 2, 2


class _Space:
    def __init__(self, shape, low=None, high=None):
        self.shape, self.low, self.high = shape, low, high


class TableEnv:
    """Deterministic stream: step s of global env e returns table entries [s, e]."""

    def __init__(self, lo, hi, device):
        from rl_x_b200.environments.types import ActionSpaceType, ObservationSpaceType, DataInterfaceType

        class P:
            observation_space_type = ObservationSpaceType.FLAT_VALUES
            action_space_type = ActionSpaceType.CONTINUOUS
            data_interface_type = DataInterfaceType.TORCH
        self.general_properties = P
        g = torch.Generator().manual_seed(1234)
        steps = T * ITERS + 1
        self.obs = torch.randn(steps, NG, OBS, generator=g)[:, lo:hi].contiguous().to(device)
        self.rew = torch.randn(steps, NG, generator=g)[:, lo:hi].contiguous().to(device)
        self.term = (torch.rand(steps, NG, generator=g) < 0.05)[:, lo:hi].contiguous().to(device)
        self.trunc = torch.zeros(hi - lo, dtype=torch.bool, device=device)
        self.single_observation_space = _Space((OBS,))
        self.single_action_space = _Space((ACT,), np.full(ACT, -1.0, np.float32), np.full(ACT, 1.0, np.float32))
        self.t = 0

    def reset(self):
        return self.obs[0], {}

    def step(self, action):
        self.t += 1
        return self.obs[self.t], self.rew[self.t], self.term[self.t], self.trunc, {}

    def get_logging_info_dict(self, info):
        return {}

    def close(self):
        pass


METRICS = ["loss/policy_gradient_loss", "loss/critic_loss", "gradients/policy_grad_norm", "gradients/critic_grad_norm", "policy_ratio/clip_fraction",
           "steps/nr_episodes", "v_value/explained_variance"]


def run_model(world, rank, local, engine, exchange="peer", single=False):
    """One training run of the table problem on this rank's env slice (`single`: the whole problem on this GPU, ignoring any process
    group).  Returns (policy dict, critic dict, {metric: series}) - the weights are replicated, any rank's copy will do."""
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.ppo.b200.default_config import get_config
    from rl_x_b200.algorithms.ppo.b200.ppo import PPO
    if single:
        world, rank = 1, 0
    nl = NG // world
    lo, hi = rank * nl, (rank + 1) * nl
    dev = torch.device("cuda", local)
    a = get_config("ppo.b200")
    a.nr_steps, a.minibatch_size, a.nr_epochs, a.nr_hidden_units, a.total_timesteps = T, MB, EPOCHS, HID, NG * T * ITERS
    a.entropy_coef, a.gemm_engine, a.gradient_exchange = 0.01, engine, exchange
    a.ignore_process_group = bool(single)
    cfg = ConfigDict(algorithm=a, environment=ConfigDict(seed=5, nr_envs=nl),
                     runner=ConfigDict(save_model=False, track_console=False, track_tb=False, track_wandb=False, load_model=""))
    env = TableEnv(lo, hi, dev)
    model = PPO(cfg, env, env, "/tmp/rlx_dist_check", None)
    noise = torch.randn(T * ITERS, NG, ACT, generator=torch.Generator().manual_seed(99))[:, lo:hi].contiguous().to(dev)
    calls = {"n": 0}

    def draw(step):
        i = calls["n"]
        calls["n"] += 1
        return noise[i]

    model._draw_noise = draw
    logged = []
    model.log = lambda name, value, step: logged.append((name, float(value)))
    model.rank = 0 if single else model.rank  # a `single` instance logs whatever its rank in the job is
    model.train()
    if world > 1:
        assert model.gradient_exchange == exchange, f"asked for the {exchange} exchange, ran {model.gradient_exchange}"
        assert (model.peer_comm is not None) == (exchange == "peer")
    pol, cri = model.params.state_dicts()
    if world > 1:  # peers may still be reading this rank's exchange slots: nobody frees them before everybody is done
        torch.cuda.synchronize()
        torch.distributed.barrier()
    return pol, cri, {n: [v for m, v in logged if m == n] for n in METRICS}


def weight_and_metric_distance(a, b):
    """(worst relative weight difference, worst relative metric difference) between two run_model results."""
    worst = 0.0
    for x, y in ((a[0], b[0]), (a[1], b[1])):
        for k in x:
            worst = max(worst, float((x[k].double() - y[k].double()).norm() / y[k].double().norm()))
    mworst = 0.0
    for n in METRICS:
        u, v = np.asarray(a[2][n], dtype=np.float64), np.asarray(b[2][n], dtype=np.float64)
        if u.shape == v.shape and u.size:
            mworst = max(mworst, float(np.max(np.abs(u - v) / np.maximum(np.abs(v), 1.0))))
    return worst, mworst


def run(out, engine, exchange="peer"):
    world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pol, cri, metrics = run_model(world, rank, local, engine, exchange)
    if rank == 0:
        torch.save({"pol": pol, "cri": cri, "metrics": metrics, "world": world}, out)
        print(f"world={world} saved {out}")
    if world > 1:
        torch.distributed.destroy_process_group()


def compare(a_path, b_path):
    a, b = torch.load(a_path), torch.load(b_path)
    worst = 0.0
    for grp in ("pol", "cri"):
        for k in a[grp]:
            x, y = a[grp][k].double(), b[grp][k].double()
            rel = float((x - y).norm() / y.norm())
            worst = max(worst, rel)
    print(f"worlds {a['world']} vs {b['world']}: worst relative weight difference {worst:.3e}")
    for n in a["metrics"]:
        print("  ", n, a["metrics"][n], b["metrics"][n])
        np.testing.assert_allclose(a["metrics"][n], b["metrics"][n], rtol=2e-4, atol=2e-5)
    assert worst < 2e-5, worst
    print("sharded == single: OK")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--engine", default="auto")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"])
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
    else:
        run(args.out, args.engine, args.exchange)
