#!/usr/bin/env python
"""Benchmark of the PPO hot path (BASELINE.json metric: env-steps/sec, PPO update included).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--epochs E] [--engine auto|simt|tcgen05] [--dump-outputs DIR]

One "step" = one full PPO iteration of BASELINE config 2 per GPU: 128 rollout steps of 4096 synthetic Box(376)/Box(17)
envs (policy+critic forward, sampling, buffer writes), bootstrap values + GAE, then nr_epochs x (B / minibatch) shuffled
minibatch updates (gather, forward, loss, backward, two clip+Adam) — the body of the reference's `while` loop
(rl_x/algorithms/ppo/pytorch/ppo.py:195-393), driven through the plugin class PPO._train_iteration().

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  roofline      dominant kernel class (the MLP GEMMs): achieved fp32-equivalent TFLOP/s from CUDA events recorded around every
                launch of the class inside a second, instrumented timed region, vs the measured bf16 tensor peak
  roofline_hbm  the HBM-bound kernels named by north_star (minibatch gather, GAE) against the measured copy bandwidth
  kernel_ms     per-kernel-class device milliseconds per step from the same instrumented region
  cpu_baseline  the CPU oracle (oracle/ppo_oracle.py, torch fp32 on all host cores) on a bounded sample of the same workload
  e2e           same metric through PPO.train()'s loop with a NUMPY-interface env: observations/rewards in pinned HOST memory,
                H2D every step, actions D2H every step, metrics D2H every iteration
`--impl reference` times the CPU oracle alone (the reference's algorithm restated with the same torch primitives; the
reference itself is Python and does not travel to the GPU box).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

C2 = dict(nr_envs=4096, nr_steps=128, obs_dim=376, act_dim=17, hidden=256, minibatch_size=32768, nr_epochs=10)
FLOP_PER_SAMPLE_TRAIN = 1_584_128  # SURVEY.md §8: fwd 656 384 + bwd 927 744 per sample per epoch
FLOP_PER_SAMPLE_ROLLOUT = 656_384


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tflops=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback (B200_PROFILING.md)")


# ---------------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc = [], None
        self.nvml_rows, self.nvml_stop = [], False
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        # NVML in-process as well (a sample every 20 ms; nvidia-smi alone manages only a few per second on a busy box)
        self.nvml_thread = threading.Thread(target=self._read_nvml, args=(gpu_index,), daemon=True)
        self.nvml_thread.start()

    def _read_nvml(self, gpu_index):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(int(gpu_index))
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            while not self.nvml_stop:
                mask = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.nvml_rows.append((time.time(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), mx,
                                       pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0, [n for n, b in bits.items() if mask & b]))
                time.sleep(0.02)
        except Exception:
            return

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.nvml_stop = True
        sm, mx, reasons, power = [], [], set(), []
        nv = [r for r in list(self.nvml_rows) if t0 <= r[0] <= t1]
        if len(nv) >= 3:
            for _, c, m, w, rs in nv:
                sm.append(c); mx.append(m); power.append(w); reasons.update(rs)
            return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                    "power_w_max": max(power), "source": "nvml, 20 ms period"}
        for ts, line in self.rows:
            if not (t0 <= ts <= t1 + 0.15):
                continue
            parts = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ------------------------------------------------------------------------------------------------------- GPU arm
def build_model(args, rank, world, interface, global_minibatch=None, bf16=False):
    from rl_x_b200.runner.runner import Runner
    argv = [f"--environment.nr_envs={args.envs}", f"--environment.obs_dim={C2['obs_dim']}", f"--environment.act_dim={C2['act_dim']}",
            f"--environment.seed={1 + rank}", f"--environment.data_interface={interface}", "--environment.horizon=1000",
            f"--environment.stream={'ring' if interface == 'numpy' else 'fresh'}",
            f"--algorithm.nr_steps={C2['nr_steps']}", f"--algorithm.nr_epochs={args.epochs}",
            f"--algorithm.minibatch_size={global_minibatch if global_minibatch else args.minibatch * world}", f"--algorithm.nr_hidden_units={C2['hidden']}",
            f"--algorithm.gemm_engine={args.engine}", "--algorithm.total_timesteps=1e15",
            f"--algorithm.exact_global_permutation={'True' if args.exact_permutation else 'False'}",
            f"--algorithm.gradient_exchange={args.exchange}", f"--algorithm.peer_exchange_algorithm={args.exchange_algo}", f"--algorithm.bf16_mixed_precision_training={'True' if bf16 else 'False'}"]
    r = Runner(argv=argv)
    train_env, eval_env = r._create_train_and_eval_env(r._config)
    # weights and the permutation stream follow RANK 0's seed inside PPO.__init__ (broadcast); env streams differ via the env seed above
    model = r._model_class(r._config, train_env, eval_env, "/tmp/rlx_bench", None)
    return model


def timed_iterations(model, steps, dist):
    """Exactly `steps` iterations between two CUDA events, barrier + synchronize on both sides."""
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for _ in range(steps):
        model._train_iteration()
    e1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    if dist is not None:
        dist.barrier()
    return e0.elapsed_time(e1) / 1e3, t0, t1


DUMP_ENV_SAMPLE = 512   # env columns kept of the [T, N, act_dim] actions (seeded choice), so that the whole dump stays far below 64 MB


def dump_outputs(model, out_dir):
    """What the last timed iteration handed to a caller, as float32 .npy files: the updated parameters and Adam moments, the per-minibatch
    metric records, and the rollout buffer (per-(step, env) arrays in full, actions for a fixed seeded sample of env columns)."""
    os.makedirs(out_dir, exist_ok=True)
    torch.cuda.synchronize()
    b = model.batch
    cols = np.sort(np.random.default_rng(0).choice(b.actions.shape[1], size=min(DUMP_ENV_SAMPLE, b.actions.shape[1]), replace=False))
    arrays = {"params": model.params.flat, "adam_exp_avg": model.exp_avg, "adam_exp_avg_sq": model.exp_avg_sq, "metrics": model.metrics_dev,
              "log_probs": b.log_probs, "values": b.values, "rewards": b.rewards, "terminations": b.terminations, "advantages": b.advantages,
              "returns": b.returns, "actions_env_sample": b.actions[:, torch.from_numpy(cols).to(b.actions.device)], "actions_env_sample_index": cols}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else t
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))


def available_cores():
    """Host cores this process may actually use: scheduler affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def calibrate_threads(limit):
    """torch's intra-op thread count that makes the oracle's minibatch update fastest on this host (more threads than the
    box can schedule makes it much slower); the baseline is reported at its best setting."""
    from oracle import ppo_oracle as O
    cands = sorted({c for c in (4, 8, 16, 32, 48, 64, 96, 128, limit) if c <= limit})
    pol, cri = O.init_params(C2["obs_dim"], C2["act_dim"], C2["hidden"], seed=1)
    g = torch.Generator().manual_seed(0)
    m = 8192
    mbatch = (torch.randn(m, C2["obs_dim"], generator=g), torch.randn(m, C2["act_dim"], generator=g), -20 + torch.randn(m, generator=g),
              torch.randn(m, generator=g), torch.randn(m, generator=g))
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        L = O.Learner(pol, cri)
        L.minibatch_step(*mbatch)
        t = time.perf_counter()
        for _ in range(2):
            L.minibatch_step(*mbatch)
        t = time.perf_counter() - t
        if t < best_t:
            best, best_t = c, t
    return best


def cpu_baseline_sample(args, threads, minibatches=8, rollout_steps=8):
    """CPU oracle on a bounded sample of config 2, composed into seconds per full iteration (see `sample` in the result)."""
    from oracle import ppo_oracle as O
    torch.set_num_threads(threads)
    N, T, E, mb = args.envs, C2["nr_steps"], args.epochs, args.minibatch
    env = O.SyntheticVecEnv(N, C2["obs_dim"], C2["act_dim"], seed=1)
    pol, cri = O.init_params(C2["obs_dim"], C2["act_dim"], C2["hidden"], seed=1)
    L = O.Learner(pol, cri)
    gen = torch.Generator().manual_seed(1)
    state = env.reset()
    t = time.perf_counter()
    batch, state = O.rollout(L, env, state, rollout_steps, gen)
    t_act = (time.perf_counter() - t) / rollout_steps
    t = time.perf_counter()
    adv, ret = O.advantages_and_returns(L, batch, 0.99, 0.95)
    t_adv = (time.perf_counter() - t) / rollout_steps
    batch["advantages"], batch["returns"] = adv, ret
    flat = O.flatten({k: v for k, v in batch.items() if k != "next_states"})
    B = flat["states"].shape[0]
    rng = np.random.default_rng(1)
    idx = np.arange(B)
    rng.shuffle(idx)
    reps = max(1, (minibatches * mb + B - 1) // B)
    pool = np.concatenate([np.random.default_rng(i).permutation(B) for i in range(reps)])
    t = time.perf_counter()
    for i in range(minibatches):
        sel = torch.as_tensor(pool[i * mb:(i + 1) * mb] if mb <= len(pool) else np.resize(pool, mb))
        L.minibatch_step(flat["states"][sel], flat["actions"][sel], flat["log_probs"][sel], flat["advantages"][sel], flat["returns"][sel])
    t_mb = (time.perf_counter() - t) / minibatches
    nmb = -(-(N * T) // mb)
    t_iter = T * t_act + T * t_adv + E * nmb * t_mb
    sample = (f"{rollout_steps} rollout steps + next-value/GAE over {rollout_steps} steps at {N} envs, {minibatches} minibatch updates of {mb} rows; "
              f"composed as T*t_step + T*t_adv + E*{nmb}*t_minibatch (t_step={t_act * 1e3:.1f} ms, t_adv={t_adv * 1e3:.1f} ms, t_minibatch={t_mb * 1e3:.1f} ms)")
    return N * T / t_iter, t_iter, sample


def reference_class_run(args, threads, warmup, steps, max_seconds, eager, timeout):
    """The UNMODIFIED reference PPO class (oracle/_ref, staged by oracle/make_ref.py) for `warmup` + `steps` REAL iterations of this
    workload on the host cores, in a child process (CXX / TORCHDYNAMO_DISABLE must be set before torch is imported).  Returns the
    child's record or raises."""
    env = dict(os.environ)
    env["CXX"], env["CC"], env["WANDB_MODE"] = "/usr/bin/g++", "/usr/bin/gcc", "disabled"
    env["CUDA_VISIBLE_DEVICES"] = ""  # the reference arm is the reference's CPU path
    if eager:
        env["TORCHDYNAMO_DISABLE"] = "1"
    else:
        env.pop("TORCHDYNAMO_DISABLE", None)
    cmd = [sys.executable, "-m", "oracle.ref_arm", "--envs", str(args.envs), "--nr-steps", str(C2["nr_steps"]), "--obs", str(C2["obs_dim"]),
           "--act", str(C2["act_dim"]), "--hidden", str(C2["hidden"]), "--minibatch", str(args.minibatch), "--epochs", str(args.epochs),
           "--warmup", str(warmup), "--steps", str(steps), "--threads", str(threads), "--min-steps", str(min(3, steps))]
    if max_seconds:
        cmd += ["--max-seconds", str(max_seconds)]
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    for line in out.stdout.splitlines():
        if line.startswith("REF_ARM_JSON "):
            return json.loads(line[len("REF_ARM_JSON "):])
    raise RuntimeError(f"oracle.ref_arm failed (rc {out.returncode}): {out.stderr.strip().splitlines()[-1] if out.stderr.strip() else 'no output'}")


def run_reference_arm(args, rank, world):
    """--impl reference: REAL iterations of the reference's own PPO class on the host cores (BASELINE.md §3: compile_mode="default",
    CXX=/usr/bin/g++), all threads the box schedules best.  One compile iteration + `warmup` (capped at 1: every extra one costs ~25 s of
    CPU) untimed, then up to `steps` timed iterations, bounded to ~5 minutes of timed work (never fewer than 3); `steps` in the line is
    the number actually timed.  The composed port sample (the previous rounds' figure) is kept as a cross-check field."""
    if rank != 0:
        return
    from oracle import make_ref
    threads = calibrate_threads(available_cores())
    line = {"impl": "reference", "metric": "env-steps/sec (PPO update incl.)", "unit": "env-steps/s", "n_gpus": args.gpus, "steps_requested": args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, 1)}
    rec, err = None, None
    t_start = time.time()
    if make_ref.available():
        warm = 1 + min(args.warmup, 1)
        for eager in (False, True):
            try:
                rec = reference_class_run(args, threads, warm if not eager else min(args.warmup, 1), args.steps, 300.0, eager, timeout=1500)
                break
            except Exception as e:  # Inductor could not build on this host: say so and time the same classes eagerly
                err = f"{'eager' if eager else 'torch.compile'} run failed: {e}"
    else:
        err = "oracle/_ref not staged (python oracle/make_ref.py needs /root/reference)"
    if rec is not None:
        secs = rec["seconds"]
        t = float(np.mean(secs))
        value = args.envs * C2["nr_steps"] / t
        line.update({"value": value, "steps": len(secs), "warmup": rec["warmup_done"], "ms_per_step": t * 1e3,
                     "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "reference",
                                      "sample": f"{len(secs)} full iterations of {rec['class']} ({rec['file']}), device=cpu, fp32, "
                                                f"compile_mode={'default (Inductor, CXX=/usr/bin/g++)' if rec['torch_compile'] else 'eager (TORCHDYNAMO_DISABLE=1)'}, "
                                                f"{threads} torch threads; iteration seconds min/mean/max = {min(secs):.2f}/{t:.2f}/{max(secs):.2f}; "
                                                f"first (compile) iteration {rec['first_iteration_s']:.1f} s excluded",
                                      "phases_s": {k: float(np.mean(v)) for k, v in rec["phases"].items() if v}},
                     "wall_s": time.time() - t_start})
        if err:
            line["note"] = err
    else:
        per_step = []
        for i in range(max(args.warmup, 1) + min(args.steps, 5)):
            v, t_iter, sample = cpu_baseline_sample(args, threads, minibatches=4, rollout_steps=4)
            if i >= max(args.warmup, 1):
                per_step.append(t_iter)
        t = float(np.mean(per_step))
        value = args.envs * C2["nr_steps"] / t
        line.update({"value": value, "steps": len(per_step), "warmup": max(args.warmup, 1), "ms_per_step": t * 1e3, "note": err,
                     "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample + " (EXTRAPOLATED, not a full iteration)"}})
    if not args.no_cpu and rec is not None:
        v, t_iter, sample = cpu_baseline_sample(args, threads, minibatches=4, rollout_steps=4)
        line["port_cross_check"] = {"value": v, "unit": "env-steps/s", "kind": "port", "sample": sample}
    line["e2e"] = {"value": line["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    print(json.dumps(line))


def run_sac(args):
    """BASELINE config 4: SAC, synthetic Box(17)/Box(6), replay 1e6, batch 4096, one update per env step (UTD = 1 / nr_envs = 1).
    value = updates/s of sample + fused update on a full replay ring; e2e = the same through SAC._train_step() with a NUMPY-interface env."""
    from rl_x_b200 import _native as nt
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.sac.b200.default_config import get_config
    from rl_x_b200.algorithms.sac.b200.sac import SAC
    from rl_x_b200.environments.synthetic.box.create_env import create_train_and_eval_env
    from rl_x_b200.environments.synthetic.box.default_config import get_config as env_config
    torch.cuda.set_device(0)
    obs, act, batch, cap = 17, 6, 4096, 1_000_000
    e = env_config("synthetic.box")
    e.nr_envs, e.obs_dim, e.act_dim, e.data_interface, e.stream, e.ring_length, e.seed = 1, obs, act, "numpy", "ring", 64, 1
    a = get_config("sac.b200")
    a.batch_size, a.buffer_size, a.learning_starts, a.logging_frequency, a.total_timesteps = batch, cap, 5000, 10**9, 1e12
    cfg = ConfigDict(algorithm=a, environment=e, runner=ConfigDict(save_model=False, track_console=False, track_tb=False, track_wandb=False, load_model=""))
    env, _ = create_train_and_eval_env(cfg)
    model = SAC(cfg, env, env, "/tmp/rlx_bench_sac", None)
    model._begin_training()
    rb = model.replay_buffer
    g = torch.Generator(device="cuda").manual_seed(0)
    for t in (rb.states, rb.next_states, rb.actions, rb.rewards):
        t.normal_(generator=g)
    rb.actions.tanh_()
    rb.size, rb.pos = rb.capacity, 0
    model.global_step = 6000  # past learning_starts
    lib = nt.load()
    for _ in range(max(args.warmup, 3) * 20):
        model.update(rb.sample(batch))
    torch.cuda.synchronize()
    K = args.steps * 100
    lib.rlx_reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        model.update(rb.sample(batch))
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3
    launches = int(lib.rlx_launch_count())
    model.use_cuda_graph = False  # per-class event timing needs eager launches
    nt.timing_begin()
    for _ in range(20):
        model.update(rb.sample(batch))
    classes = nt.timing_end()
    model.use_cuda_graph = True
    # e2e: the full per-step loop (act, env.step on host arrays, replay add, sample, update)
    for _ in range(50):
        model._train_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        model._train_step()
    torch.cuda.synchronize()
    sec2 = time.perf_counter() - t0
    line = {"metric": "SAC updates/sec (sample + twin-Q/actor/alpha update), batch 4096", "value": K / sec, "unit": "updates/s", "n_gpus": 1, "steps": K,
            "warmup": max(args.warmup, 3) * 20, "ms_per_step": sec / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": "SAC synthetic Box(obs=17, act=6), replay=1e6 (full), batch=4096, nr_envs=1, hidden=256 (BASELINE.json configs[3])"},
            "gpu_launches": launches, "cuda_graph": True, "kernel_ms_eager": {k: round(v["ms"] / 20, 4) for k, v in classes.items() if v["launches"]},
            "e2e": {"value": K / sec2, "unit": "updates/s (= env-steps/s at nr_envs=1)", "h2d_bytes_per_step": 2 * batch * 8 + (2 * obs + act + 2) * 4,
                    "d2h_bytes_per_step": act * 4, "path": "SAC._train_step(): act -> env.step(numpy) -> replay add -> sample -> fused update"}}
    if not args.no_cpu:
        from oracle import sac_oracle as S
        threads = calibrate_threads(available_cores())
        torch.set_num_threads(threads)
        pol, q1, q2 = S.init_params(obs, act, 256, seed=1)
        L = S.Learner(pol, q1, q2, torch.full((act,), -1.0), torch.full((act,), 1.0))
        gg = torch.Generator().manual_seed(0)
        mk = lambda: (torch.randn(batch, obs, generator=gg), torch.randn(batch, obs, generator=gg), torch.tanh(torch.randn(batch, act, generator=gg)),
                      torch.randn(batch, generator=gg), torch.zeros(batch), torch.randn(batch, act, generator=gg), torch.randn(batch, act, generator=gg))
        L.update(*mk())
        t0 = time.perf_counter()
        n = 0
        while time.perf_counter() - t0 < 10.0:
            L.update(*mk())
            n += 1
        line["cpu_baseline"] = {"value": n / (time.perf_counter() - t0), "unit": "updates/s", "cores": threads, "kind": "port",
                                "sample": f"{n} oracle updates at batch 4096 in ~10 s (batch generation included, replay sampling excluded)"}
    # ~10 GFLOP of dense algebra per update (SURVEY.md §8 a15); every layer is < 10 us, so the bound that matters is launch latency
    flop = 2.0 * batch * (3 * (obs * 256 + 256 * 256 + 2 * 256 * act) + 3 * 4 * ((obs + act) * 256 + 256 * 256 + 256))
    line["roofline"] = {"bound": "tensor", "achieved": flop * line["value"] / 1e12, "peak": measured_peaks()["tflops"], "unit": "TFLOP/s",
                        "frac": flop * line["value"] / 1e12 / measured_peaks()["tflops"],
                        "note": "launch/latency-bound by size (every GEMM < 10 us); algorithmic FLOPs per update ~ fwd+bwd of policy and 4 Q passes"}
    return line


_AUX_VERDICT = None


def aux_paths_verdict():
    """May the FastSAC / PPO+LSTM workloads use (1) the tcgen05 3xTF32 engine for their dense layers (rlx_set_aux_gemm_engine) and (2) the
    one-launch-per-direction LSTM recurrence (rlx_set_lstm_persistent)?  Both switches were written after the round's GPU budget was spent,
    so they have to prove themselves ON THIS BOX before a timed run may use them: a subprocess (a kernel that traps or faults takes its CUDA
    context along - not this process's) runs, with the switches on, the FastSAC golden-batch parity test, the SIMT-vs-tensor gradient
    agreement at batch 1024, the PPO+LSTM oracle parity tests at the config-5 shape (T=128, 256 envs) and a smaller one, and the bit-for-bit
    comparison of the two recurrence paths.  Green AND the paths actually counted -> on.  If both together fail, each is tried alone.  The
    record carries every attempt.  No CPU oracle is timed here: the tests use it as the checker only."""
    global _AUX_VERDICT
    if _AUX_VERDICT is not None:
        return _AUX_VERDICT
    import subprocess
    import tempfile
    fastsac = ["tests/test_gpu_zzzz_fastsac.py::test_fastsac_updates_match_oracle_on_golden_batches",
               "tests/test_gpu_zzzz_fastsac.py::test_fastsac_engines_agree_at_batch_1024"]
    lstm = ["tests/test_gpu_zzz_ppo_lstm.py::test_lstm_fwdbwd_matches_oracle_autograd[16-24-64-8-256-128-64-0]",
            "tests/test_gpu_zzz_ppo_lstm.py::test_lstm_fwdbwd_matches_oracle_autograd[128-256-64-8-256-128-64-0]"]
    bitwise = ["tests/test_gpu_zzz_ppo_lstm.py::test_lstm_one_launch_recurrence_equals_per_step_recurrence_bit_for_bit"]

    def attempt(tensor, persistent):
        tests = (fastsac if tensor else []) + lstm + (bitwise if persistent else [])
        report = os.path.join(tempfile.mkdtemp(prefix="rlx_aux_"), "paths.txt")
        env = dict(os.environ, RLX_AUX_GEMM_ENGINE="1" if tensor else "0", RLX_LSTM_PERSISTENT="1" if persistent else "0", RLX_AUX_ENGINE_REPORT=report)
        rec = {"tensor_engine": tensor, "persistent_recurrence": persistent, "tests": len(tests)}
        try:
            proc = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider"] + tests, env=env, cwd=ROOT, capture_output=True,
                                  text=True, timeout=240)
            counts = open(report).read().split() if os.path.exists(report) else []
            tail = ((proc.stdout + proc.stderr).strip().splitlines() or [""])[-1]
            used = len(counts) == 2 and all(x.isdigit() for x in counts) and (not tensor or int(counts[0]) > 0) and (not persistent or int(counts[1]) > 0)
            rec.update(pytest=tail, returncode=proc.returncode, tensor_gemms=counts[0] if counts else None, persistent_launches=counts[1] if len(counts) > 1 else None)
            rec["green"] = bool(proc.returncode == 0 and used and f"{len(tests)} passed" in tail)
        except Exception as exc:  # timeout, no pytest, ...
            rec.update(error=f"{type(exc).__name__}: {exc}", green=False)
        return rec

    attempts = [attempt(True, True)]
    tensor = persistent = attempts[0]["green"]
    if not attempts[0]["green"]:
        attempts.append(attempt(True, False))
        tensor = attempts[-1]["green"]
        attempts.append(attempt(False, True))
        persistent = attempts[-1]["green"]
    _AUX_VERDICT = {"tensor_engine": bool(tensor), "persistent_recurrence": bool(persistent), "attempts": attempts}
    return _AUX_VERDICT


def with_aux_paths(fn, args):
    """Run a nested workload with the opt-in paths the verdict allows; the record says which ran and carries the counters as evidence."""
    from rl_x_b200 import _native as nt
    lib = nt.load()
    verdict = dict(aux_paths_verdict())

    def switches(tensor, persistent):
        lib.rlx_set_aux_gemm_engine(1 if tensor else 0)
        lib.rlx_set_lstm_persistent(1 if persistent else 0)
        return int(lib.rlx_aux_tc_gemm_count()), int(lib.rlx_lstm_persistent_launch_count())

    before = switches(verdict["tensor_engine"], verdict["persistent_recurrence"])
    try:
        line = fn(args)
    except Exception as exc:
        if not (verdict["tensor_engine"] or verdict["persistent_recurrence"]):
            raise
        # green check, failing workload: the number must not be lost to an opt-in - time it on the default paths and say so
        verdict.update(tensor_engine=False, persistent_recurrence=False, fell_back_after=f"{type(exc).__name__}: {exc}")
        before = switches(False, False)
        line = fn(args)
    finally:
        after = switches(False, False)
    line["gemm_engine"] = dict(verdict, engine="tcgen05-3xTF32" if verdict["tensor_engine"] else "simt", tensor_gemms_in_run=after[0] - before[0],
                               persistent_launches_in_run=after[1] - before[1])
    return line


def run_fastsac(args):
    """FastSAC (SURVEY.md §8 f4) at the reference's default update shape: batch 8192, 4 critic updates per policy update, 2 policy updates per
    environment step (rl_x/algorithms/fastsac/pytorch/default_config.py), 1024 x 4096 ring, synthetic Box(48) / Box(12).  One "step" =
    what the reference does after one vector-env step: sample 8 x 8192 rows (n-step gather), normalise states and next states (updating
    the running statistics), 8 critic + entropy updates with polyak, 2 policy updates.  value = critic updates/s."""
    from rl_x_b200 import _native as nt
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.fastsac.b200.default_config import get_config
    from rl_x_b200.algorithms.fastsac.b200.fastsac import FastSAC
    from rl_x_b200.algorithms.fastsac.b200.replay_buffer import ReplayBuffer
    from rl_x_b200.environments.types import ActionSpaceType, ObservationSpaceType, DataInterfaceType
    torch.cuda.set_device(0)
    N, obs, act, n_steps = 4096, 48, 12, 3

    class Space:
        def __init__(self, shape, **kw):
            self.shape = shape
            self.__dict__.update(kw)

    class Props:
        observation_space_type, action_space_type, data_interface_type = ObservationSpaceType.FLAT_VALUES, ActionSpaceType.CONTINUOUS, DataInterfaceType.TORCH

    class Env:
        general_properties, horizon = Props, 1000
        single_observation_space = Space((obs,))
        single_action_space = Space((act,), low=np.full(act, -1.0, np.float32), high=np.full(act, 1.0, np.float32), center=np.zeros(act, np.float32),
                                    scale=np.ones(act, np.float32))

    a = get_config("fastsac.b200")
    a.n_steps = n_steps
    cfg = ConfigDict(algorithm=a, environment=ConfigDict(seed=1, nr_envs=N),
                     runner=ConfigDict(save_model=False, track_console=False, track_tb=False, track_wandb=False, load_model=""))
    model = FastSAC(cfg, Env(), Env(), "/tmp/rlx_bench_fastsac", None)
    model.set_train_mode()
    rb = ReplayBuffer(a.buffer_size_per_env, N, (obs,), (act,), n_steps, a.gamma, model.device)
    g = torch.Generator(device="cuda").manual_seed(0)
    for t in (rb.states, rb.next_states, rb.actions, rb.rewards):
        t.normal_(generator=g)
    rb.actions.tanh_()
    rb.dones.copy_((torch.rand(rb.dones.shape, device="cuda", generator=g) < 0.01).float())
    rb.size, rb.pos = rb.capacity, 0
    npu, ncu, B = a.nr_policy_updates_per_step, a.nr_critic_updates_per_policy_update, a.batch_size
    cm, pm = torch.zeros(8, device="cuda"), torch.zeros(8, device="cuda")

    def step():
        ts, tns, ta, tr, td, ttr, teff = rb.sample(npu * ncu * B)
        ts = model.normalize(ts, update=True).view(npu, ncu, B, -1)
        tns = model.normalize(tns, update=True).view(npu, ncu, B, -1)
        ta = ta.view(npu, ncu, B, -1)
        tr, td, ttr, teff = (t.view(npu, ncu, B) for t in (tr, td, ttr, teff))
        for i in range(npu):
            for j in range(ncu):
                model.critic_update(ts[i, j], tns[i, j], ta[i, j], tr[i, j], td[i, j], ttr[i, j], teff[i, j], cm)
            model.policy_update(ts[i, -1], pm)

    lib = nt.load()
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    K = args.steps * 4
    lib.rlx_reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3
    line = {"metric": "FastSAC critic updates/sec (n-step sample + C51 twin-critic / actor / alpha updates), batch 8192", "value": K * npu * ncu / sec,
            "unit": "critic updates/s", "n_gpus": 1, "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": sec / K * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"FastSAC synthetic Box(obs={obs}, act={act}), ring 1024 x {N}, n_steps={n_steps}, batch={B}, {ncu} critic per policy update, "
                                   f"{npu} policy updates per step (reference defaults)"},
            "gpu_launches": int(lib.rlx_launch_count()), "q_loss": float(cm[0]), "policy_loss": float(pm[0])}
    if not args.no_cpu:
        from oracle import fastsac_oracle as FS
        threads = calibrate_threads(available_cores())
        torch.set_num_threads(threads)
        pol, q1, q2 = FS.reference_init(obs, act, int(a.nr_atoms), 1)
        L = FS.Learner(pol, q1, q2, torch.ones(act), a.learning_rate, a.weight_decay, (a.adam_beta1, a.adam_beta2), a.gamma, a.tau, a.v_min, a.v_max, int(a.nr_atoms),
                       a.target_entropy, a.alpha_init, a.log_std_min, a.log_std_max)
        gg = torch.Generator().manual_seed(0)
        rn = lambda *s_: torch.randn(*s_, generator=gg)
        mk = lambda: (rn(B, obs), rn(B, obs), torch.tanh(rn(B, act)), rn(B), torch.zeros(B), torch.zeros(B), torch.ones(B), rn(B, act))
        L.critic_and_entropy_step(*mk())
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < 10.0:
            L.critic_and_entropy_step(*mk())
            n += 1
        line["cpu_baseline"] = {"value": n / (time.perf_counter() - t0), "unit": "critic updates/s", "cores": threads, "kind": "port",
                                "sample": f"{n} oracle critic updates at batch {B} in ~10 s (policy updates and sampling excluded)"}
    return line


def run_ppo_lstm(args):
    """BASELINE config 5: PPO+LSTM, synthetic Box(obs=64, act=8), 2048 envs x 128 steps, minibatch 32768 rows (= 256 envs x 128 steps), 10
    epochs, reference widths (encoders 128, LSTM 64, torso 256).  value = env-steps/s of full iterations through PPO_LSTM.train()."""
    from rl_x_b200 import _native as nt
    from rl_x_b200.config_dict import ConfigDict
    from rl_x_b200.algorithms.ppo_lstm.b200.default_config import get_config
    from rl_x_b200.algorithms.ppo_lstm.b200.ppo_lstm import PPO_LSTM
    from rl_x_b200.environments.synthetic.box.create_env import create_train_and_eval_env
    from rl_x_b200.environments.synthetic.box.default_config import get_config as env_config
    torch.cuda.set_device(0)
    N, T, obs, act, mb, E = 2048, 128, 64, 8, 32768, 10
    W, K = 1, max(2, min(args.steps, 3))

    def make(n_envs, steps, minibatch, epochs, iterations, graph):
        e = env_config("synthetic.box")
        e.nr_envs, e.obs_dim, e.act_dim, e.seed = n_envs, obs, act, 1
        a = get_config("ppo_lstm.b200")
        a.nr_steps, a.minibatch_size, a.nr_epochs, a.total_timesteps, a.use_cuda_graph = steps, minibatch, epochs, float(n_envs * steps * iterations), graph
        cfg = ConfigDict(algorithm=a, environment=e, runner=ConfigDict(save_model=False, track_console=False, track_tb=False, track_wandb=False, load_model=""))
        env, _ = create_train_and_eval_env(cfg)
        m = PPO_LSTM(cfg, env, env, "/tmp/rlx_bench_lstm", None)
        m.start_logging, m.log, m.end_logging = (lambda *a_, **k_: None), (lambda *a_, **k_: None), (lambda *a_, **k_: None)
        return m

    # The timed run replays each minibatch update as ONE captured CUDA graph (use_cuda_graph).  That path's first hardware run is this one,
    # so it has to earn its place here: two iterations at a small shape, replayed vs eagerly launched, must leave bit-identical weights
    # (same kernels, same order, no atomics); otherwise - or if capture fails - the timed run launches eagerly and the record says why.
    graph_note = {"enabled": True, "check": "weights bit-identical to eager launches after 2 iterations (64 envs x 16 steps, 2 epochs x 4 minibatches)"}
    try:
        pair = []
        for graph in (False, True):
            m = make(64, 16, 256, 2, 2, graph)
            m.train()
            torch.cuda.synchronize()
            pair.append((m.policy_params.clone(), m.critic_params.clone()))
        if not (torch.equal(pair[0][0], pair[1][0]) and torch.equal(pair[0][1], pair[1][1])):
            graph_note = {"enabled": False, "check": "replayed update differs from eager launches: max |d| = %.3e" % float((pair[0][0] - pair[1][0]).abs().max())}
    except Exception as exc:  # a failed capture must not cost the workload its number
        graph_note = {"enabled": False, "check": f"capture failed: {type(exc).__name__}: {exc}"}
    model = make(N, T, mb, E, W + K, graph_note["enabled"])
    lib = nt.load()
    stamps, launches = [], []

    def start_logging(step):
        torch.cuda.synchronize()
        stamps.append(time.perf_counter())
        launches.append(int(lib.rlx_launch_count()))

    model.start_logging = start_logging
    torch.cuda.synchronize()
    lib.rlx_reset_launch_count()
    stamps.append(time.perf_counter())
    launches.append(0)
    model.train()
    it = np.diff(np.asarray(stamps))[W:]
    sec = float(np.mean(it))
    line = {"metric": "env-steps/sec (PPO+LSTM update incl.)", "value": N * T / sec, "unit": "env-steps/s", "n_gpus": 1, "steps": len(it), "warmup": W,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"PPO+LSTM synthetic Box(obs={obs}, act={act}), num_envs={N}, seq_len={T}, minibatch={mb} rows (256 envs), nr_epochs={E} "
                                   "(BASELINE.json configs[4])"},
            "gpu_launches": int((launches[-1] - launches[W]) / max(len(it), 1)), "timing": "host clock around synchronised iterations of PPO_LSTM.train()",
            "cuda_graph": graph_note}
    if not args.no_cpu:
        from oracle import ppo_lstm_oracle as LO
        threads = calibrate_threads(available_cores())
        torch.set_num_threads(threads)
        pol, cri = LO.init_params(obs, act, hidden=256, enc=128, lstm=64, std_dev=1.0, seed=1)
        learner = LO.Learner(pol, cri)
        n_env = 64  # a quarter-of-a-quarter minibatch keeps the leg ~10 s; cost is linear in envs
        g = torch.Generator().manual_seed(0)
        rn = lambda *s_: torch.randn(*s_, generator=g)
        mbatch = dict(states=rn(T, n_env, obs), actions=rn(T, n_env, act), log_probs=rn(T, n_env) * 0.1 - 8.0, returns=rn(T, n_env), advantages=rn(T, n_env),
                      dones=(torch.rand(T, n_env, generator=g) < 0.01).float(), init_carry=(torch.zeros(n_env, 64), torch.zeros(n_env, 64)))
        learner.minibatch_step(mbatch)
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < 8.0:
            learner.minibatch_step(mbatch)
            n += 1
        t_mb = (time.perf_counter() - t0) / n * (256 / n_env)
        t_iter = E * (N // 256) * t_mb
        line["cpu_baseline"] = {"value": N * T / t_iter, "unit": "env-steps/s", "cores": threads, "kind": "port (parity unpinned: the Flax reference cannot run here)",
                                "sample": f"{n} oracle minibatch updates of {n_env} envs x {T} steps; composed as E*8*t_minibatch (update only, rollout excluded)"}
    return line


def workload_config(args, world):
    return {"workload": f"PPO synthetic Box(obs={C2['obs_dim']}, act={C2['act_dim']}) ~Humanoid, num_envs={args.envs}/GPU, horizon={C2['nr_steps']}, "
                        f"hidden={C2['hidden']}, nr_epochs={args.epochs}, minibatch={args.minibatch}/GPU (BASELINE.json configs[1])",
            "num_envs_global": args.envs * world, "minibatch_size_global": args.minibatch * world, "nr_epochs": args.epochs,
            "parallelism": (f"dp{world} (env-sharded, " + ("reference-exact global permutation" if args.exact_permutation else "rank-local PCG64 shuffles")
                            + (", 1 peer-memory all-reduce kernel (rlx_comm, NVLink loads) of the flat gradient per minibatch)" if args.exchange == "peer"
                               else ", 1 NCCL all-reduce of the flat gradient per minibatch)")) if world > 1 else "single GPU",
            "l2_policy": "per-step working set (rollout buffer 0.83 GB + gathered copy 0.83 GB + activations) exceeds the 126 MB L2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--epochs", type=int, default=C2["nr_epochs"])
    ap.add_argument("--envs", type=int, default=C2["nr_envs"], help="envs per GPU")
    ap.add_argument("--minibatch", type=int, default=C2["minibatch_size"], help="minibatch rows per GPU")
    ap.add_argument("--engine", default="auto")
    ap.add_argument("--exact-permutation", action="store_true",
                    help="multi-GPU: reference-exact global permutation on every rank (host-bound) instead of rank-local shuffles")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="multi-GPU gradient exchange: library peer-memory kernel or NCCL")
    ap.add_argument("--exchange-algo", default="auto", choices=["auto", "one_shot", "two_shot"], help="peer exchange kernel: one-shot (auto) / two-shot (experimental)")
    ap.add_argument("--head-engine", default="fused", choices=["fused", "gemm", "mma"],
                    help="PPO loss head: fused SIMT kernel, the GEMM formulation, or the fused mma.sync kernel")
    ap.add_argument("--workload", default="ppo", choices=["ppo", "sac", "fastsac", "ppo_lstm"])
    ap.add_argument("--tc-pair", default="", help="tcgen05 CTA-pair engine: MODE[:FWD_BN], MODE 0 off / 1 weight gradients (default) / 2 all GEMMs, FWD_BN 128|256")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-bf16", action="store_true", help="N=1: skip the bf16-autocast sub-line")
    ap.add_argument("--no-workloads", action="store_true", help="N=1: skip the nested SAC / FastSAC / PPO+LSTM records")
    ap.add_argument("--no-aux-engine", action="store_true", help="FastSAC / PPO+LSTM workloads: stay on the SIMT GEMM engine without running the tensor-engine check")
    ap.add_argument("--no-parity-check", action="store_true", help="N>1: skip the sharded-vs-single parity run before timing")
    ap.add_argument("--no-strict", action="store_true", help="N>1: skip the second timed region at the contract's GLOBAL minibatch of 32768")
    ap.add_argument("--global-minibatch", type=int, default=0, help="N>1: headline region with this GLOBAL minibatch instead of --minibatch per GPU")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="PPO workload: write what the last timed step computed to DIR/<name>.npy (rank 0), for output-by-output comparison of two builds")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)

    if args.workload in ("sac", "fastsac", "ppo_lstm"):
        if rank == 0:
            fn = {"sac": run_sac, "fastsac": run_fastsac, "ppo_lstm": run_ppo_lstm}[args.workload]
            print(json.dumps(fn(args) if args.workload == "sac" or args.no_aux_engine else with_aux_paths(fn, args)))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback; use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from rl_x_b200 import _native as nt
    lib = nt.load()
    lib.rlx_set_head_engine({"fused": 0, "gemm": 1, "mma": 2}[args.head_engine])
    if args.tc_pair:
        mode, _, bn = args.tc_pair.partition(":")
        lib.rlx_set_tc_pair(int(mode), int(bn or 0))

    # ---- multi-GPU parity, visible to whoever runs the bench: the env-sharded run (reference-exact global permutation, this exchange, this
    # GEMM engine) against the same global problem on ONE GPU (tests/dist_check_ppo.py: 64 envs x 16 steps, obs 376 / act 17 / hidden 256,
    # 2 iterations x 2 epochs of 6 minibatches), before anything is timed
    parity_check = None
    if world > 1 and not args.no_parity_check:
        import importlib.util
        spec = importlib.util.spec_from_file_location("dist_check_ppo", os.path.join(ROOT, "tests", "dist_check_ppo.py"))
        chk = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(chk)
        sharded = chk.run_model(world, rank, local_rank, args.engine, args.exchange)
        dist.barrier()
        if rank == 0:
            single = chk.run_model(world, rank, local_rank, args.engine, args.exchange, single=True)
            wrel, mrel = chk.weight_and_metric_distance(sharded, single)
            parity_check = {"max_rel": wrel, "metrics_max_rel": mrel, "mode": "exact_global_permutation", "exchange": args.exchange, "world": world,
                            "problem": f"{chk.NG} envs x {chk.T} steps, obs {chk.OBS} act {chk.ACT} hidden {chk.HID}, minibatch {chk.MB}, "
                                       f"{chk.ITERS} iterations x {chk.EPOCHS} epochs", "passed": bool(wrel < 2e-5 and mrel < 2e-4),
                            "bar": "weights 2e-5 of the norm, logged metrics 2e-4 (tests/dist_check_ppo.py)"}
        dist.barrier()

    model = build_model(args, rank, world, "torch", global_minibatch=args.global_minibatch or None)
    model._begin_training()
    for _ in range(args.warmup):
        model._train_iteration()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    lib.rlx_reset_launch_count()
    seconds, t0, t1 = timed_iterations(model, args.steps, dist)
    launches = int(lib.rlx_launch_count())
    clocks = sampler.stop(t0, t1) if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(model, args.dump_outputs)
    if dist is not None:
        tt = torch.tensor([seconds], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        seconds = float(tt.item())
    steps_per_iter = args.envs * world * C2["nr_steps"]
    value = steps_per_iter * args.steps / seconds

    # instrumented second region: CUDA events around every launch, per kernel class
    nt.timing_begin()
    for _ in range(2):
        model._train_iteration()
    classes = nt.timing_end()
    kernel_ms = {k: round(v["ms"] / 2, 4) for k, v in classes.items() if v["launches"]}
    tc_shape_ok = C2["hidden"] % 128 == 0 and C2["obs_dim"] % 4 == 0
    engine = "tcgen05-3xTF32" if lib.rlx_get_gemm_engine() == 1 and tc_shape_ok else "simt-fp32"
    peaks = measured_peaks()
    gemm = {k: classes[k] for k in ("gemm_fwd", "gemm_dx", "gemm_dw")}
    gflops, gms = sum(v["flops"] for v in gemm.values()), sum(v["ms"] for v in gemm.values())
    achieved_tf = gflops / (gms * 1e-3) / 1e12 if gms > 0 else 0.0
    total_ms = sum(v["ms"] for v in classes.values())
    roofline = {"bound": "tensor", "kernel": f"MLP GEMMs ({engine}): gemm_fwd + gemm_dx + gemm_dw", "achieved": achieved_tf, "peak": peaks["tflops"],
                "unit": "TFLOP/s", "frac": achieved_tf / peaks["tflops"], "traffic": None, "peak_source": peaks["source"],
                "share_of_step": gms / total_ms if total_ms else None,
                "note": "fp32-equivalent algorithmic FLOPs (2*M*N*K) of the exact-fp32 path against the dense bf16 tensor peak"}
    # DRAM traffic per GEMM launch from the committed ncu --set full capture (profiles/roofline_traffic.json), next to the algorithmic bytes
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
            tr = json.load(fh)
        roofline["traffic"] = tr["gemm_dram_bytes_per_minibatch"] / tr["gemm_launches_per_minibatch"]
        roofline["traffic_source"] = tr["note"]
    except (OSError, KeyError, ValueError):
        pass
    glaunch = sum(v["launches"] for v in gemm.values())
    roofline["algorithmic_bytes_per_launch"] = sum(v["bytes"] for v in gemm.values()) / glaunch if glaunch else None
    # what the tensor pipe actually executes: 3 TF32 MMAs per fp32 product, against the tf32 dense rate (half the measured bf16 rate)
    roofline["mma"] = {"achieved": 3 * achieved_tf, "peak": peaks["tflops"] / 2, "unit": "TFLOP/s tf32", "frac": 3 * achieved_tf / (peaks["tflops"] / 2),
                       "note": "3xTF32 split (hi*hi + hi*lo + lo*hi); tf32 peak taken as half of the measured bf16 peak"}
    hbm = {}
    for name in ("gather", "gae", "clip_adam", "head_train", "peer_allreduce"):
        c = classes[name]
        if c["launches"]:
            gbs = c["bytes"] / (c["ms"] * 1e-3) / 1e9
            hbm[name] = {"achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                         "bytes_per_launch": c["bytes"] / c["launches"], "us_per_launch": c["ms"] * 1e3 / c["launches"]}

    # the GAE kernel at config 2 is one 10 MB wave (latency-bound); the same kernel on a rollout that fills the machine shows its HBM rate
    if rank == 0:
        Tg, Ng = C2["nr_steps"], 65536
        gr, gt, gv = (torch.randn(Tg, Ng, device="cuda"), (torch.rand(Tg, Ng, device="cuda") < 0.02).float(), torch.randn(Tg, Ng, device="cuda"))
        ga, gret, glv = torch.empty_like(gr), torch.empty_like(gr), torch.randn(Ng, device="cuda")
        for _ in range(3):
            model.kernels.gae(gr, gt, gv, model.gamma, model.gae_lambda, ga, gret, last_value=glv)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            model.kernels.gae(gr, gt, gv, model.gamma, model.gae_lambda, ga, gret, last_value=glv)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / 10
        gbs = 20.0 * Tg * Ng / (us * 1e-6) / 1e9
        hbm["gae_65536_envs"] = {"achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                                 "bytes_per_launch": 20.0 * Tg * Ng, "us_per_launch": us,
                                 "note": "same kernel, T=128 x 65 536 envs (168 MB working set > L2), 20 B per (t, env)"}
        del gr, gt, gv, ga, gret, glv

    line = {"metric": "env-steps/sec (PPO update incl.)", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": seconds / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, world), "gpu_launches": launches, "clocks": clocks,
            "roofline": roofline, "roofline_hbm": hbm, "kernel_ms": kernel_ms, "gemm_engine": engine,
            "gradient_exchange": (model.gradient_exchange if world > 1 else None),
            "train_tflops_per_step": FLOP_PER_SAMPLE_TRAIN * args.envs * C2["nr_steps"] * args.epochs / 1e12}

    if parity_check is not None:
        line["parity_check"] = parity_check
    # end-to-end through the host-buffer path (NUMPY-interface env: pinned host observations, H2D/D2H every step)
    model._end_training()
    if world > 1 and not args.no_strict and not args.global_minibatch:
        # SURVEY.md §8(d) C3 as the contract wrote it: the GLOBAL minibatch stays 32768 (4096 rows per rank at 8 GPUs, 128 exchanges per
        # epoch instead of 16): strong-scaled minibatches, reported next to the weak-scaling headline
        torch.cuda.synchronize()
        dist.barrier()  # peers may still be reading this rank's exchange slots
        del model
        torch.cuda.empty_cache()
        m3 = build_model(args, rank, world, "torch", global_minibatch=C2["minibatch_size"])
        m3._begin_training()
        for _ in range(args.warmup):
            m3._train_iteration()
        s3, _, _ = timed_iterations(m3, args.steps, dist)
        tt = torch.tensor([s3], device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        s3 = float(tt.item())
        line["strict_c3"] = {"value": steps_per_iter * args.steps / s3, "unit": "env-steps/s", "ms_per_step": s3 / args.steps * 1e3,
                             "minibatch_size_global": C2["minibatch_size"], "rows_per_rank_per_minibatch": C2["minibatch_size"] // world,
                             "exchanges_per_step": args.epochs * (args.envs * world * C2["nr_steps"] // C2["minibatch_size"]),
                             "note": "same envs per GPU; global minibatch fixed at the contract's 32768 (config C3 of SURVEY.md §8)"}
        m3._end_training()
        model = m3
    if not args.no_e2e:
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        del model
        torch.cuda.empty_cache()
        m2 = build_model(args, rank, world, "numpy")
        m2._begin_training()
        for _ in range(max(1, args.warmup - 1)):
            m2._train_iteration()
        s2, _, _ = timed_iterations(m2, args.steps, dist)
        if dist is not None:
            tt = torch.tensor([s2], device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            s2 = float(tt.item())
        T, N = C2["nr_steps"], args.envs
        h2d = T * N * (C2["obs_dim"] * 4 + 4 + 2) + args.epochs * N * T * 8 + 4
        d2h = T * N * C2["act_dim"] * 4 + m2.metrics_host.numel() * 4 + 16
        line["e2e"] = {"value": steps_per_iter * args.steps / s2, "unit": "env-steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "ms_per_step": s2 / args.steps * 1e3,
                       "path": "PPO._train_iteration() with a NUMPY-interface env: obs/reward/done from pinned host buffers every env step, actions read back every env step"}
        m2._end_training()
        del m2
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import make_ref
        threads = calibrate_threads(available_cores())
        v, t_iter, sample = cpu_baseline_sample(args, threads)
        port = {"value": v, "unit": "env-steps/s", "cores": threads, "host_cores_available": available_cores(), "kind": "port", "sample": sample, "s_per_step": t_iter}
        line["cpu_baseline"] = port
        if make_ref.available():
            # the reference's own class on this box's host cores: ONE full iteration of this workload after one warm-up iteration, eager
            # (Inductor's ~1 min of compilation does not fit a bounded leg; `--impl reference` times the compiled classes)
            try:
                rec = reference_class_run(args, threads, 1, 1, None, True, timeout=600)
                t = float(np.mean(rec["seconds"]))
                line["cpu_baseline"] = {"value": args.envs * C2["nr_steps"] / t, "unit": "env-steps/s", "cores": threads, "host_cores_available": available_cores(),
                                        "kind": "reference", "s_per_step": t,
                                        "sample": f"1 full iteration of {rec['class']} ({rec['file']}) on this workload after 1 warm-up iteration; device=cpu, fp32, "
                                                  f"eager (TORCHDYNAMO_DISABLE=1), {threads} torch threads", "port_cross_check": port}
            except Exception as e:
                line["cpu_baseline"]["note"] = f"reference class run failed ({e}); port sample reported"
    if rank == 0 and world == 1 and not args.no_bf16:
        # the reference's DEFAULT precision mode (bf16 autocast, ppo/pytorch/default_config.py:11) as a separate sub-line: same workload, same
        # timing rules, kept apart from the fp32 headline (BASELINE.md's CPU numbers and the parity bar of 1e-5 are fp32)
        try:
            torch.cuda.empty_cache()
            mb16 = build_model(args, rank, world, "torch", bf16=True)
            mb16._begin_training()
            for _ in range(args.warmup):
                mb16._train_iteration()
            sb, _, _ = timed_iterations(mb16, args.steps, None)
            nt.timing_begin()
            for _ in range(2):
                mb16._train_iteration()
            cls16 = nt.timing_end()
            g16 = {k: cls16[k] for k in ("gemm_fwd", "gemm_dx", "gemm_dw")}
            tf16 = sum(v["flops"] for v in g16.values()) / (sum(v["ms"] for v in g16.values()) * 1e-3) / 1e12
            line["bf16_autocast"] = {"value": steps_per_iter * args.steps / sb, "unit": "env-steps/s", "ms_per_step": sb / args.steps * 1e3, "dtype": "bf16-autocast",
                                     "note": "bf16_mixed_precision_training=True: bf16 values in fp32 storage, ONE tcgen05 kind::tf32 MMA per product (exact for bf16 operands), "
                                             "fp32 accumulation, losses / clipping / Adam in fp32 as in the reference",
                                     "kernel_ms": {k: round(v["ms"] / 2, 4) for k, v in cls16.items() if v["launches"]},
                                     "roofline": {"bound": "tensor", "achieved": tf16, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": tf16 / peaks["tflops"],
                                                  "note": "algorithmic FLOPs of the MLP GEMMs against the measured dense bf16 peak; the tf32 pipe this mode runs on peaks at half of it"}}
            mb16._end_training()
            del mb16
            lib.rlx_set_autocast_bf16(0)
        except Exception as e:
            line["bf16_autocast"] = {"error": f"{type(e).__name__}: {e}"}
            lib.rlx_set_autocast_bf16(0)
    if rank == 0 and world == 1 and not args.no_workloads:
        # the other BASELINE.json configs, each with its own value / cpu_baseline (SAC also its roofline), nested so that the one parsed
        # line carries them (they are separate workloads, not part of `value`)
        line["workloads"] = {}
        for name, fn in (("sac", run_sac), ("fastsac", run_fastsac), ("ppo_lstm", run_ppo_lstm)):
            try:
                torch.cuda.empty_cache()
                line["workloads"][name] = fn(args) if name == "sac" or args.no_aux_engine else with_aux_paths(fn, args)
            except Exception as e:
                line["workloads"][name] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
