#!/usr/bin/env python
"""bench.py -- env steps/sec of the Anakin ff_ppo training step (BASELINE.json metric) on N B200s.

  python bench.py --gpus N --steps K --warmup W            (N>1: launch under torchrun)
  python bench.py ... --dump-outputs DIR                   also write the last timed step's outputs as DIR/<name>.npy
  python bench.py --impl reference ...                     CPU arm: the torch-CPU port of the same step

One "step" = one Anakin update step per GPU: T=128 env steps of E=4096 envs (rollout with the
actor/critic MLP[256,256] forwards on synthetic Box obs_dim=64 observations), the GAE scan, and
4 epochs x 16 minibatches of the fused PPO loss/backward + clip/Adam (+ gradient all-reduce for N>1).
value = N * T * E * K / time (whole-job env steps/s), timed with CUDA events on the stream the work
runs on, barrier + synchronize on both sides, MAX over ranks.  Two timed regions of K steps each run:
the device-resident one (value) and the end-to-end one with host copies (e2e, with the spread over its
K steps).  The inputs are seeded (arch.seed), so the same arguments give the same inputs on every
run and the dumped outputs of two builds can be compared array for array.  Working set per step (trajectory obs +
next_obs = 2 x 128 MiB fp32, or 2 x 64 MiB bf16) exceeds L2 together with weights/activations, so no
explicit L2 flush is needed between steps (stated in config.l2).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env steps/sec Anakin PPO at 1/2/4/8 B200; GAE-scan HBM GB/s vs roofline"
E_PER_GPU, T, D, A, HIDDEN, EPOCHS, NMB = 4096, 128, 64, 8, (256, 256), 4, 16


def flops_per_env_step():
    """SURVEY.md 8d: MLP FLOPs (2MNK, biases ignored) per env step."""
    actor = 2 * (D * HIDDEN[0] + HIDDEN[0] * HIDDEN[1] + HIDDEN[1] * A)
    critic = 2 * (D * HIDDEN[0] + HIDDEN[0] * HIDDEN[1] + HIDDEN[1] * 1)
    rollout = actor + 2 * critic
    update = 3 * EPOCHS * (actor + critic)
    return rollout, update


def executed_update_flops_per_env_step():
    """What the update kernels actually execute per env step: forward + dW of every layer + dX of layers 1.. (the
    gradient w.r.t. the observations, dX of layer 0, is never formed), heads padded to the MMA N = 16."""
    def net(a_pad):
        fwd = 2 * (D * HIDDEN[0] + HIDDEN[0] * HIDDEN[1] + HIDDEN[1] * a_pad)
        dw = fwd
        dx = 2 * (HIDDEN[0] * HIDDEN[1] + HIDDEN[1] * a_pad)
        return fwd + dw + dx
    return EPOCHS * (net(16) + net(16))


def committed_k3_traffic():
    """dram__bytes_read + dram__bytes_write of the K3 launches of one minibatch step, from the newest committed ncu
    capture of this build (profiles/rNN_k3_traffic.json); None if there is none."""
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_k3_traffic.json")))
    if not files:
        return None, None
    d = json.load(open(files[-1]))
    return float(d["k3_bytes_per_minibatch_step"]), os.path.relpath(files[-1], ROOT)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.samples, self._stop = index, [], threading.Event()
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())
            if self._stop.is_set():
                break

    def stop(self):
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
def run_reference(args):
    """CPU arm: the reference's algorithm on the host cores (torch-CPU port, oracle/torch_cpu_ppo.py;
    the reference's own JAX/XLA CPU path is not installable here -- DESIGN.md).  Each "step" is the
    bounded sample of cpu_baseline_sample() (a few rollout steps + GAE + a few minibatch steps of the
    SAME workload, extrapolated to one update step) so K steps finish within minutes."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    samples = [cpu_baseline_sample(budget_s=18.0) for _ in range(steps)]
    value = statistics.median(s["value"] for s in samples)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env_steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": 0,
        "ms_per_step": T * E_PER_GPU / value * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args.gpus, "f32"),
        "cpu_baseline": {"value": value, "unit": "env_steps/s", "cores": samples[0]["cores"], "kind": "port", "sample": samples[0]["sample"]},
        "e2e": {"value": value, "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(n, precision):
    return {"workload": f"ff_ppo Anakin, synthetic Box obs_dim={D}, MLP{list(HIDDEN)}, num_envs={E_PER_GPU}/GPU, rollout_len={T}, actions={A}, epochs={EPOCHS}, minibatches={NMB}",
            "total_num_envs": E_PER_GPU * n, "parallelism": f"dp{n}", "precision": precision,
            "l2": "per-step working set (2x trajectory obs >= 128 MiB + activations) exceeds the 126 MB L2; no explicit flush"}


def _pick_threads():
    """Host threads for the CPU arm: the container may see more cores than it is allowed to use, so the
    count is calibrated on a short GEMM (all visible cores, 32 or 8 -- whichever is fastest)."""
    import torch

    visible = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best, best_t = 1, float("inf")
    a, b = torch.randn(4096, 256), torch.randn(256, 256)
    for n in sorted({visible, min(visible, 32), min(visible, 8)}, reverse=True):
        torch.set_num_threads(n)
        torch.mm(a, b)
        t0 = time.perf_counter()
        for _ in range(20):
            torch.mm(a, b)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_baseline_sample(budget_s=24.0):
    """Bounded CPU sample of the same workload (rank 0, N=1), about `budget_s` seconds of CPU work:
    as many of the T rollout steps as fit in a third of the budget (each step costs the same: three MLP
    applies on E rows + env + sampling), the GAE scan, and as many of the update's 64 minibatch steps as
    fit in the rest; each part is extrapolated linearly to one full update step."""
    import numpy as np
    import torch

    from oracle.torch_cpu_ppo import CpuAnakinPPO

    cores = _pick_threads()
    model = CpuAnakinPPO(E=E_PER_GPU, T=T, D=D, A=A, hidden=HIDDEN, epochs=EPOCHS, num_minibatches=NMB)
    # rollout: time a short rollout (T_s steps) and scale to T
    t_s = 2
    model.T = t_s
    model.rollout()  # warm-up
    t0 = time.perf_counter()
    model.rollout()
    per_step = (time.perf_counter() - t0) / t_s
    t_s = int(max(2, min(T, (budget_s / 3) / max(per_step, 1e-6))))
    model.T = t_s
    t0 = time.perf_counter()
    model.rollout()
    t_roll = (time.perf_counter() - t0) / t_s * T
    model.T = T
    g = torch.Generator().manual_seed(0)
    tr = {k: torch.randn(T, E_PER_GPU, generator=g) for k in ("value", "reward", "bootstrap", "log_prob")}
    tr["log_prob"] = -tr["log_prob"].abs() - 1.0
    tr["obs"] = torch.randn(T, E_PER_GPU, D, generator=g)
    tr["action"] = torch.randint(0, A, (T, E_PER_GPU), generator=g)
    tr["done"] = torch.rand(T, E_PER_GPU, generator=g) < 0.005
    tr["trunc"] = (~tr["done"]) & (torch.rand(T, E_PER_GPU, generator=g) < 0.002)
    t0 = time.perf_counter()
    model._adv = model.gae(tr["reward"], tr["value"], tr["bootstrap"], tr["done"], tr["trunc"], model.gamma, model.lam)
    t_gae = time.perf_counter() - t0
    B = T * E_PER_GPU
    mb = B // NMB
    perm = np.random.default_rng(0).permutation(B)
    _one_minibatch(model, tr, perm, 0, mb)  # warm-up
    done_mb = 0
    t0 = time.perf_counter()
    while done_mb < EPOCHS * NMB and (time.perf_counter() - t0) < budget_s / 2:
        _one_minibatch(model, tr, perm, (done_mb + 1) % NMB, mb)
        done_mb += 1
    t_mb = (time.perf_counter() - t0) / max(done_mb, 1)
    total = t_roll + t_gae + t_mb * EPOCHS * NMB
    return {"value": T * E_PER_GPU / total, "unit": "env_steps/s", "cores": cores, "kind": "port",
            "sample": f"torch-CPU fp32 port, {cores} threads: {t_s} of {T} rollout steps (-> {t_roll:.2f}s/rollout) + GAE ({t_gae:.3f}s) + "
                      f"{done_mb} of {EPOCHS * NMB} minibatch steps ({t_mb:.3f}s each), extrapolated to one update step ({total:.1f}s)"}


def _one_minibatch(model, tr, perm, i, mb):
    import torch

    B = model.T * model.E
    f = lambda x: x.reshape((B,) + x.shape[2:])
    idx = torch.as_tensor(perm[i * mb:(i + 1) * mb], dtype=torch.long)
    adv, tgt = model._adv
    from oracle.torch_cpu_ppo import mlp

    x = f(tr["obs"])[idx]
    ap = [p.detach().requires_grad_(True) for p in model.actor]
    lp_all = torch.log_softmax(mlp(ap, x), -1)
    logp = lp_all.gather(1, f(tr["action"])[idx][:, None])[:, 0]
    ratio = torch.exp(logp - f(tr["log_prob"])[idx])
    a = f(adv)[idx]
    loss = -torch.minimum(ratio * a, torch.clamp(ratio, 0.8, 1.2) * a).mean() - 0.01 * (-(lp_all.exp() * lp_all).sum(-1).mean())
    ag = torch.autograd.grad(loss, ap)
    cp = [p.detach().requires_grad_(True) for p in model.critic]
    v = mlp(cp, x)[:, 0]
    vo, tg = f(tr["value"])[idx], f(tgt)[idx]
    vclip = vo + (v - vo).clamp(-0.2, 0.2)
    cg = torch.autograd.grad(0.5 * 0.5 * torch.maximum((v - tg) ** 2, (vclip - tg) ** 2).mean(), cp)
    model.count += 1
    model._apply(model.actor, ag, 3e-4, model.count)
    model._apply(model.critic, cg, 3e-4, model.count)


# ----------------------------------------------------------------------------------------------------
def output_arrays(out):
    """What one learn() call hands its caller (AnakinExperimentOutput), as float32 / float64 host arrays: the parameters
    and Adam state of the learner state, the observation the next call starts from, and the episode / train metrics.
    About 9 MB at the bench shape, so nothing needs sampling."""
    import torch

    ls = out.learner_state
    host = lambda t, dt=torch.float32: t.detach().to("cpu", dt).numpy()
    arrays = {"actor_params": host(ls.params.actor_params.flat), "critic_params": host(ls.params.critic_params.flat)}
    for side, st in (("actor", ls.opt_states.actor_opt_state), ("critic", ls.opt_states.critic_opt_state)):
        arrays[f"{side}_adam_mu"], arrays[f"{side}_adam_nu"] = host(st.mu), host(st.nu)
        arrays[f"{side}_adam_count"], arrays[f"{side}_schedule_count"] = host(st.count, torch.float64), host(st.sched_count, torch.float64)
    for u, ts in enumerate(ls.timestep):
        arrays[f"next_observation_shard{u}"] = host(ts.observation)
    for name, t in out.episode_metrics.items():
        arrays[name] = host(t)
    for name, t in out.train_metrics.items():
        arrays[f"train_{name}"] = host(t)
    return arrays


def dump_outputs(arrays, directory):
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes exceed the 64 MiB budget"
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def run_ours(args):
    # Libraries (NCCL prints its version banner on stdout) must not pollute the ONE JSON line: everything
    # written to fd 1 during the run goes to stderr; the JSON line is written to the real stdout at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the stoix_b200 kernels have no CPU fallback")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"

    from stoix_b200 import _lib, ops, random as srandom
    from stoix_b200.config import compose
    from stoix_b200.systems.ppo.anakin import ff_ppo
    from stoix_b200.utils import make_env
    from stoix_b200.utils.total_timestep_checker import check_total_timesteps

    lib = _lib.load()
    precision = args.precision
    total_updates = args.steps * 2 + args.warmup + 8
    cfg = compose("default_ff_ppo", [
        "env=synthetic/box", f"env.kwargs.obs_dim={D}", f"env.kwargs.num_actions={A}",
        f"arch.total_num_envs={E_PER_GPU * world}", f"system.rollout_length={T}", f"system.epochs={EPOCHS}",
        f"system.num_minibatches={NMB}", f"arch.total_timesteps={E_PER_GPU * world * T * total_updates}",
        "arch.num_evaluation=1", f"arch.precision={precision}", "logger.use_console=False",
        f"arch.fused_allreduce={not args.nccl_allreduce}",
    ])
    cfg.num_devices, cfg.rank = world, rank
    cfg = check_total_timesteps(cfg, quiet=True)
    env, _ = make_env.make(cfg)
    keys = srandom.split(srandom.PRNGKey(cfg.arch.seed), 4)
    learn, _, state = ff_ppo.learner_setup(env, (keys[0], keys[2], keys[3]), cfg)
    cfg.arch.num_updates_per_eval = 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def progress(msg):
        if os.environ.get("STX_BENCH_VERBOSE"):
            print(f"[bench r{rank} {time.time() % 1000:.1f}] {msg}", file=sys.stderr, flush=True)

    # ---- warm-up (first update eager: module load / NCCL init; second captures the CUDA graph) ----
    progress("setup done")
    l0 = lib.stx_launch_count()
    state = learn(state).learner_state
    torch.cuda.synchronize()
    launches_per_update = lib.stx_launch_count() - l0
    progress("eager update done")
    for _ in range(max(args.warmup, 3)):
        state = learn(state).learner_state
    barrier()
    progress("warm-up done")

    # ---- timed region A: device-resident (value) ----
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        state = learn(state).learner_state
    ev1.record()
    barrier()
    dt = ev0.elapsed_time(ev1) * 1e-3
    progress(f"timed region A done {dt:.3f}s")

    # ---- timed region B: end to end through the public API with host buffers (e2e) ----
    sh = learn.built["shards"][0]
    host_obs = torch.empty(sh.obs[T].shape, dtype=sh.obs.dtype).pin_memory()
    host_obs.copy_(sh.obs[T])
    host_train = torch.empty(EPOCHS, NMB, len(ff_ppo._METRIC_NAMES), dtype=torch.float32).pin_memory()
    host_ret = torch.empty(T, E_PER_GPU, dtype=torch.float32).pin_memory()
    host_term = torch.empty(T, E_PER_GPU, dtype=torch.bool).pin_memory()
    h2d = host_obs.numel() * host_obs.element_size()
    d2h = host_train.numel() * 4 + host_ret.numel() * 4 + host_term.numel() + h2d  # + the carried observation
    barrier()
    # an event after every step (the stream is idle there, waiting for the host) gives the spread over the K steps
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    evs[0].record()
    for ev in evs[1:]:
        sh.obs[T].copy_(host_obs, non_blocking=True)      # H2D: the step's input observations (pinned)
        out = learn(state)
        state = out.learner_state
        host_train.copy_(torch.stack([out.train_metrics[n][0] for n in ff_ppo._METRIC_NAMES], -1), non_blocking=True)
        host_ret.copy_(out.episode_metrics["episode_return"][0, 0], non_blocking=True)
        host_term.copy_(out.episode_metrics["is_terminal_step"][0, 0], non_blocking=True)
        torch.cuda.current_stream().synchronize()         # the host consumes the step's result
        host_obs.copy_(sh.obs[T])                         # D2H: the observation the next step starts from
        ev.record()
    barrier()
    dt_e2e = evs[0].elapsed_time(evs[-1]) * 1e-3
    step_ms = [a.elapsed_time(b) for a, b in zip(evs, evs[1:])]
    clocks = sampler.stop()
    progress("timed region B done")
    if args.dump_outputs and rank == 0:  # before the phase replays below move the learner state on
        dump_outputs(output_arrays(out), args.dump_outputs)

    # ---- max over ranks ----
    times = torch.tensor([dt, dt_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dt, dt_e2e = times.tolist()

    # ---- phase breakdown (rank 0, one CUDA graph per phase, events around each replay) ----
    peaks = load_peaks()
    phase_ms = {}
    roofline = gae_roof = None
    if True:  # every rank replays the phases (the update phase holds the all-reduce); rank 0 reports
        phases = learn.phases
        for name in ("rollout", "gae", "update"):
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                phases[name](state)
            ts = []
            for _ in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                if name == "gae":  # the GAE inputs (11.5 MB) would sit in L2: flush so HBM is what is measured
                    ops._zeros_scratch(("flush",), 256 << 20, torch.device("cuda", local)).fill_(1)
                a.record()
                g.replay()
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            phase_ms[name] = statistics.median(ts)
            progress(f"phase {name} done")
        roll_f, upd_f = flops_per_env_step()
        upd_exec = executed_update_flops_per_env_step()
        upd_tflops = upd_f * T * E_PER_GPU / (phase_ms["update"] * 1e-3) / 1e12
        # the timed region is a sub-second burst at (or near) the maximum SM clock with no power cap: the BURST cuBLAS
        # figure is the honest denominator; the sustained one (seconds under the 1 kW cap) is given beside it
        burst = (dt < 1.0) and not (set(clocks.get("reasons", [])) & {"sw_power_cap"})
        peak = peaks["bf16_tflops"] if burst else peaks["bf16_tflops_sustained"]
        traffic, traffic_src = committed_k3_traffic() if precision == "bf16" else (None, None)
        roofline = {"kernel": "K3 PPO minibatch forward/loss/backward (+K4 clip/Adam), 64 minibatch steps",
                    "bound": "tensor", "achieved": upd_tflops, "peak": peak, "unit": "TFLOP/s", "frac": upd_tflops / peak,
                    "frac_of_sustained_peak": upd_tflops / peaks["bf16_tflops_sustained"],
                    "frac_of_burst_peak": upd_tflops / peaks["bf16_tflops"],
                    "traffic": traffic, "traffic_unit": "dram bytes per minibatch step (K3a+K3b)", "traffic_source": traffic_src,
                    "peak_source": f"{peaks['source']} ({'burst' if burst else 'sustained'} bf16 cuBLAS)",
                    "flops_per_env_step": upd_f, "flops_per_env_step_executed": upd_exec,
                    "achieved_executed": upd_exec * T * E_PER_GPU / (phase_ms["update"] * 1e-3) / 1e12}
        gae_gbs = 22.0 * T * E_PER_GPU / (phase_ms["gae"] * 1e-3) / 1e9
        gae_roof = {"kernel": "K2 gae_scan_kernel", "bound": "hbm", "shape": [T, E_PER_GPU], "achieved": gae_gbs, "peak": peaks["hbm_gbs"],
                    "unit": "GB/s", "frac": gae_gbs / peaks["hbm_gbs"], "bytes_per_element": 22, "us": phase_ms["gae"] * 1e3,
                    "note": "named shape is launch/latency-bound (11.5 MB); `saturating` is the same kernel entry at (128, 1048576)"}
        if world == 1:   # BASELINE's second metric (GAE-scan HBM GB/s vs roofline) at a shape that can saturate HBM: 2.95 GB per launch
            try:
                Tg, Eg = 128, 1 << 20
                gg = torch.Generator(device="cuda").manual_seed(0)
                rr, vv, bb = (torch.randn(Tg, Eg, device="cuda", generator=gg) for _ in range(3))
                dd = torch.rand(Tg, Eg, device="cuda", generator=gg) < 0.005
                tt = (~dd) & (torch.rand(Tg, Eg, device="cuda", generator=gg) < 0.002)
                oa, ot = torch.empty_like(rr), torch.empty_like(rr)
                for _ in range(3):
                    ops.gae_ppo(rr, vv, bb, dd, tt, 0.99, 0.95, 1.0, 1, out=(oa, ot))
                ts = []
                reps = 5             # launches per event pair: behind the first one the queue is never empty, so the pair times the
                for _ in range(7):   # GPU, not the Python call; inputs (1.9 GB) + outputs (1.1 GB) >> 126 MB L2: no flush needed
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for _ in range(reps):
                        ops.gae_ppo(rr, vv, bb, dd, tt, 0.99, 0.95, 1.0, 1, out=(oa, ot))
                    b.record()
                    torch.cuda.synchronize()
                    ts.append(a.elapsed_time(b) / reps)
                us = statistics.median(ts) * 1e3
                sat = 22.0 * Tg * Eg / (us * 1e-6) / 1e9
                gae_roof["saturating"] = {"kernel": "K2 gae_tma_kernel<64,64>", "shape": [Tg, Eg], "achieved": sat, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                          "frac": sat / peaks["hbm_gbs"], "us": us, "bytes_per_launch": 22 * Tg * Eg}
                del rr, vv, bb, dd, tt, oa, ot
            except Exception as e:  # never lose the headline line over the side measurement
                gae_roof["saturating"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        value = world * T * E_PER_GPU * args.steps / dt
        e2e = world * T * E_PER_GPU * args.steps / dt_e2e
        line = {
            "metric": METRIC, "value": value, "unit": "env_steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic", "config": workload_config(world, precision),
            "e2e": {"value": e2e, "unit": "env_steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": dt_e2e / args.steps * 1e3,
                    "ms_per_step_spread": {"steps": len(step_ms), "median": statistics.median(step_ms), "min": min(step_ms),
                                           "max": max(step_ms)}},
            "gpu_launches": int(launches_per_update * args.steps), "launches_per_step": int(launches_per_update),
            "allreduce": ("none" if world == 1 else ("fused NVLink one-shot all-reduce inside the optimiser kernel" if learn.built.get("peers_obj") is not None else "NCCL all-reduce")),
            "clocks": clocks, "roofline": roofline, "gae_roofline": gae_roof, "phase_ms": phase_ms,
            "tensor_roofline_env_steps_per_s_per_gpu": peaks["bf16_tflops_sustained"] * 1e12 / sum(flops_per_env_step()),
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_sample()
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    sys.stdout.flush()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        # NCCL/TCPStore teardown can hang at interpreter exit in this container (observed: workers print their
        # last line and never return to torchrun), so leave without running the destructors.
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("STX_BENCH_PRECISION", "bf16"), choices=["f32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nccl-allreduce", action="store_true", help="N>1: NCCL all-reduce + K4 instead of the fused NVLink all-reduce/optimiser kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
