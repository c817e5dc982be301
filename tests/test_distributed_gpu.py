"""Data-parallel update (the reference's pmap 'device' axis, ff_ppo.py:253-261 -> one process per GPU, mean of ONE flat
gradient arena per minibatch step) on the GPU, checked against the ORACLE:

* `test_fused_allreduce_kernel_on_one_device` (runs on a 1-GPU box): the fused all-reduce + clip + Adam kernel, two-shot
  (`stx_allreduce2_clip_adam_step`, the default) and one-shot (`stx_allreduce_clip_adam_step`), driven through the C ABI with
  W = 2 / 4 / 8 "virtual ranks" whose gradient arenas and signal pads are plain buffers of the same device; every virtual rank's parameters / moments must equal
  `oracle.clip_adam_step(mean of the W gradients)` and be bit-identical to each other.
* `test_two_rank_update_matches_oracle` (needs >= 2 GPUs): two torchrun ranks run three whole update
  steps (eager, graph capture, graph replay); each rank replays its own trajectory through `oracle.ppo_update` with the
  gradient exchange as `grad_sync` (a gloo all-reduce between the two oracle instances: SUM, then 1/world) and compares its
  post-update optimiser state and parameters with the oracle's, for the fused NVLink all-reduce and for NCCL.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

WORKER = r'''
import os, sys, json
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, os.getcwd())
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
cpu_group = dist.new_group(backend="gloo")       # carries the ORACLE's gradient exchange (CPU tensors)
from oracle import ppo_oracle as O
from stoix_b200 import ops, random as srandom
from stoix_b200.config import compose
from stoix_b200.systems.ppo.anakin import ff_ppo
from stoix_b200.utils import make_env
from stoix_b200.utils.total_timestep_checker import check_total_timesteps
precision, fused = sys.argv[1], sys.argv[2]
bf16 = precision == "bf16"
E, T, nmb, n_upd = 256, 16, 4, 3
cfg = compose("default_ff_ppo", ["env=synthetic/box", f"arch.total_num_envs={E * world}", f"system.rollout_length={T}",
                                 f"system.num_minibatches={nmb}", f"arch.total_timesteps={E * world * T * n_upd}", "arch.num_evaluation=1",
                                 f"arch.precision={precision}", f"arch.fused_allreduce={fused}", "logger.use_console=False",
                                 "env.kwargs.p_term=0.05", "env.kwargs.p_trunc=0.05"] + os.environ.get("STX_TEST_EXTRA", "").split())
cfg.num_devices, cfg.rank = world, rank
cfg = check_total_timesteps(cfg, quiet=True)
assert cfg.arch.num_envs == E and cfg.arch.num_updates == n_upd
env, _ = make_env.make(cfg)
keys = srandom.split(srandom.PRNGKey(cfg.arch.seed), 4)
learn, _, state = ff_ppo.learner_setup(env, (keys[0], keys[2], keys[3]), cfg)
with torch.no_grad():   # non-trivial biases / heads, identical on every rank
    g = torch.Generator(device="cuda").manual_seed(1)
    arena = state.params.actor_params.arena
    arena.add_(torch.randn(arena.shape, device="cuda", generator=g) * float(os.environ.get("STX_TEST_PERTURB", "0.05")))
    if bf16:
        ops.cast_bf16(arena, out=state.params.actor_params.arena_bf16)
cfg.arch.num_updates_per_eval = 1
f64 = lambda t: t.detach().float().cpu().numpy().astype(np.float64)
tree = lambda tr: O.MLPParams.from_flat(f64(tr.flat), list(tr.spec.sizes))
actor, critic = tree(state.params.actor_params), tree(state.params.critic_params)
n_a, n_c = actor.flat().size, critic.flat().size
a_st, c_st = O.AdamState(np.zeros(n_a), np.zeros(n_a)), O.AdamState(np.zeros(n_c), np.zeros(n_c))
h = O.PPOHyper(num_minibatches=nmb, num_updates=n_upd)
rel = lambda a, b: float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))

def grad_sync(a_g, c_g, info):   # pmean over "device": all-reduce SUM of one flat arena, 1/world in the optimiser
    flat = torch.from_numpy(np.concatenate([a_g, c_g]).astype(np.float64))
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=cpu_group)
    flat = flat.numpy() * (1.0 / world)
    m = torch.tensor([info["actor_loss"], info["entropy"], info["value_loss"]], dtype=torch.float64)
    dist.all_reduce(m, op=dist.ReduceOp.SUM, group=cpu_group)
    m = m.numpy() / world
    return flat[: a_g.size], flat[a_g.size:], {**info, "actor_loss": m[0], "entropy": m[1], "value_loss": m[2]}

worst = {"params_abs": 0.0, "moments_rel": 0.0, "metrics_rel": 0.0}
per_update = []
ok, why = True, ""
for upd in range(n_upd):   # eager, graph capture, graph replay
    out = learn(state); state = out.learner_state
    torch.cuda.synchronize()
    sh = learn.built["shards"][0]
    traj = O.Trajectory(obs=f64(sh.obs[:T]), action=sh.action.cpu().numpy(), reward=f64(sh.reward),
                        done=sh.done.cpu().numpy().astype(bool), truncated=sh.truncated.cpu().numpy().astype(bool), next_obs=f64(sh.next_obs))
    O.evaluate_rollout(actor, critic, traj, bf16=bf16)
    if bf16:
        traj.value, traj.bootstrap_value, traj.log_prob = f64(sh.value), f64(sh.bootstrap_value), f64(sh.log_prob)
    perms = np.stack([ops.make_permutation(T * E, state.key[1], ep + 4 * upd, device="cuda").cpu().numpy() for ep in range(4)])
    actor, critic, metrics, _, _ = O.ppo_update(actor, critic, a_st, c_st, traj, perms, h, grad_sync=grad_sync, bf16=bf16)
    a_tree, c_tree = state.params.actor_params, state.params.critic_params
    _, coff, _ = ops.arena_offsets(a_tree.spec, c_tree.spec)
    mu, nu = f64(a_tree.arena_mu), f64(a_tree.arena_nu)
    mom = max(rel(mu[:n_a], a_st.mu), rel(nu[:n_a], a_st.nu), rel(mu[coff:coff + n_c], c_st.mu), rel(nu[coff:coff + n_c], c_st.nu))
    worst["moments_rel"] = max(worst["moments_rel"], mom)
    per_update.append({"mu_a": rel(mu[:n_a], a_st.mu), "nu_a": rel(nu[:n_a], a_st.nu), "mu_c": rel(mu[coff:coff + n_c], c_st.mu),
                       "nu_c": rel(nu[coff:coff + n_c], c_st.nu), "p_a": float(np.abs(f64(a_tree.flat) - actor.flat()).max()),
                       "p_c": float(np.abs(f64(c_tree.flat) - critic.flat()).max())})
    pa, pc = f64(a_tree.flat), f64(c_tree.flat)
    worst["params_abs"] = max(worst["params_abs"], float(np.abs(pa - actor.flat()).max()), float(np.abs(pc - critic.flat()).max()))
    for name in ("actor_loss", "entropy", "value_loss"):
        got, ref = f64(out.train_metrics[name][0]), metrics[name]
        worst["metrics_rel"] = max(worst["metrics_rel"], float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-6)))
    pu = per_update[-1]
    mu_err, nu_err, p_err = max(pu["mu_a"], pu["mu_c"]), max(pu["nu_a"], pu["nu_c"]), max(pu["p_a"], pu["p_c"])
    # Every update is checked on its own: afterwards the oracle continues from the kernels' parameters and moments.  Bounds:
    #  bf16 (tcgen05 path vs the bf16-rounding oracle): the end-state bounds of the single-device whole-update test
    #       (tests/test_tc_gpu.py: mu 0.3, nu 0.1, params 0.15 -- trajectory drift under Adam normalisation; the strict check
    #       of that path is the per-step teacher-forced gradient test there, 5e-3);
    #  f32  (CUDA-core path vs the fp64 oracle): per-step gradients agree to 3e-7 (scripts/diag_bf16_steps.py ... f32), but over
    #       the 16 optimiser steps of an update single updates show moment differences up to ~1e-2 (seen: 7e-3 at N=2,
    #       4e-4 at N=1, most updates 1e-6; identical eager / captured, NCCL / fused): parameters within a third of one Adam
    #       step (lr = 3e-4) and moments within 2e-2.
    lim = (0.3, 0.1, 0.15) if bf16 else (2e-2, 2e-2, 1e-4)
    if mu_err > lim[0] or nu_err > lim[1] or p_err > lim[2]:
        ok, why = False, f"update {upd}: mu {mu_err:.3e} nu {nu_err:.3e} params {p_err:.3e} (limits {lim})"
    actor, critic = tree(a_tree), tree(c_tree)
    a_st.mu, a_st.nu, c_st.mu, c_st.nu = mu[:n_a].copy(), nu[:n_a].copy(), mu[coff:coff + n_c].copy(), nu[coff:coff + n_c].copy()
arena = state.params.actor_params.arena
gathered = [torch.empty_like(arena) for _ in range(world)]
dist.all_gather(gathered, arena)
obs_sum = learn.built["shards"][0].obs[:T].float().sum()
sums = [torch.empty_like(obs_sum) for _ in range(world)]
dist.all_gather(sums, obs_sum)
flags = torch.tensor([1.0 if ok else 0.0], device="cuda")
dist.all_reduce(flags, op=dist.ReduceOp.MIN)
if rank == 0:
    print(json.dumps({"oracle_ok_all_ranks": bool(flags.item() == 1.0), "why": why, **worst, "per_update": per_update,
                      "params_identical_across_ranks": all(torch.equal(gathered[0], g) for g in gathered),
                      "shards_differ": len({float(s) for s in sums}) == world, "fused_used": learn.built["peers_obj"] is not None,
                      "counts": state.params.actor_params.arena_counts.cpu().tolist()}))
dist.barrier(); torch.cuda.synchronize(); sys.stdout.flush(); os._exit(0)  # NCCL teardown can hang at exit here
'''


@pytest.mark.parametrize("precision,fused", [("f32", "False"), ("bf16", "False"), ("bf16", "True"), ("f32", "True")])
def test_two_rank_update_matches_oracle(precision, fused, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("NEEDS 2 GPUs (NCCL refuses two ranks on one device): run `python -m pytest tests/test_distributed_gpu.py -m gpu` "
                    "on a machine with two; the fused all-reduce kernel itself is covered on one device by "
                    "test_fused_allreduce_kernel_on_one_device")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29511", str(script), precision, fused]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    print(res)
    assert res["oracle_ok_all_ranks"], res
    assert res["params_identical_across_ranks"] and res["shards_differ"], res
    assert res["fused_used"] == (fused == "True"), res
    assert res["counts"] == [3 * 4 * 4] * 4, res


@pytest.mark.parametrize("mode", [2, 1])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_fused_allreduce_kernel_on_one_device(world, mode):
    """The fused all-reduce + clip + Adam kernel with `world` virtual ranks on ONE device, both forms.  Each virtual rank owns a
    gradient arena, a reduced-gradient buffer, a signal pad, parameters, moments, counters and scratch.
    mode 1 (`stx_allreduce_clip_adam_step`, one-shot): the kernels run one after the other, so before virtual rank r's launch
      the test itself writes the announcements of the ranks that have not run yet into r's pad (their gradients ARE complete).
    mode 2 (`stx_allreduce2_clip_adam_step`, two-shot, the learner's default): every rank needs every other rank's slice, so the
      W kernels run CONCURRENTLY, one stream each, with a small grid (8 blocks) so that all of them are co-resident.
    Three calls, so that the generation counter, bias correction and LR schedule advance."""
    from oracle import ppo_oracle as O
    from stoix_b200 import _lib, ops

    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(world)
    sa, sc = ops.MlpSpec((12, 32, 32, 5)), ops.MlpSpec((12, 32, 32, 1))
    _, coff, total = ops.arena_offsets(sa, sc)
    n_a, n_c = sa.param_count, sc.param_count
    p0 = np.zeros(total, np.float32)
    p0[:n_a] = rng.standard_normal(n_a) * 0.3
    p0[coff:coff + n_c] = rng.standard_normal(n_c) * 0.3
    segs = [(0, n_a, 3e-3, 0.5), (coff, n_c, 1e-3, 0.05)]  # the critic optimiser clips
    lib = _lib.load()
    slot, pad_words = 16, 64
    ranks = []
    for r in range(world):
        ranks.append(dict(
            params=torch.tensor(p0, device=dev), mu=torch.zeros(total, device=dev), nu=torch.zeros(total, device=dev),
            grads=torch.zeros(total, device=dev), gsum=torch.zeros(total + 128, device=dev), pad=torch.zeros(pad_words, dtype=torch.int32, device=dev),
            plan=ops.AdamPlan(segs, dev, decay=True, steps_per_update=2, num_updates=4), stream=torch.cuda.Stream(device=dev)))
    grad_ptrs = (C.c_void_p * world)(*[rk["grads"].data_ptr() for rk in ranks])
    gsum_ptrs = (C.c_void_p * world)(*[rk["gsum"].data_ptr() for rk in ranks])
    pad_ptrs = (C.c_void_p * world)(*[rk["pad"].data_ptr() for rk in ranks])
    ref_p = [p0[:n_a].astype(np.float64), p0[coff:coff + n_c].astype(np.float64)]
    ref_st = [O.AdamState(np.zeros(n_a), np.zeros(n_a)), O.AdamState(np.zeros(n_c), np.zeros(n_c))]
    P = lambda t: C.c_void_p(t.data_ptr())
    for call in range(1, 4):
        g_np = [np.zeros(total, np.float32) for _ in range(world)]
        for r in range(world):
            g_np[r][:n_a] = rng.standard_normal(n_a) * 0.05
            g_np[r][coff:coff + n_c] = rng.standard_normal(n_c) * (0.5 if r == 0 else 0.05)
            ranks[r]["grads"].copy_(torch.tensor(g_np[r]))
        torch.cuda.synchronize()
        for r in range(world):
            rk = ranks[r]
            rk["plan"].hyper.grad_scale = 1.0 / world
            rk["plan"].hyper.prenorm = 0
            if mode == 1:
                rk["pad"][slot:slot + world] = call  # the virtual ranks that run later have (logically) announced already
                rc = lib.stx_allreduce_clip_adam_step(P(rk["params"]), grad_ptrs, pad_ptrs, world, r, slot, P(rk["gsum"]), P(rk["mu"]), P(rk["nu"]),
                                                      P(rk["plan"].counts), P(rk["plan"].segs), rk["plan"].nseg, C.byref(rk["plan"].hyper), None,
                                                      P(rk["plan"].gnorm), P(rk["plan"].scratch), C.c_void_p(torch.cuda.current_stream().cuda_stream))
                _lib.check(rc, "stx_allreduce_clip_adam_step")
                torch.cuda.synchronize()
            else:
                rc = lib.stx_allreduce2_clip_adam_step(P(rk["params"]), grad_ptrs, gsum_ptrs, total, pad_ptrs, world, r, slot, P(rk["mu"]), P(rk["nu"]),
                                                       P(rk["plan"].counts), P(rk["plan"].segs), rk["plan"].nseg, C.byref(rk["plan"].hyper), None,
                                                       P(rk["plan"].gnorm), P(rk["plan"].scratch), 8, C.c_void_p(rk["stream"].cuda_stream))
                _lib.check(rc, "stx_allreduce2_clip_adam_step")
        torch.cuda.synchronize()
        for r in range(world):
            assert int(ranks[r]["pad"][slot + r].item()) == call  # its own announcement arrived in its own pad too
            if mode == 2:
                assert ranks[r]["pad"][slot + 8:slot + 8 + world].cpu().tolist() == [call] * world
        mean = np.mean(np.stack([g.astype(np.float64) for g in g_np]), axis=0)
        for s, (off, cnt, lr, mgn) in enumerate(segs):
            k = ref_st[s].sched_count // 2
            ref_p[s], gnorm = O.clip_adam_step(ref_p[s], mean[off:off + cnt], ref_st[s], lr * (1.0 - k / 4), mgn)
            for r in range(world):
                rk = ranks[r]
                np.testing.assert_allclose(rk["params"][off:off + cnt].cpu().numpy(), ref_p[s], rtol=2e-5, atol=2e-7)
                np.testing.assert_allclose(rk["mu"][off:off + cnt].cpu().numpy(), ref_st[s].mu, rtol=2e-5, atol=1e-9)
                np.testing.assert_allclose(rk["nu"][off:off + cnt].cpu().numpy(), ref_st[s].nu, rtol=2e-5, atol=1e-12)
                np.testing.assert_allclose(float(rk["plan"].gnorm[s].item()), gnorm, rtol=1e-5)
        for r in range(1, world):  # identical association order on every rank => bit-identical replicas
            for k in ("params", "mu", "nu", "gsum"):
                assert torch.equal(ranks[0][k], ranks[r][k]), f"virtual rank {r}: {k} differs from rank 0 after call {call}"
        assert ranks[0]["plan"].counts.cpu().tolist() == [call] * 4


NEXT_ROW_WORKER = r'''
import os, sys, json
import torch, torch.distributed as dist
sys.path.insert(0, os.getcwd())
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
from stoix_b200 import random as srandom
from stoix_b200.config import compose
from stoix_b200.utils import make_env
from stoix_b200.utils.total_timestep_checker import check_total_timesteps
system = sys.argv[1]
if system == "rec_ppo":
    from stoix_b200.systems.ppo.anakin import rec_ppo as S
    cfg = compose("default_rec_ppo", ["env=synthetic/box", "env.kwargs.obs_dim=12", "env.kwargs.num_actions=5", f"arch.total_num_envs={64 * world}",
                                      "system.rollout_length=16", "system.num_minibatches=4", "system.epochs=2", f"arch.total_timesteps={64 * world * 16 * 3}",
                                      "arch.num_evaluation=1", "logger.use_console=False", "network.actor_network.rnn_layer.cell_type=lstm",
                                      "network.critic_network.rnn_layer.cell_type=lstm"], config_dir="default/anakin")
else:
    from stoix_b200.systems.sac import ff_sac as S
    cfg = compose("default_ff_sac", [f"arch.total_num_envs={64 * world}", f"system.total_batch_size={128 * world}", f"system.total_buffer_size={4096 * world}",
                                     "system.warmup_steps=4", f"arch.total_timesteps={64 * world * 30}", "arch.num_evaluation=1", "logger.use_console=False",
                                     "network.actor_network.pre_torso.layer_sizes=[64,64]", "network.q_network.pre_torso.layer_sizes=[64,64]"],
                  config_dir="default/anakin")
cfg.num_devices, cfg.rank = world, rank
cfg = check_total_timesteps(cfg, quiet=True)
env, _ = make_env.make(cfg)
learn, _, state = S.learner_setup(env, tuple(srandom.split(srandom.PRNGKey(cfg.arch.seed), 3)), cfg)
arena0 = state.params.actor_params.arena.clone()
out = learn(state)
torch.cuda.synchronize()
arena = out.learner_state.params.actor_params.arena
gathered = [torch.empty_like(arena) for _ in range(world)]
dist.all_gather(gathered, arena)
sh = learn.built["shards"][0]
sig = sh.reward.float().sum()
sigs = [torch.empty_like(sig) for _ in range(world)]
dist.all_gather(sigs, sig)
if rank == 0:
    print(json.dumps({"identical": all(torch.equal(gathered[0], g) for g in gathered), "moved": bool((arena - arena0).abs().max() > 0),
                      "finite": bool(torch.isfinite(arena).all()), "shards_differ": len({float(s) for s in sigs}) == world}))
dist.barrier(); torch.cuda.synchronize(); sys.stdout.flush(); os._exit(0)
'''


@pytest.mark.parametrize("system", ["rec_ppo", "ff_sac"])
def test_two_rank_next_row_systems_stay_in_lockstep(system, tmp_path):
    """The data-parallel path of the recurrent PPO (LSTM) and SAC learners on two real ranks: rank-local rollouts / replay rings, NCCL
    all-reduce of the flat gradient arena, 1/world inside the optimiser kernel -> bit-identical replicas that moved and stayed finite."""
    if torch.cuda.device_count() < 2:
        pytest.skip("NEEDS 2 GPUs: run `python -m pytest tests/test_distributed_gpu.py -m gpu` on a machine with two")
    script = tmp_path / "worker.py"
    script.write_text(NEXT_ROW_WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", "29513",
           str(script), system]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert res == {"identical": True, "moved": True, "finite": True, "shards_differ": True}, res
