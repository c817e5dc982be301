"""Sebulba ff_ppo (SURVEY.md 8f row 1, MLP torso) on the GPU.

* inference server (pinned host obs -> side stream -> forward + sampling kernels -> pinned actions) vs the oracle;
* learner step (hstack of actor shards, GAE through the `values=` interface, epochs x minibatches) vs oracle.ppo_update on
  the equivalent trajectory (value = values[:-1], bootstrap_value = values[1:], no truncation:
  stoix/systems/ppo/sebulba/ff_ppo.py:394-411, 516-519);
* a whole threaded run (2 actor threads + learner + async evaluator on CPU environments)."""
import numpy as np
import pytest
import torch

from oracle import ppo_oracle as O

pytestmark = pytest.mark.gpu


def _cfg(extra=()):
    from stoix_b200.config import compose
    from stoix_b200.utils.total_timestep_checker import check_total_timesteps

    c = compose("default_ff_ppo", ["arch.total_num_envs=256", "system.rollout_length=8", "system.num_minibatches=2",
                                   "arch.total_timesteps=40960", "arch.actor.actor_per_device=2", "arch.num_evaluation=2",
                                   "arch.num_eval_episodes=8", "logger.use_console=False", "env.kwargs.p_term=0.05",
                                   "env.kwargs.p_trunc=0.05"] + list(extra), config_dir="default/sebulba")
    c.num_actor_devices, c.num_learner_devices, c.arch.world_size = 1, 1, 1
    c.arch.total_num_actor_threads = 2
    return check_total_timesteps(c, quiet=True)


def _setup(cfg):
    from stoix_b200 import random as srandom
    from stoix_b200.envs import cpu as cpu_envs
    from stoix_b200.systems.ppo.sebulba import ff_ppo as seb

    torch.cuda.set_device(0)
    factory = cpu_envs.make_factory(cfg)
    keys = srandom.split(srandom.PRNGKey(cfg.arch.seed), 4)
    learn_step, apply_fns, state = seb.learner_setup(factory, (keys[0], keys[2], keys[3]), [torch.device("cuda", 0)], cfg)
    with torch.no_grad():   # non-trivial biases / heads
        g = torch.Generator(device="cuda").manual_seed(1)
        arena = state.params.actor_params.arena
        arena.add_(torch.randn(arena.shape, device="cuda", generator=g) * 0.05)
        if state.params.actor_params.arena_bf16 is not None:
            from stoix_b200 import ops

            ops.cast_bf16(arena, out=state.params.actor_params.arena_bf16)
    return seb, factory, learn_step, apply_fns, state


f64 = lambda t: t.detach().float().cpu().numpy().astype(np.float64)
tree = lambda tr: O.MLPParams.from_flat(f64(tr.flat), list(tr.spec.sizes))


@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_inference_server_matches_oracle(precision):
    from stoix_b200 import ops
    from stoix_b200.utils.sebulba_utils import ParamSnapshot

    cfg = _cfg([f"arch.precision={precision}"])
    seb, factory, _, apply_fns, state = _setup(cfg)
    a_tree, c_tree = state.params.actor_params, state.params.critic_params
    E, T = 128, 8
    server = seb.InferenceServer((a_tree.spec, c_tree.spec), torch.device("cuda", 0), E, T, seb._precision(cfg), seed=123, thread_id=0)
    snap = ParamSnapshot(a_tree.arena, a_tree.arena_bf16, None, 0)
    rng = np.random.default_rng(0)
    actor, critic = tree(a_tree), tree(c_tree)
    for slot in range(3):
        obs = rng.standard_normal((E, 64)).astype(np.float32)
        action = server.act(snap, obs, slot).copy()
        assert action.dtype == np.int32 and action.shape == (E,) and action.min() >= 0 and action.max() < 8
        np.testing.assert_array_equal(action, server.action[slot].cpu().numpy())
        bf16 = precision == "bf16"
        stored = f64(server.obs[slot])
        np.testing.assert_allclose(stored, obs, rtol=2 ** -8 if bf16 else 0, atol=0)
        logits, _ = O.mlp_forward(actor, stored, bf16)
        v, _ = O.mlp_forward(critic, stored, bf16)
        tol = dict(rtol=2e-3, atol=2e-2) if bf16 else dict(rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(f64(server.log_prob[slot]), O.categorical_log_prob(logits, action), **tol)
        np.testing.assert_allclose(f64(server.value[slot]), v[:, 0], **tol)
    assert server.h2d_bytes == 3 * E * 64 * 4 and server.d2h_bytes == 3 * E * 4
    # the public act_fn face (get_act_fn) runs the same kernels through the network objects
    act_fn = seb.get_act_fn(apply_fns)
    a, v, lp, _ = act_fn(state.params, torch.as_tensor(obs, device="cuda"), 7)
    logits, _ = O.mlp_forward(actor, obs.astype(np.float64), bf16)
    np.testing.assert_allclose(f64(lp), O.categorical_log_prob(logits, a.cpu().numpy()), **tol)


@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_learner_step_matches_oracle(precision):
    """Two actors' (T+1)-step storages -> learner_step_fn, twice (LR schedule / Adam counters advance), vs the oracle."""
    from stoix_b200 import ops

    bf16 = precision == "bf16"
    cfg = _cfg([f"arch.precision={precision}"])
    seb, factory, learn_step, _, state = _setup(cfg)
    T, E_a, D, A = 8, 128, 64, 8
    E = 2 * E_a
    a_tree, c_tree = state.params.actor_params, state.params.critic_params
    actor, critic = tree(a_tree), tree(c_tree)
    n_a, n_c = actor.flat().size, critic.flat().size
    a_st, c_st = O.AdamState(np.zeros(n_a), np.zeros(n_a)), O.AdamState(np.zeros(n_c), np.zeros(n_c))
    h = O.PPOHyper(num_minibatches=2, num_updates=int(cfg.arch.num_updates))
    rng = np.random.default_rng(3)
    rel = lambda a, b: float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))
    for upd in range(2):
        obs = rng.standard_normal((T + 1, E, D)).astype(np.float32)
        if bf16:
            obs = torch.tensor(obs).to(torch.bfloat16).float().numpy()
        act = rng.integers(0, A, (T + 1, E)).astype(np.int32)
        logits, _ = O.mlp_forward(actor, obs.reshape(-1, D).astype(np.float64), bf16)
        lp = (O.categorical_log_prob(logits, act.reshape(-1)) + rng.standard_normal((T + 1) * E) * 0.1).reshape(T + 1, E).astype(np.float32)
        v, _ = O.mlp_forward(critic, obs.reshape(-1, D).astype(np.float64), bf16)
        val = (v[:, 0] + rng.standard_normal((T + 1) * E) * 0.1).reshape(T + 1, E).astype(np.float32)
        rew = rng.standard_normal((T + 1, E)).astype(np.float32)
        done = rng.random((T + 1, E)) < 0.1
        dev = lambda x, dt: torch.as_tensor(np.ascontiguousarray(x), device="cuda").to(dt)
        obs_dt = torch.bfloat16 if bf16 else torch.float32
        shards = []
        for k in range(2):
            sl = slice(k * E_a, (k + 1) * E_a)
            shards.append(seb.PPOTransition(dev(done[:, sl], torch.uint8), dev(np.zeros_like(done[:, sl]), torch.uint8), dev(act[:, sl], torch.int32),
                                            dev(val[:, sl], torch.float32), dev(rew[:, sl], torch.float32), dev(lp[:, sl], torch.float32),
                                            dev(obs[:, sl], obs_dt)))
        out = learn_step(state, shards)
        state = out.learner_state
        torch.cuda.synchronize()
        b = learn_step.built
        perms = np.stack([ops.make_permutation(T * E, state.key, ep + 4 * upd, device="cuda").cpu().numpy() for ep in range(4)])
        assert np.array_equal(perms, b["perms"].cpu().numpy())
        traj = O.Trajectory(obs=obs[:-1].astype(np.float64), action=act[:-1], reward=rew[:-1].astype(np.float64), done=done[:-1],
                            truncated=np.zeros_like(done[:-1]), next_obs=obs[1:].astype(np.float64), value=val[:-1].astype(np.float64),
                            bootstrap_value=val[1:].astype(np.float64), log_prob=lp[:-1].astype(np.float64))
        actor, critic, metrics, adv, tgt = O.ppo_update(actor, critic, a_st, c_st, traj, perms, h, bf16=bf16)
        np.testing.assert_allclose(f64(b["targets"]), tgt, rtol=1e-4, atol=2e-5)
        if bf16:
            _, coff, _ = ops.arena_offsets(a_tree.spec, c_tree.spec)
            mu, nu = f64(a_tree.arena_mu), f64(a_tree.arena_nu)
            assert max(rel(mu[:n_a], a_st.mu), rel(mu[coff:coff + n_c], c_st.mu)) < 0.3
            assert max(rel(nu[:n_a], a_st.nu), rel(nu[coff:coff + n_c], c_st.nu)) < 0.1
            actor, critic = tree(a_tree), tree(c_tree)
            a_st.mu, a_st.nu, c_st.mu, c_st.nu = mu[:n_a].copy(), nu[:n_a].copy(), mu[coff:coff + n_c].copy(), nu[coff:coff + n_c].copy()
        else:
            np.testing.assert_allclose(f64(a_tree.flat), actor.flat(), rtol=1e-4, atol=2e-6)
            np.testing.assert_allclose(f64(c_tree.flat), critic.flat(), rtol=1e-4, atol=2e-6)
            for name in ("actor_loss", "entropy", "value_loss"):
                np.testing.assert_allclose(f64(out.train_metrics[name]), metrics[name], rtol=2e-4, atol=2e-6)
    assert a_tree.arena_counts.cpu().tolist() == [2 * 4 * 2] * 4


@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_threaded_run_completes(precision):
    """2 actor threads (CPU synthetic envs) + learner + async evaluator: the experiment runs to the end, the parameters
    move and stay finite, every actor delivered (T+1)-step storages with a one-update policy lag (sebulba/ff_ppo.py:204-213)."""
    from stoix_b200.config import compose
    from stoix_b200.systems.ppo.sebulba import ff_ppo as seb

    cfg = compose("default_ff_ppo", ["arch.total_num_envs=256", "system.rollout_length=8", "system.num_minibatches=2",
                                     "arch.total_timesteps=24576", "arch.actor.actor_per_device=2", "arch.num_evaluation=2",
                                     "arch.num_eval_episodes=8", "logger.use_console=False", f"arch.precision={precision}",
                                     "arch.max_eval_steps=300"], config_dir="default/sebulba")
    perf = seb.run_experiment(cfg)
    assert np.isfinite(perf)


def test_threaded_run_with_actor_and_learner_on_different_gpus():
    """The Sebulba split proper (configs/arch/sebulba.yaml: actor.device_ids != learner.device_ids): inference servers on cuda:0, learner on
    cuda:1, rollouts cross by peer copy of the (T+1)-step storages, parameters come back by peer copy of the flat arena."""
    if torch.cuda.device_count() < 2:
        pytest.skip("NEEDS 2 GPUs: run `python -m pytest tests/test_sebulba_gpu.py -m gpu` on a machine with two")
    from stoix_b200.config import compose
    from stoix_b200.systems.ppo.sebulba import ff_ppo as seb

    for precision in ("bf16", "f32"):
        cfg = compose("default_ff_ppo", ["arch.total_num_envs=256", "system.rollout_length=8", "system.num_minibatches=2", "arch.total_timesteps=24576",
                                         "arch.actor.actor_per_device=2", "arch.num_evaluation=2", "arch.num_eval_episodes=8", "logger.use_console=False",
                                         f"arch.precision={precision}", "arch.max_eval_steps=300", "arch.actor.device_ids=[0]", "arch.learner.device_ids=[1]",
                                         "arch.evaluator_device_id=0"], config_dir="default/sebulba")
        assert np.isfinite(seb.run_experiment(cfg))
