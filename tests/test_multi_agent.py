"""Multi-agent face of the batched env (qdsim.multi_agent) against the reference wrapper's own methods
(src/qadapt/environment/multi_agent_wrapper.py), compiled from the reference's source text and run per env."""
import ast
import os
import types

import numpy as np
import pytest

from util import reference_path

REF = reference_path("qadapt", "environment", "multi_agent_wrapper.py")


def _make(n_env=5, n_dot=4, engine=None, **cfg):
    from qdsim.multi_agent import BatchedMultiAgentEnv
    from qdsim.vector_env import BatchedDeviceEnv, EnvConfig
    base = BatchedDeviceEnv(n_env, n_dot, engine=engine, config=EnvConfig(resolution=16, max_steps=3, **cfg), seed=4)
    return BatchedMultiAgentEnv(base)


def _reference_methods(names):
    tree = ast.parse(open(REF).read(), filename=REF)
    body = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in names]
    ns = {"np": np, "Dict": dict}
    exec(compile(ast.Module(body=body, type_ignores=[]), REF, "exec"), ns)
    return ns


def test_episode_flow_without_gpu():
    env = _make()
    obs, infos = env.reset()
    assert obs is None and set(infos) == set(env.all_agent_ids)
    rng = np.random.default_rng(0)
    total = np.zeros(5)
    for t in range(3):
        acts = {aid: rng.uniform(-1, 1, size=(5, 1)) for aid in env.all_agent_ids}
        obs, rew, term, trunc, infos = env.step(acts, skip_obs=True)
        assert set(rew) == set(env.all_agent_ids) and all(r.shape == (5,) for r in rew.values())
        total += sum(rew.values())
        g = np.concatenate([acts[a] for a in env.gate_agent_ids], axis=1)
        want = (np.clip(g, -1, 1) + 1) / 2 * (env.base_env.plunger_max - env.base_env.plunger_min) + env.base_env.plunger_min
        np.testing.assert_allclose(env.base_env.gate_v, want, rtol=1e-5, atol=1e-5)      # actions are float32
        assert infos["plunger_2"]["current_voltage"].shape == (5,)
        assert trunc["__all__"] == (t == 2) and not term["__all__"]
    stats = env.episode_stats()
    assert stats.shape == (5, 4) and stats.dtype == np.float32
    np.testing.assert_allclose(stats[:, 0], total, rtol=1e-6)
    assert (stats[:, 1] == 3).all() and (stats[:, 2:] >= 0).all()


@pytest.mark.skipif(not os.path.exists(REF), reason="reference tree not present")
def test_matches_reference_wrapper_methods():
    ns = _reference_methods(["_combine_agent_actions", "_distribute_rewards", "_setup_channel_assignments"])
    env = _make(n_env=3, n_dot=5)
    me = types.SimpleNamespace(num_gates=5, num_barriers=4, gate_agent_ids=env.gate_agent_ids,
                               barrier_agent_ids=env.barrier_agent_ids)
    ns["_setup_channel_assignments"](me)
    assert me.agent_channel_map == env.agent_channel_map
    rng = np.random.default_rng(1)
    acts = {aid: rng.uniform(-1, 1, size=3) for aid in env.all_agent_ids}
    gate, barrier = env._combine_agent_actions(acts)
    rewards = {"gates": rng.uniform(size=(3, 5)), "barriers": rng.uniform(size=(3, 4))}
    ours = env._distribute_rewards(rewards)
    for e in range(3):
        ref = ns["_combine_agent_actions"](me, {aid: np.array([a[e]]) for aid, a in acts.items()})
        np.testing.assert_array_equal(gate[e], ref["action_gate_voltages"])
        np.testing.assert_array_equal(barrier[e], ref["action_barrier_voltages"])
        ref_r = ns["_distribute_rewards"](me, {k: v[e] for k, v in rewards.items()})
        assert {aid: float(ours[aid][e]) for aid in ours} == ref_r


@pytest.mark.gpu
def test_multi_agent_observations_on_gpu(engine):
    from qdsim import agents
    env = _make(n_env=4, n_dot=4, engine=engine)
    obs, _ = env.reset()
    assert set(obs) == set(env.all_agent_ids)
    assert obs["plunger_1"]["image"].shape == (4, 2, 16, 16) and obs["barrier_0"]["image"].shape == (4, 1, 16, 16)
    base_img = env.base_env.z_dev.view(4, 3, 16, 16)
    assert obs["plunger_1"]["image"][:, 1].data_ptr() != 0
    np.testing.assert_array_equal(obs["plunger_1"]["image"][:, 1].cpu().numpy(),
                                  base_img[:, 1].transpose(-1, -2).cpu().numpy())
    np.testing.assert_array_equal(obs["plunger_3"]["image"].cpu().numpy(),
                                  agents.agent_image(base_img, "plunger_3").cpu().numpy())
    acts = {aid: np.zeros((4, 1)) for aid in env.all_agent_ids}
    obs, rew, term, trunc, infos = env.step(acts)
    assert obs["plunger_0"]["voltage"].shape == (4, 1)
