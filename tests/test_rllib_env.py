"""RLlib-facing adaptor (qdsim.rllib_env.VectorMultiAgentEnv) against the reference wrapper's own methods
(src/qadapt/environment/multi_agent_wrapper.py:311-457, compiled from its source text) and its MultiAgentEnv contract
(:459-584).  Importable and testable without ray / gymnasium."""
import ast
import os
import types

import numpy as np
import pytest

from util import reference_path

REF = reference_path("qadapt", "environment", "multi_agent_wrapper.py")


def _reference_methods(names):
    tree = ast.parse(open(REF).read(), filename=REF)
    body = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in names]
    ns = {"np": np, "Dict": dict}
    exec(compile(ast.Module(body=body, type_ignores=[]), REF, "exec"), ns)
    return ns


def _env(n_env=1, n_dot=4, engine=None, **kw):
    from qdsim.rllib_env import VectorMultiAgentEnv
    from qdsim.vector_env import EnvConfig
    return VectorMultiAgentEnv(n_env, n_dot, engine=engine, config=EnvConfig(resolution=12, max_steps=3), seed=2, **kw)


def test_importable_without_ray_and_has_the_multi_agent_env_surface():
    import sys
    assert "ray" not in sys.modules
    env = _env(n_dot=5)
    assert env.all_agent_ids == [f"plunger_{i}" for i in range(5)] + [f"barrier_{j}" for j in range(4)]
    assert env._agent_ids == env.agents == env.possible_agents == set(env.all_agent_ids)
    assert set(env.observation_space.keys()) == set(env.action_space.keys()) == set(env.all_agent_ids)
    assert env.observation_space["plunger_2"]["image"].shape == (12, 12, 2)
    assert env.observation_space["barrier_1"]["image"].shape == (12, 12, 1)
    assert env.observation_space["plunger_0"]["voltage"].shape == (1,) and env.action_space["barrier_3"].shape == (1,)
    for name in ("reset", "step", "close"):
        assert callable(getattr(env, name))


@pytest.mark.skipif(not os.path.exists(REF), reason="reference tree not present")
@pytest.mark.parametrize("n_dot,return_global", [(4, False), (6, True), (2, False)])
def test_observation_extraction_equals_the_reference_wrapper(n_dot, return_global):
    """_extract_agent_observation of the reference, run per env on the same global observation."""
    ns = _reference_methods(["_extract_agent_observation", "_setup_channel_assignments"])
    E, res = 3, 12
    env = _env(n_env=E, n_dot=n_dot, return_global_state=return_global)
    rng = np.random.default_rng(0)
    image = rng.uniform(size=(E, n_dot - 1, res, res)).astype(np.float32)                # batched layout: channels first
    gobs = {"image": image, "obs_gate_voltages": rng.uniform(-1, 1, (E, n_dot)).astype(np.float32),
            "obs_barrier_voltages": rng.uniform(-1, 1, (E, n_dot - 1)).astype(np.float32)}
    me = types.SimpleNamespace(num_gates=n_dot, num_barriers=n_dot - 1, gate_agent_ids=env.gate_agent_ids,
                               barrier_agent_ids=env.barrier_agent_ids, gif_config=None, return_voltage=True,
                               return_global_state=return_global)
    ns["_setup_channel_assignments"](me)
    assert me.agent_channel_map == env.agent_channel_map
    for aid in env.all_agent_ids:
        ours = env._extract_agent_observation(gobs, aid)
        for e in range(E):
            ref_obs = {"image": np.transpose(image[e], (1, 2, 0)), "obs_gate_voltages": gobs["obs_gate_voltages"][e],
                       "obs_barrier_voltages": gobs["obs_barrier_voltages"][e]}                # reference: (H, W, N-1)
            ref = ns["_extract_agent_observation"](me, ref_obs, aid)
            assert set(ref) == set(ours)
            for k in ref:
                assert ref[k].dtype == np.float32 and ours[k][e].dtype == np.float32
                np.testing.assert_array_equal(ours[k][e], ref[k], err_msg=f"{aid} {k}")


@pytest.mark.skipif(not os.path.exists(REF), reason="reference tree not present")
def test_step_contract_without_gpu_matches_reference_action_and_reward_plumbing():
    ns = _reference_methods(["_combine_agent_actions", "_distribute_rewards"])
    env = _env(n_env=1, n_dot=4)
    obs, infos = env.reset(seed=11)
    assert obs is None and set(infos) == set(env.all_agent_ids)          # no engine: the shell runs, no images
    rng = np.random.default_rng(3)
    me = types.SimpleNamespace(num_gates=4, num_barriers=3, gate_agent_ids=env.gate_agent_ids,
                               barrier_agent_ids=env.barrier_agent_ids)
    for t in range(3):
        acts = {aid: rng.uniform(-1, 1, size=(1,)).astype(np.float32) for aid in env.all_agent_ids}
        ref_act = ns["_combine_agent_actions"](me, acts)
        env.base_env.eng = None
        obs, rew, term, trunc, infos = env.step(acts)
        want = (ref_act["action_gate_voltages"] + 1) / 2 * (env.base_env.plunger_max[0] - env.base_env.plunger_min[0]) \
            + env.base_env.plunger_min[0]
        np.testing.assert_allclose(env.base_env.gate_v[0], want, rtol=1e-6)
        assert set(rew) == set(env.all_agent_ids) and all(isinstance(r, float) for r in rew.values())
        glob = env.base_env._reward()
        ref_r = ns["_distribute_rewards"](me, {k: v[0] for k, v in glob.items()})
        assert rew == ref_r
        assert set(term) == set(trunc) == set(env.all_agent_ids) | {"__all__"}
        assert trunc["__all__"] == (t == 2) and term["__all__"] is False
        assert set(infos["barrier_1"]) == {"ground_truth", "current_voltage"}
    with pytest.raises(AssertionError):
        env.step({"plunger_0": np.zeros(1)})                                # all agents must act (:474-479)


def test_vector_form_carries_an_env_axis_and_slices_back_to_reference_shapes():
    env = _env(n_env=4, n_dot=3)
    env.reset()
    acts = {aid: np.zeros((4, 1), dtype=np.float32) for aid in env.all_agent_ids}
    obs, rew, term, trunc, infos = env.step(acts)
    assert rew["plunger_1"].shape == (4,) and term["plunger_0"].shape == (4,)
    one = env.sub_env(infos, 2)
    assert np.ndim(one["barrier_0"]["ground_truth"]) == 0
    assert env.episode_stats().shape == (4, 4)


@pytest.mark.gpu
def test_two_episode_rollout_on_the_gpu(engine):
    env = _env(n_env=1, n_dot=4, engine=engine)
    rng = np.random.default_rng(5)
    for ep in range(2):
        obs, infos = env.reset(seed=20 + ep)
        assert set(obs) == set(env.all_agent_ids)
        for aid in env.all_agent_ids:
            sp = env.observation_space[aid]
            assert obs[aid]["image"].shape == sp["image"].shape and obs[aid]["image"].dtype == np.float32
            assert obs[aid]["voltage"].shape == (1,)
            assert 0.0 <= obs[aid]["image"].min() and obs[aid]["image"].max() <= 1.0
        done = False
        steps = 0
        while not done:
            acts = {aid: rng.uniform(-1, 1, size=(1,)).astype(np.float32) for aid in env.all_agent_ids}
            obs, rew, term, trunc, infos = env.step(acts)
            steps += 1
            done = term["__all__"] or trunc["__all__"]
            # plunger_1: second channel is the transpose of global channel 1; barrier_j is channel j
            g = env.base_env.z_dev.view(1, 3, 12, 12).cpu().numpy()[0]
            np.testing.assert_array_equal(obs["plunger_1"]["image"][:, :, 0], g[0])
            np.testing.assert_array_equal(obs["plunger_1"]["image"][:, :, 1], g[1].T)
            np.testing.assert_array_equal(obs["barrier_2"]["image"][:, :, 0], g[2])
            np.testing.assert_array_equal(obs["plunger_3"]["image"][:, :, 0], g[2].T)
        assert steps == 3


@pytest.mark.gpu
def test_vector_rollout_on_the_gpu(engine):
    env = _env(n_env=8, n_dot=4, engine=engine)
    obs, _ = env.reset(seed=1)
    assert obs["plunger_2"]["image"].shape == (8, 12, 12, 2)
    acts = {aid: np.zeros((8, 1), dtype=np.float32) for aid in env.all_agent_ids}
    obs2, rew, term, trunc, infos = env.step(acts)
    one = env.sub_env(obs2, 5)
    assert one["barrier_0"]["image"].shape == (12, 12, 1) and one["plunger_0"]["voltage"].shape == (1,)
