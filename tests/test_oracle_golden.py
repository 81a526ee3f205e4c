"""Pin the oracle (and the product's host-side tables) to vectors produced by the reference's own code
(tools/gen_golden.py ran tasks/rewards.py, rl/storage/rollout_storage.py, rl/policies, rl/envs/wrappers)."""
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def gold(name):
    return json.load(open(os.path.join(GOLD, name)))


def test_gait_clock_table_matches_reference_splines():
    from learninghumanoidwalking_b200.tasks.gait_clock import phase_clock_table
    g = gold("gait_clocks.json")
    period, table = phase_clock_table(0.75, 0.35, 0.1, "grounded", 40, total_duration=1.1)
    assert period == g["period"] == 88
    for row, key in enumerate(("r_frc", "r_vel", "l_frc", "l_vel")):
        assert np.abs(table[row] - np.array(g[key])).max() < 1e-12
    # WalkingTask.step tests `clock == 1` exactly (tasks/walking_task.py:156): double-support phases must be exact
    dbl = [p for p in range(88) if table[0][p] == 1.0 and table[2][p] == 1.0]
    assert dbl == [p for p in range(88) if g["r_frc"][p] == 1 and g["l_frc"][p] == 1] == list(range(32, 43)) + list(range(76, 87))


def test_roll_pitch_matches_static_xyz_euler(oracle_tight):
    for c in gold("roll_pitch.json"):
        r, p = oracle_tight.quat2rp(c["quat"])
        assert abs(r - c["roll"]) < 1e-12 and abs(p - c["pitch"]) < 1e-12


def test_reward_terms_match_reference(oracle_tight):
    """Drive oracle calc_reward through its env fields so that each term sees exactly the golden inputs."""
    o = oracle_tight
    envs = o.make_envs(1)
    W = dict(fwd_vel=0.15, yaw_vel=0.15, action=0.025, torque=0.025, height=0.05, root_accel=0.05, foot_frc=0.225, foot_vel=0.225)
    for c in gold("reward_terms.json"):
        ph = c["foot_frc"]["phase"]
        o.set_field(envs, 0, "phase", [ph])
        o.set_field(envs, 0, "mode", [2])  # FORWARD: refs (yaw 0, vx, vy=0)
        # com velocity: identity root frame, goal (vx, 0)
        o.set_field(envs, 0, "root_xmat", np.eye(3).reshape(-1))
        rv, gv = c["fwd_vel"]["root_vel"], c["fwd_vel"]["goal"]
        o.set_field(envs, 0, "mode_ref", [0.0, gv[0], 0.0])
        o.set_field(envs, 0, "root_vlin", [rv[0], rv[1] - gv[1], 0.0])
        qv = np.array(c["root_accel"]["qvel"])
        qv[5] = c["yaw_vel"]["yaw_vel"] - c["yaw_vel"]["ref"]  # yaw ref is 0 in FORWARD
        o.set_field(envs, 0, "qvel", qv)
        o.set_field(envs, 0, "qacc", c["root_accel"]["qacc"])
        o.set_field(envs, 0, "lfoot_grf", [c["foot_frc"]["l"]])
        o.set_field(envs, 0, "rfoot_grf", [c["foot_frc"]["r"]])
        o.set_field(envs, 0, "lfoot_vel", c["foot_vel"]["l"])
        o.set_field(envs, 0, "rfoot_vel", c["foot_vel"]["r"])
        o.set_field(envs, 0, "prev_torque", c["torque"]["prev"])
        o.set_field(envs, 0, "act_force", c["torque"]["t"])
        o.set_field(envs, 0, "prev_action", c["action"]["prev"])
        t = o.calc_reward(envs, 0, c["action"]["a"])
        assert abs(t[0] - W["foot_frc"] * c["foot_frc"]["out"]) < 1e-12
        assert abs(t[1] - W["foot_vel"] * c["foot_vel"]["out"]) < 1e-12
        qv_ref = np.array(c["root_accel"]["qvel"])
        exp_acc = np.exp(-0.25 * (np.abs(qv[3:6]).sum() + np.abs(np.array(c["root_accel"]["qacc"])[0:3]).sum()))
        assert abs(t[2] - W["root_accel"] * exp_acc) < 1e-12
        assert abs(t[4] - W["fwd_vel"] * c["fwd_vel"]["out"]) < 1e-12
        assert abs(t[5] - W["yaw_vel"] * c["yaw_vel"]["out"]) < 1e-12
        assert abs(t[8] - W["torque"] * c["torque"]["out"]) < 1e-12
        assert abs(t[9] - W["action"] * c["action"]["out"]) < 1e-12
        del qv_ref
    # root_accel and height with their own golden inputs (FORWARD speed couples height's dead zone to vx)
    for c in gold("reward_terms.json"):
        o.set_field(envs, 0, "mode", [2])
        o.set_field(envs, 0, "mode_ref", [0.0, c["height"]["speed"], 0.0])
        o.set_field(envs, 0, "root_xpos", [0.0, 0.0, c["height"]["h"]])
        o.set_field(envs, 0, "contact_z_min", [c["height"]["cz"]])
        o.set_field(envs, 0, "ncon_r", [1])
        o.set_field(envs, 0, "qvel", c["root_accel"]["qvel"])
        o.set_field(envs, 0, "qacc", c["root_accel"]["qacc"])
        t = o.calc_reward(envs, 0, np.zeros(12))
        assert abs(t[3] - 0.05 * c["height"]["out"]) < 1e-12
        assert abs(t[2] - 0.05 * c["root_accel"]["out"]) < 1e-12


def test_known_answers_from_survey_appendix_b():
    from oracle.ppo_oracle import gae_path
    r = gae_path([1, 2, 3, 4, 5], [0, .5, 1, 1.5, 2], 2.0, 0.99, 0.95)
    assert np.allclose(r, [14.542834082482912, 14.3732951435225, 13.103450445, 10.66369, 6.98], atol=1e-12)


def test_gae_oracle_matches_reference_buffer():
    from oracle.ppo_oracle import gae_rollout
    for c in gold("gae.json"):
        T = len(c["rewards"])
        ended = np.zeros((T, 1), dtype=int)
        boot = np.zeros((T, 1))
        for e_, lv in zip(c["path_ends"], c["last_vals"]):
            ended[e_ - 1, 0] = 1
            boot[e_ - 1, 0] = lv
        ret = gae_rollout(np.array(c["rewards"])[:, None], np.array(c["values"])[:, None], ended, boot, np.zeros(1),
                          c["gamma"], c["lam"])
        assert np.abs(ret[:, 0] - np.array(c["returns"])).max() < 1e-12


def test_model_constants():
    from learninghumanoidwalking_b200.model import load_model
    m = load_model("jvrc_walk")
    assert abs(m["total_mass"] - 62.4) < 1e-9                       # SURVEY Appendix B
    assert len(m["links"]) == 13 and m["cfg"]["frame_skip"] == 25
    names = [lk["joint"]["name"] for lk in m["links"][1:]]
    assert names == ["R_HIP_P", "R_HIP_R", "R_HIP_Y", "R_KNEE", "R_ANKLE_R", "R_ANKLE_P",
                     "L_HIP_P", "L_HIP_R", "L_HIP_Y", "L_KNEE", "L_ANKLE_R", "L_ANKLE_P"]  # envs/jvrc/gen_xml.py:42-55
    assert abs(m["total_mass"] * 9.8 * 0.5 - 305.76) < 1e-9


@pytest.mark.skipif(not os.path.isdir(os.environ.get("LHW_REFERENCE", "")),
                    reason="needs LHW_REFERENCE: a checkout of the upstream project")
def test_compiled_model_is_reproducible_from_reference():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools"))
    import compile_model
    from learninghumanoidwalking_b200.model import load_model
    fresh, stored = compile_model.compile_jvrc(), load_model("jvrc_walk")
    for a, b in zip(fresh["links"], stored["links"]):
        assert a["name"] == b["name"] and np.allclose(a["inertia"], b["inertia"]) and np.allclose(a["com"], b["com"])
    assert np.allclose(fresh["dof_invweight0"], stored["dof_invweight0"])


def test_rollout_bootstrap_semantics_match_the_reference_worker():
    """tests/golden/rollout_worker.json = the reference's RolloutWorker.sample run on a scripted env for three consecutive
    calls (tools/gen_golden_rollout.py).  The oracle's time-major GAE (ppo_oracle.gae_rollout: what the CUDA GAE kernel and the
    device rollout worker are tested against) must give the reference's returns from the same per-step rewards / values /
    episode-end flags with boot = (not done) * critic(pre-reset next state) and the open tail closed by critic(current state)."""
    import torch
    from oracle.ppo_oracle import gae_rollout
    Gr = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rollout_worker.json")))
    W, b = torch.tensor(Gr["critic_w"], dtype=torch.float32), Gr["critic_b"]
    V = lambda s: float((torch.tensor(s, dtype=torch.float32) @ W + b).reshape(-1)[0])
    T, carried = Gr["T"], 0
    for call in Gr["calls"]:
        ended = np.array(call["dones"]).astype(bool)
        done = np.array(call["env_done"])
        assert (ended >= done).all()                                  # every true termination ends the episode ...
        boot = np.array([(0.0 if done[t] else V(call["next_obs"][t])) if ended[t] else 0.0 for t in range(T)])
        last_val = V(call["open_state"]) if call["open_state"] is not None else 0.0
        assert (call["open_state"] is None) == bool(ended[-1])
        ret = gae_rollout(np.array(call["rewards"])[:, None], np.array(call["values"])[:, None], ended[:, None], boot[:, None],
                          np.array([last_val]), Gr["gamma"], Gr["lam"])[:, 0]
        assert np.abs(ret - np.array(call["returns"])).max() < 1e-6
        # ... and truncation at max_traj_len does too; episode lengths carry over between calls; only completed episodes report
        lens, run = [], carried
        for t in range(T):
            run += 1
            if ended[t]:
                assert done[t] or run == Gr["max_traj_len"]
                lens.append(run)
                run = 0
        carried = run
        assert lens == call["ep_lens"] and len(call["ep_rewards"]) == len(lens)


def test_walking_task_matches_the_reference_class():
    """WalkingTask.reset / step / calc_reward / done (tasks/walking_task.py:85-205) run from the reference's own file on recorded
    inputs (tools/gen_golden_walk_task.py), its numpy RNG fed with the Philox words the oracle draws for the same event key.  The
    terrain extension's re-pose event is checked against the reference's manip_hfield hook (:172-179) the same way: same third
    `randint(200)` decision, same three uniforms in the same order (the shipped terrain model lists the z range sorted; the hook's
    call has it as (-0.015, -0.035), which is what this test passes so that the same uniform maps to the same offset)."""
    import copy
    from oracle.oracle import Oracle, load_model_json
    cases = gold("walk_task.json")
    o = Oracle("jvrc_walk", tolerance=1e-14)
    tm = copy.deepcopy(load_model_json("jvrc_walk_terrain"))
    assert sorted((tm["terrain"]["z_lo"], tm["terrain"]["z_hi"])) == [-0.035, -0.015] and tm["terrain"]["xy"] == 0.5
    assert tm["terrain"]["interval"] == 200
    tm["terrain"].update(z_lo=-0.015, z_hi=-0.035, bump=0.0)
    ot = Oracle(model_dict=tm, tolerance=1e-14)
    cfg = o.mj["cfg"]
    assert cases[0]["names"] == ["foot_frc_score", "foot_vel_score", "root_accel", "height_error", "com_vel_error", "yaw_vel_error",
                                 "upper_body_reward", "posture_error", "torque_penalty", "action_penalty"]
    seen_modes, n_switch, n_hook, n_done = set(), 0, 0, 0
    for c in cases:
        envs, envt = o.make_envs(1, seed=c["seed"], first_id=c["env_id"]), ot.make_envs(1, seed=c["seed"], first_id=c["env_id"])
        for oo, ee in ((o, envs), (ot, envt)):
            oo.set_field(ee, 0, "rng_ctr", c["reset_ctr"])
            oo.task_reset(ee, 0)
            assert int(oo.field(ee, 0, "mode")[0]) == c["mode"] and int(oo.field(ee, 0, "phase")[0]) == c["phase"]
            assert np.abs(oo.field(ee, 0, "mode_ref") - np.array(c["mode_ref"])).max() < 1e-15
        assert c["period"] == round(2 * cfg["task"]["total_duration"] / cfg["control_dt"])
        seen_modes.add(c["mode"])
        for s in c["steps"]:
            seq_before = ot.field(envt, 0, "seq").reshape(20, 4).copy()
            for oo, ee in ((o, envs), (ot, envt)):
                oo.set_field(ee, 0, "mode", s["pre"]["mode"]); oo.set_field(ee, 0, "mode_ref", s["pre"]["mode_ref"])
                oo.set_field(ee, 0, "phase", s["pre"]["phase"]); oo.set_field(ee, 0, "rng_ctr", s["ctr"])
                oo.task_step(ee, 0)
                assert int(oo.field(ee, 0, "mode")[0]) == s["mode"] and int(oo.field(ee, 0, "phase")[0]) == s["phase"], s["kind"]
                assert np.abs(oo.field(ee, 0, "mode_ref") - np.array(s["mode_ref"])).max() < 1e-15
            n_switch += s["mode"] != s["pre"]["mode"]
            seq = ot.field(envt, 0, "seq").reshape(20, 4)
            if s["kind"] == "hook":
                hp = np.array(s["hfield_pos"])
                assert np.abs(seq[:, 0] - (hp[0] + (np.arange(20) - 4) * tm["terrain"]["pitch"])).max() < 1e-15
                assert np.abs(seq[:, 1] - hp[1]).max() < 1e-15 and np.abs(seq[:, 2] - hp[2]).max() < 1e-15
                assert -0.5 <= hp[0] <= 0.5 and -0.035 <= hp[2] <= -0.015
                n_hook += 1
            else:
                assert (seq == seq_before).all()
            st = s["state"]
            o.set_field(envs, 0, "root_xmat", np.eye(3).reshape(-1))    # get_body_vel(root, frame=1) is already root-local
            o.set_field(envs, 0, "root_vlin", st["root_vloc"])
            o.set_field(envs, 0, "root_xpos", st["root"]); o.set_field(envs, 0, "head_xpos", st["head"])
            o.set_field(envs, 0, "qvel", st["qvel"]); o.set_field(envs, 0, "qacc", st["qacc"])
            o.set_field(envs, 0, "lfoot_grf", st["lgrf"]); o.set_field(envs, 0, "rfoot_grf", st["rgrf"])
            o.set_field(envs, 0, "lfoot_vel", st["lvel"]); o.set_field(envs, 0, "rfoot_vel", st["rvel"])
            o.set_field(envs, 0, "ncon_r", s["ncon_r"]); o.set_field(envs, 0, "ncon_l", s["ncon_l"])
            o.set_field(envs, 0, "contact_z_min", s["contact_z_min"])
            o.set_field(envs, 0, "act_len", st["pose"]); o.set_field(envs, 0, "act_force", st["torque"])
            o.set_field(envs, 0, "prev_torque", s["prev_torque"]); o.set_field(envs, 0, "prev_action", s["prev_action"])
            t = o.calc_reward(envs, 0, s["action"])
            assert np.abs(t - np.array(s["terms"])).max() < 1e-13, (s["kind"], t - np.array(s["terms"]))
            z = st["qpos"][2]
            assert ((z < 0.6) or (z > 1.4) or st["selfcol"]) == s["done"]    # the bounds oracle.pack_model / model.loader pack
            n_done += s["done"]
    assert seen_modes == {0, 1, 2} and n_switch >= 30 and n_hook >= 15 and 5 <= n_done < 80


def test_policy_trained_on_the_gpu_simulator_walks_in_the_oracle():
    """tests/golden/trained_actor_jvrc_walk.pt is the actor of a 40-iteration `run_experiment.py train --env jvrc_walk --num-procs 4096
    --seed 0` run on the fp32 CUDA simulator (mean episode length 398 of 400 there).  Driven by the same actor (float64 forward,
    deterministic mean + 0.05 exploration noise), the CPU oracle's environments also survive the 400-step horizon: the two
    implementations agree at the level of behaviour, not only step by step (tests/test_gpu_parity_shipped.py holds them to 1e-4
    along such trajectories)."""
    import torch
    from learninghumanoidwalking_b200.rl.policies import install_reference_aliases
    from oracle.oracle import Oracle
    install_reference_aliases()
    actor = torch.load(os.path.join(os.path.dirname(__file__), "golden", "trained_actor_jvrc_walk.pt"), map_location="cpu",
                       weights_only=False).double().eval()
    o = Oracle("jvrc_walk")
    n = 8
    envs = o.make_envs(n, seed=31, first_id=5)
    obs = o.batch_reset(envs, n)
    rng = np.random.RandomState(3)
    ended_at = []
    total = np.zeros(n)
    for k in range(400):
        with torch.no_grad():
            act = actor(torch.from_numpy(obs), deterministic=True).numpy()
        obs, _, _, rew, done, end = o.batch_step(envs, n, act + 0.05 * rng.normal(size=(n, 12)), max_traj_len=400)
        total += rew * (len(ended_at) == 0)
        if end.any():
            ended_at.append(k)
            assert k == 399 and end.all() and not done.any()      # truncation, not a fall
    assert ended_at == [399] and total.mean() > 200.0, (ended_at, total.mean())
