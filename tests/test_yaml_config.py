"""`partial(Env, path_to_yaml)` (run_experiment.py:115): a user YAML overlaid on the compiled model's cfg block, and the
host-side BaseTask descriptors / interface views of the env protocol (SURVEY.md §8b).  CPU only: the overlay and the packing
are host code; the GPU side is covered by tests/test_gpu_parity.py::test_single_env_reference_protocol."""
import os

import numpy as np
import pytest

REF = os.environ.get("LHW_REFERENCE", "")     # a checkout of rohanpsingh/LearningHumanoidWalking, if one is at hand


def _write(tmp_path, text):
    p = tmp_path / "cfg.yaml"
    p.write_text(text)
    return p


def test_yaml_overlay_reaches_the_packed_model_constants(tmp_path):
    from learninghumanoidwalking_b200.envs.config import apply_config, load_yaml
    from learninghumanoidwalking_b200.model import load_model, pack_model
    mj = load_model("jvrc_walk")
    base = pack_model(mj)
    y = _write(tmp_path, "sim_dt: 0.0005\ncontrol_dt: 0.02\naction_smoothing: 0.3\n"
                         "kp: [100, 100, 100, 125, 40, 40, 100, 100, 100, 125, 40, 40]\n"
                         "half_sitting_pose: [-20, 0, 0, 40, 0, -20, -20, 0, 0, 40, 0, -20]\n"
                         "task:\n  goal_height: 0.78\n  total_duration: 0.9\n  swing_duration: 0.6\n  stance_duration: 0.3\n"
                         "xml_export_path: /tmp/whatever\n")
    m2 = apply_config(mj, load_yaml(y))
    assert mj["cfg"]["kp"][0] == 200.0, "the compiled model must not be edited in place"
    c = m2["cfg"]
    assert c["frame_skip"] == 40 and m2["opt"]["timestep"] == 0.0005 and c["action_smoothing"] == 0.3
    assert c["kp"][3] == 125.0 and c["kd"] == mj["cfg"]["kd"]
    assert np.allclose(c["nominal_qpos"][7:], np.deg2rad([-20, 0, 0, 40, 0, -20] * 2)) and c["nominal_qpos"][:7] == mj["cfg"]["nominal_qpos"][:7]
    flat = pack_model(m2)
    # the gait clock is rebuilt from the YAML's durations: period = floor(2 * total_duration / control_dt) = 90 (88 by default)
    from learninghumanoidwalking_b200.tasks.gait_clock import phase_clock_table
    period, table = phase_clock_table(0.6, 0.3, 0.1, "grounded", 1 / 0.02, total_duration=0.9)
    assert period == 90 and flat.size == base.size + 4 * (90 - 88)
    assert any(np.array_equal(flat[i:i + 4 * period], table.reshape(-1)) for i in range(flat.size - 4 * period + 1))
    with pytest.raises(ValueError, match="gait period"):
        apply_config(mj, {"task": {"total_duration": 2.0}})


def test_yaml_rejects_what_it_cannot_honour(tmp_path):
    from learninghumanoidwalking_b200.envs.config import apply_config
    from learninghumanoidwalking_b200.model import load_model
    walk, h1 = load_model("jvrc_walk"), load_model("h1")
    with pytest.raises(ValueError, match="integer multiple"):
        apply_config(walk, {"sim_dt": 0.003, "control_dt": 0.025})          # robots/robot_base.py:36-38
    with pytest.raises(ValueError, match="compile_model"):
        apply_config(h1, {"reduced_xml": False})
    with pytest.raises(ValueError, match="history"):
        apply_config(walk, {"obs_history_len": 3})
    with pytest.raises(ValueError, match="does not know"):
        apply_config(walk, {"no_such_key": 1})
    with pytest.raises(ValueError, match="only the H1"):
        apply_config(walk, {"perturbation": {"enable": True}})
    m = apply_config(h1, {"pdgains": {"left_knee": [150, 15], "torso": [40, 4]}, "init_noise": 0,
                          "observation_noise": {"enabled": False}, "perturbation": {"force_magnitude": 30}})
    names = [lk["joint"]["name"] for lk in m["links"][1:]]
    assert m["cfg"]["kp"][names.index("left_knee")] == 150 and m["cfg"]["kd"][names.index("left_knee")] == 15
    assert m["cfg"]["init_noise_deg"] == 0 and m["cfg"]["observation_noise"]["enabled"] is False
    assert m["cfg"]["perturbation"]["force_magnitude"] == 30 and m["cfg"]["perturbation"]["torque_magnitude"] == 2


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs LHW_REFERENCE: a checkout of the upstream project")
@pytest.mark.parametrize("model,rel", [("jvrc_walk", "envs/jvrc/configs/base.yaml"), ("jvrc_step", "envs/jvrc/configs/base.yaml"),
                                       ("h1", "envs/h1/configs/base.yaml")])
def test_the_references_own_yaml_is_the_compiled_configuration(model, rel):
    """Applying the reference's default YAML must change nothing: the compiled cfg block IS that file."""
    from learninghumanoidwalking_b200.envs.config import apply_config, load_yaml
    from learninghumanoidwalking_b200.model import load_model, pack_model
    mj = load_model(model)
    m2 = apply_config(mj, load_yaml(os.path.join(REF, rel)))
    assert np.array_equal(pack_model(m2), pack_model(mj))


def test_task_descriptors_carry_the_reference_attributes():
    from learninghumanoidwalking_b200.tasks.base_task import BaseTask
    from learninghumanoidwalking_b200.tasks.descriptors import STAND_WEIGHTS, STEP_WEIGHTS, WALK_WEIGHTS, make_task
    from learninghumanoidwalking_b200.envs.batched_env import REWARD_NAMES, STAND_REWARD_NAMES, STEP_REWARD_NAMES
    from learninghumanoidwalking_b200.model import load_model
    from types import SimpleNamespace
    assert tuple(WALK_WEIGHTS) == REWARD_NAMES and abs(sum(WALK_WEIGHTS.values()) - 1) < 1e-12      # tasks/walking_task.py:131-146
    assert tuple(STEP_WEIGHTS) == STEP_REWARD_NAMES and tuple(STAND_WEIGHTS) == STAND_REWARD_NAMES
    for model, dur in (("jvrc_walk", 88), ("jvrc_step", 88), ("h1", None)):
        mj = load_model(model)
        env = SimpleNamespace(mj=mj, model_name=model, dt=mj["cfg"]["control_dt"], interface=object(), robot=SimpleNamespace())
        t = make_task(env)
        assert isinstance(t, BaseTask) and t._client is env.interface
        for hook in ("reset", "step", "calc_reward", "done", "substep"):
            assert callable(getattr(t, hook))
        if dur:
            assert t._period == dur and t._goal_height_ref == 0.8 and t._swing_duration == 0.75 and len(t._neutral_pose) == 12
        t.reset(iter_count=4000)
        assert env.robot.iteration_count == 4000
    assert make_task(SimpleNamespace(mj=load_model("jvrc_step"), model_name="jvrc_step", dt=0.025, interface=None,
                                     robot=SimpleNamespace()))._mass == 62.4 + 20 * 800      # SURVEY Appendix C-3
