"""Self-collision termination (SURVEY.md Appendix C-4, row S7): the capsule proxies against exact intersection of the reference's
convex leg hulls on sampled poses (tools/eval_collision_proxies.py -> tests/golden/self_collision_eval.json; the STL files are
only in the reference checkout, so the evaluation is committed and, where the checkout is present, spot-checked again)."""
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_committed_evaluation_bounds_the_proxy_error():
    ev = json.load(open(os.path.join(ROOT, "tests", "golden", "self_collision_eval.json")))
    assert ev["n_samples"] >= 1000 and ev["pairs"] == {"cross_leg": 16, "same_leg": 6}
    for name, d in ev["distributions"].items():
        # same-leg geom pairs (HIP_R-KNEE, HIP_R-foot, HIP_Y-foot) never intersect inside the joint ranges: leaving them out of
        # the kernel's pair list is exact, not an approximation
        assert d["same_leg"]["hull"] == 0 and d["same_leg"]["proxy"] == 0, name
        # cross-leg: the proxies disagree with the hulls on < 2 % of the poses in either direction
        assert d["cross_leg"]["fp"] < 0.02 and d["cross_leg"]["fn"] < 0.02, (name, d["cross_leg"])
        assert abs(d["cross_leg"]["proxy"] - d["cross_leg"]["hull"]) < 0.01
    # on the poses of an actual gait (a trained policy walking in the oracle) neither the hulls nor the proxies touch
    gait = [d for name, d in ev["distributions"].items() if name.startswith("states of a trained walking policy")]
    assert len(gait) == 1 and gait[0]["cross_leg"] == {"hull": 0.0, "proxy": 0.0, "fp": 0.0, "fn": 0.0}
    from learninghumanoidwalking_b200.model import load_model
    for model in ("jvrc_walk", "jvrc_step", "jvrc_walk_terrain"):
        sc = load_model(model)["self_collision"]
        assert len(sc["capsules"]) == 12 and len(sc["pairs"]) == 36
        legs = [0 if c["link"] <= 6 else 1 for c in sc["capsules"]]
        assert all(legs[a] != legs[b] for a, b in sc["pairs"])


REF = os.environ.get("LHW_REFERENCE", "")     # a checkout of rohanpsingh/LearningHumanoidWalking, if one is at hand


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "models/jvrc_mj_description/meshes/convex")),
                    reason="needs LHW_REFERENCE: a checkout of the upstream project (its STL hulls)")
def test_spot_check_against_the_hulls():
    import sys
    sys.path.insert(0, ROOT)
    from tools.compile_model import kinematics
    from tools.eval_collision_proxies import hulls_intersect, seg_seg_dist2
    from tools.fit_collision_proxies import GEOM_QUAT, MESH_DIR, load_stl, quat2mat
    from learninghumanoidwalking_b200.model import load_model
    mj = load_model("jvrc_walk")
    li = {lk["name"]: i for i, lk in enumerate(mj["links"])}
    hull = {n: load_stl(os.path.join(MESH_DIR, n + ".stl")) @ quat2mat(GEOM_QUAT[n.split("_", 1)[1][:-2]]).T for n in ("R_HIP_Y_S", "L_HIP_Y_S")}
    caps = [c for c in mj["self_collision"]["capsules"] if c["name"] in hull]
    q = np.array(mj["cfg"]["nominal_qpos"])
    for roll, expect in ((0.0, False), (0.45, True)):      # thighs apart in the nominal stance, crossed at +-0.45 rad of hip roll
        q2 = q.copy()
        q2[7 + 1], q2[7 + 7] = roll, -roll
        xpos, xmat = kinematics(mj, q2)
        W = {n: xpos[li[n]] + v @ np.asarray(xmat[li[n]]).T for n, v in hull.items()}
        assert hulls_intersect(W["R_HIP_Y_S"], W["L_HIP_Y_S"]) == expect
        E = [(xpos[c["link"]] + xmat[c["link"]] @ np.array(c["p0"]), xpos[c["link"]] + xmat[c["link"]] @ np.array(c["p1"]), c["radius"], c["link"]) for c in caps]
        prox = any(seg_seg_dist2(a[0], a[1], b[0], b[1]) < (a[2] + b[2]) ** 2 for a in E for b in E if a[3] <= 6 < b[3])
        assert prox == expect


def test_leg_meshes_stay_clear_of_the_stepping_stones_before_termination():
    """jvrc_step collides the stepping stones with the foot boxes only (DESIGN.md 4.3); MuJoCo would also test the thigh / shin
    meshes.  tools/shin_clearance.py measured the capsule proxies' clearance on pre-termination states of oracle rollouts at the
    top of the height curriculum: under the early-training action spread no capsule comes within 6 cm of a stone; under
    sigma = 1.0 a shin is inside a stone on < 1 % of the steps, nearly all of them the fall that is about to end the episode."""
    ev = json.load(open(os.path.join(ROOT, "tests", "golden", "shin_clearance.json")))
    early, wild = ev["sigma_0.223"], ev["sigma_1.0"]
    assert early["pairs"] > 40000 and early["fraction_of_steps_with_a_leg_capsule_inside_a_stone"] == 0.0
    assert min(c["clearance_m_quantiles_0_1_5_50"][0] for c in early["per_capsule"].values()) > 0.06
    assert wild["pairs"] > 10000 and wild["fraction_of_steps_with_a_leg_capsule_inside_a_stone"] < 0.01
    assert wild["of_those_root_below_0.65m"] > 0.9
