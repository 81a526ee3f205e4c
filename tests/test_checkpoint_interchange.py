"""Checkpoint interchange with a reference checkout, both directions (the reference pickles WHOLE modules:
rl/utils/checkpointer.py:36-83, loaded back at run_experiment.py:274-277 and rl/algos/ppo.py:69-82).

  reference -> this build   tests/golden/ref_actor.pt / ref_critic.pt were written by the reference's own classes
                            (tools/gen_golden_ckpt.py); they load here with no reference on the path, give the recorded
                            outputs, and PPO.load_pretrained takes their weights / normalisation but not their stds.
  this build -> reference   a pair written by PPO.save's exporter is unpickled in a fresh interpreter that has ONLY the
                            reference on its path (LHW_REFERENCE names the checkout; skipped without one).
"""
import io
import json
import os
import subprocess
import sys
import zipfile

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
REF = os.environ.get("LHW_REFERENCE", "")     # a checkout of rohanpsingh/LearningHumanoidWalking, if one is at hand


def test_reference_checkpoint_loads_here_and_gives_the_recorded_outputs():
    from learninghumanoidwalking_b200.rl.policies import FF_V, Gaussian_FF_Actor
    g = json.load(open(os.path.join(GOLD, "ref_ckpt.json")))
    actor = torch.load(os.path.join(GOLD, "ref_actor.pt"), weights_only=False)
    critic = torch.load(os.path.join(GOLD, "ref_critic.pt"), weights_only=False)
    assert isinstance(actor, Gaussian_FF_Actor) and isinstance(critic, FF_V)      # resolved through the rl.policies alias
    assert sorted(actor.state_dict()) == g["actor_keys"] and sorted(critic.state_dict()) == g["critic_keys"]
    x = torch.tensor(g["x"])
    assert (actor(x) - torch.tensor(g["mu"])).abs().max() < 1e-6
    assert (critic(x) - torch.tensor(g["v"])).abs().max() < 1e-6
    assert (actor.distribution(x).mean - torch.tensor(g["mu"])).abs().max() < 1e-6
    # a freshly built network of this build takes the state dict as is
    mine = Gaussian_FF_Actor(37, 12, layers=(24, 24))
    mine.load_state_dict(actor.state_dict())


def test_continued_takes_weights_and_normalisation_but_reinitialises_stds():
    """rl/algos/ppo.py:69-82 through PPO.load_pretrained (host logic only: no CUDA)."""
    from learninghumanoidwalking_b200.rl.policies import FF_V, Gaussian_FF_Actor
    from learninghumanoidwalking_b200.rl.ppo import PPO
    g = json.load(open(os.path.join(GOLD, "ref_ckpt.json")))
    actor = torch.load(os.path.join(GOLD, "ref_actor.pt"), weights_only=False)
    critic = torch.load(os.path.join(GOLD, "ref_critic.pt"), weights_only=False)
    ppo = object.__new__(PPO)
    ppo.device = torch.device("cpu")
    for learn_std in (False, True):
        ppo.policy = Gaussian_FF_Actor(37, 12, layers=(24, 24), init_std=0.223, learn_std=learn_std)
        ppo.critic = FF_V(37, layers=(24, 24))
        ppo.policy.obs_mean, ppo.policy.obs_std = torch.zeros(37), torch.ones(37)
        ppo.critic.obs_mean, ppo.critic.obs_std = torch.zeros(37), torch.ones(37)
        import copy
        ppo.old_policy = copy.deepcopy(ppo.policy)
        ppo.load_pretrained(actor, critic)
        x = torch.tensor(g["x"])
        assert (ppo.policy(x) - torch.tensor(g["mu"])).abs().max() < 1e-6 and (ppo.critic(x) - torch.tensor(g["v"])).abs().max() < 1e-6
        assert (ppo.old_policy(x) - torch.tensor(g["mu"])).abs().max() < 1e-6
        assert torch.allclose(torch.as_tensor(ppo.policy.stds), torch.full((12,), 0.223))     # not the checkpoint's 0.3
    bad = Gaussian_FF_Actor(37, 12, layers=(16, 16))
    ppo.policy = Gaussian_FF_Actor(37, 12, layers=(24, 24))
    with pytest.raises((ValueError, RuntimeError)):
        ppo.load_pretrained(bad, critic)


def _export_pair(tmp_path, flat=True):
    from learninghumanoidwalking_b200.rl.optim import flatten_modules_
    from learninghumanoidwalking_b200.rl.policies import FF_V, Gaussian_FF_Actor, export_module
    torch.manual_seed(7)
    actor, critic = Gaussian_FF_Actor(37, 12, init_std=0.223), FF_V(37)
    actor.obs_mean = critic.obs_mean = torch.linspace(-1, 1, 37)
    actor.obs_std = critic.obs_std = torch.linspace(0.5, 4, 37)
    if flat:      # the trainer's modules are views of one flat (actor + critic) buffer
        try:
            flatten_modules_([actor, critic])
        except Exception:
            pass
    pa, pc = tmp_path / "actor_7.pt", tmp_path / "critic_7.pt"
    torch.save(export_module(actor), pa)
    torch.save(export_module(critic), pc)
    return actor, critic, pa, pc


def test_exported_files_name_the_reference_classes_and_hold_only_their_own_parameters(tmp_path):
    actor, critic, pa, pc = _export_pair(tmp_path)
    for path, cls, n in ((pa, b"rl.policies.actor", 78604), (pc, b"rl.policies.critic", 75777)):
        z = zipfile.ZipFile(path)
        pkl = z.read([k for k in z.namelist() if k.endswith("data.pkl")][0])
        assert cls in pkl and b"learninghumanoidwalking" not in pkl
        data = sum(z.getinfo(k).file_size for k in z.namelist() if "/data/" in k)
        assert data < (n + 200) * 4, "the file must not carry the flat actor+critic buffer"
    back = torch.load(pa, weights_only=False)
    x = torch.randn(3, 37)
    assert torch.equal(back(x), actor(x))


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs LHW_REFERENCE: a checkout of the upstream project")
def test_a_reference_checkout_unpickles_our_files_with_its_own_classes(tmp_path):
    actor, critic, pa, pc = _export_pair(tmp_path)
    x = torch.randn(4, 37)
    torch.save(x, tmp_path / "x.pt")
    code = (
        "import sys, torch\n"
        f"sys.path.insert(0, {REF!r})\n"
        f"a = torch.load({str(pa)!r}, weights_only=False); c = torch.load({str(pc)!r}, weights_only=False)\n"
        "import rl.policies.actor as A, rl.policies.critic as C\n"
        f"assert A.__file__.startswith({REF!r}) and type(a) is A.Gaussian_FF_Actor and type(c) is C.FF_V\n"
        "assert 'learninghumanoidwalking_b200' not in sys.modules\n"
        f"x = torch.load({str(tmp_path / 'x.pt')!r})\n"
        "a.eval(); c.eval()\n"                                  # run_experiment.py:276-277
        "d = a.distribution(x)\n"
        f"torch.save((a(x, deterministic=True), c(x), d.stddev, a.stds), {str(tmp_path / 'out.pt')!r})\n")
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path), env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    mu, v, sd, stds = torch.load(tmp_path / "out.pt")
    assert torch.allclose(mu, actor(x), atol=1e-6) and torch.allclose(v, critic(x), atol=1e-6)
    assert torch.allclose(stds, torch.full((12,), 0.223))
