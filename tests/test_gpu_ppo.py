"""GPU tests of the PPO data path through the C-ABI (GAE, advantage normalisation, minibatch gather, clip+Adam)
against oracle/ppo_oracle.py (pinned to the reference's PPOBuffer by tests/golden/gae.json), and of the
DeviceRolloutWorker / PPO host classes against the reference's behavioural contract (tests/test_training.py)."""
import json
import os
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _lib():
    from learninghumanoidwalking_b200 import _lib
    return _lib


def _gae_gpu(rew, val, ended, boot, last, gamma, lam):
    L = _lib()
    T, N = rew.shape
    d = lambda a, dt=torch.float32: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device="cuda")
    r, v, e, b, lv = d(rew), d(val), d(ended, torch.int32), d(boot), d(last)
    ret = torch.empty_like(r)
    part = torch.zeros(L.lib().lhw_gae_partial_words(N), dtype=torch.float64, device="cuda")
    L.check(L.lib().lhw_gae(r.data_ptr(), v.data_ptr(), e.data_ptr(), b.data_ptr(), lv.data_ptr(), ret.data_ptr(), T, N,
                            gamma, lam, part.data_ptr(), L.current_stream_ptr()))
    # the advantage statistics the launch leaves behind (sum, sumsq of returns - values per block) equal a direct reduction
    adv = ret.double() - v.double()
    nb = part.numel() // 2
    assert abs(part[:nb].sum().item() - adv.sum().item()) < 1e-6 * max(1.0, adv.abs().sum().item())
    assert abs(part[nb:].sum().item() - (adv * adv).sum().item()) < 1e-9 * max(1.0, (adv * adv).sum().item())
    return ret.cpu().numpy()


def test_gae_matches_reference_buffer_golden():
    for c in json.load(open(os.path.join(GOLD, "gae.json"))):
        T = len(c["rewards"])
        ended, boot = np.zeros((T, 1), np.int32), np.zeros((T, 1))
        for e_, lv in zip(c["path_ends"], c["last_vals"]):
            ended[e_ - 1, 0], boot[e_ - 1, 0] = 1, lv
        ret = _gae_gpu(np.array(c["rewards"])[:, None], np.array(c["values"])[:, None], ended, boot, np.zeros(1), c["gamma"], c["lam"])
        assert np.abs(ret[:, 0] - np.array(c["returns"])).max() < 2e-6 * max(1, np.abs(c["returns"]).max())


def test_gae_full_size_against_oracle_and_linearity():
    from oracle.ppo_oracle import gae_rollout
    rng = np.random.RandomState(0)
    T, N = 400, 4096
    rew, val = rng.uniform(-1, 1, (T, N)).astype(np.float32), rng.uniform(-2, 2, (T, N)).astype(np.float32)
    ended = (rng.rand(T, N) < 0.02).astype(np.int32)
    boot = (rng.uniform(-2, 2, (T, N)) * (rng.rand(T, N) < 0.5)).astype(np.float32)
    last = rng.uniform(-2, 2, N).astype(np.float32)
    ret = _gae_gpu(rew, val, ended, boot, last, 0.99, 0.95)
    sub = slice(0, 64)
    exp = gae_rollout(rew[:, sub].astype(np.float64), val[:, sub].astype(np.float64), ended[:, sub], boot[:, sub].astype(np.float64),
                      last[sub].astype(np.float64), 0.99, 0.95)
    assert np.abs(ret[:, sub] - exp).max() < 1e-4
    # size-independent property: GAE is linear in (rewards, values, boot, last_val)
    ret2 = _gae_gpu(2 * rew, 2 * val, ended, 2 * boot, 2 * last, 0.99, 0.95)
    assert np.abs(ret2 - 2 * ret).max() < 1e-4


def test_advantage_normalisation():
    from oracle.ppo_oracle import adv_normalize
    L = _lib()
    rng = np.random.RandomState(1)
    n = 4096 * 400
    ret, val = rng.normal(size=n).astype(np.float32), rng.normal(size=n).astype(np.float32) * 0.5 + 0.1
    r, v = torch.as_tensor(ret, device="cuda"), torch.as_tensor(val, device="cuda")
    stats = torch.zeros(L.lib().lhw_adv_stats_words(), dtype=torch.float64, device="cuda")
    adv = torch.empty_like(r)
    st = L.current_stream_ptr()
    L.check(L.lib().lhw_adv_stats(r.data_ptr(), v.data_ptr(), stats.data_ptr(), n, st))
    L.check(L.lib().lhw_adv_apply(r.data_ptr(), v.data_ptr(), adv.data_ptr(), stats.data_ptr(), n, n, 1e-5, st))
    exp = adv_normalize(ret, val, 1e-5)
    assert np.abs(adv.cpu().numpy() - exp).max() < 1e-5
    a = adv.double()
    assert abs(a.mean().item()) < 1e-6 and abs(a.std().item() - 1) < 1e-4
    # run-to-run deterministic
    adv2 = torch.empty_like(r)
    L.check(L.lib().lhw_adv_stats(r.data_ptr(), v.data_ptr(), stats.data_ptr(), n, st))
    L.check(L.lib().lhw_adv_apply(r.data_ptr(), v.data_ptr(), adv2.data_ptr(), stats.data_ptr(), n, n, 1e-5, st))
    assert torch.equal(adv, adv2)


def test_gather_minibatch_is_exact():
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(0)
    n, B = 50000, 64
    obs, act = torch.randn(n, 37, device="cuda", generator=g), torch.randn(n, 12, device="cuda", generator=g)
    ret, adv = torch.randn(n, 1, device="cuda", generator=g), torch.randn(n, 1, device="cuda", generator=g)
    idx = torch.randperm(n, device="cuda")[:B]
    o, a, r, d = (torch.empty(B, 37, device="cuda"), torch.empty(B, 12, device="cuda"), torch.empty(B, 1, device="cuda"), torch.empty(B, 1, device="cuda"))
    L.check(L.lib().lhw_gather_minibatch(obs.data_ptr(), act.data_ptr(), ret.data_ptr(), adv.data_ptr(), idx.data_ptr(), o.data_ptr(),
                                         a.data_ptr(), r.data_ptr(), d.data_ptr(), B, 37, 12, L.current_stream_ptr()))
    assert torch.equal(o, obs[idx]) and torch.equal(a, act[idx]) and torch.equal(r, ret[idx]) and torch.equal(d, adv[idx])


def test_fused_clip_adam_matches_torch_clip_grad_norm_and_adam():
    from learninghumanoidwalking_b200.rl import FusedClipAdam, Gaussian_FF_Actor
    from oracle.ppo_oracle import clip_adam
    torch.manual_seed(0)
    a = Gaussian_FF_Actor(37, 12).cuda()
    b = Gaussian_FF_Actor(37, 12).cuda()
    b.load_state_dict(a.state_dict())
    opt_a = FusedClipAdam(a, lr=3e-4, eps=1e-5, max_norm=0.05)
    opt_b = torch.optim.Adam(b.parameters(), lr=3e-4, eps=1e-5)
    p0 = opt_a.flat.double().cpu().numpy().copy()
    m = v = np.zeros_like(p0)
    p = p0
    x = torch.randn(64, 37, device="cuda")
    for step in range(1, 4):
        for net, opt in ((a, opt_a), (b, opt_b)):
            opt.zero_grad()
            (net(x).pow(2).mean() * 50).backward()
        g_np = opt_a.grad.double().cpu().numpy().copy()
        torch.nn.utils.clip_grad_norm_(b.parameters(), 0.05)
        opt_a.step()
        opt_b.step()
        p, m, v, tn = clip_adam(p, g_np, m, v, step, 3e-4, 1e-5, 0.05)
        assert abs(opt_a.total_norm().item() - tn) < 1e-4 * max(1, tn)
        flat_b = torch.cat([q.data.reshape(-1) for q in b.parameters()])
        assert (opt_a.flat - flat_b).abs().max().item() < 2e-6
        assert np.abs(opt_a.flat.double().cpu().numpy() - p).max() < 2e-6


# checkpoints of the training runs below go to a private directory (a fixed /tmp path may belong to another user), removed at exit
_LOGDIR = tempfile.TemporaryDirectory(prefix="lhw_test_logs_")


def _args(**kw):
    d = dict(gamma=0.99, lam=0.95, lr=3e-4, eps=1e-5, entropy_coeff=0.0, clip=0.2, minibatch_size=256, epochs=1,
             max_traj_len=50, num_procs=64, max_grad_norm=0.05, mirror_coeff=0.4, eval_freq=100, recurrent=False,
             imitate_coeff=0.0, std_dev=0.223, learn_std=False, logdir=_LOGDIR.name, steps_per_env=20)
    d.update(kw)
    return SimpleNamespace(**d)


def _env_fn(n=64, seed=0):
    from learninghumanoidwalking_b200.envs import BatchedHumanoidEnv
    from learninghumanoidwalking_b200.rl.symmetric import SymmetricEnv
    base = lambda: BatchedHumanoidEnv(n, precision=32, seed=seed)
    probe = base()
    r = probe.robot
    probe.close()
    return lambda: SymmetricEnv(base, mirrored_obs=r.mirrored_obs, mirrored_act=r.mirrored_acts, clock_inds=r.clock_inds)


def test_rollout_worker_contract_and_gae_consistency():
    """tests/test_training.py:79-129 contract + returns == GAE of the stored (rewards, values, boot)."""
    from learninghumanoidwalking_b200.rl import PPO, BatchData
    from oracle.ppo_oracle import gae_rollout
    ppo = PPO(_env_fn(), _args(), seed=0)
    batch = ppo.sample_parallel_with_workers()
    assert isinstance(batch, BatchData)
    n = 64 * 20
    assert batch.states.shape == (n, 37) and batch.actions.shape == (n, 12)
    for t in (batch.rewards, batch.values, batch.returns, batch.dones):
        assert t.shape == (n, 1) and torch.isfinite(t).all()
    buf = ppo.workers[0]._buf
    exp = gae_rollout(buf.rewards.double().cpu().numpy(), buf.values.double().cpu().numpy(), buf.ended.cpu().numpy(),
                      buf.boot.double().cpu().numpy(), buf.last_val.double().cpu().numpy(), 0.99, 0.95)
    assert np.abs(buf.returns.cpu().numpy() - exp).max() < 1e-4
    # env-major flattening: sample k of env e sits at e*T + k
    assert torch.equal(batch.states[3 * 20 + 5], buf.states[5, 3])
    # episodes persist across calls: traj_len keeps counting
    tl0 = ppo.env.state_i[:, 2].clone()
    ppo.sample_parallel_with_workers()
    assert (ppo.env.state_i[:, 2] != tl0).any()
    # completed episodes only
    assert batch.ep_lens.numel() == int(batch.dones.sum().item()) and (batch.ep_lens > 0).all()


def test_ppo_update_changes_weights_and_returns_seven_scalars(tmp_path):
    from learninghumanoidwalking_b200.rl import PPO
    ppo = PPO(_env_fn(), _args(logdir=str(tmp_path)), seed=1)
    ppo.make_optimizers()
    before = ppo._flat_param.clone()
    batch = ppo.sample_parallel_with_workers()
    adv = ppo.normalize_advantages(batch.returns.contiguous(), batch.values.contiguous())
    # the statistics left behind by the GAE launch of this batch (single 12 B/sample normalisation pass) give the same result
    adv_fused = ppo.normalize_advantages(batch.returns.contiguous(), batch.values.contiguous(), from_rollout=True)
    assert (adv - adv_fused).abs().max().item() < 1e-5 and abs(adv_fused.double().std().item() - 1) < 1e-4
    env = ppo.env
    out = ppo.update_actor_critic(batch.states[:256], batch.actions[:256], batch.returns[:256], adv[:256], 1,
                                  mirror_observation=env.mirror_clock_observation, mirror_action=env.mirror_action)
    assert len(out) == 7 and all(np.isfinite(float(s)) for s in out)
    assert not torch.equal(before, ppo._flat_param)
    log = ppo.train(None, 1, verbose=False)
    assert (tmp_path / "actor_0.pt").exists() and (tmp_path / "critic_0.pt").exists()
    assert np.isfinite(log[0]["critic_loss"])
    # the evaluation pass of iteration 0 (rl/algos/ppo.py:597-615): 5 deterministic batches, completed episodes only, and the
    # un-suffixed "best" pair next to the suffixed one (rl/utils/checkpointer.py:54-83)
    assert np.isfinite(log[0]["eval_rew"]) and 0 < log[0]["eval_len"] <= 50
    assert (tmp_path / "actor.pt").exists() and (tmp_path / "critic.pt").exists() and ppo._best_eval == log[0]["eval_rew"]
    best = torch.load(tmp_path / "actor.pt", weights_only=False)
    # checkpoints are self-contained CPU copies under the reference's class path (rl/policies/__init__.py: export_module)
    assert type(best).__module__ == "rl.policies.actor" and all(not p.is_cuda for p in best.parameters())
    assert list(best.state_dict()) == list(ppo.policy.state_dict())
    assert all(torch.equal(a, b.cpu()) for a, b in zip(best.state_dict().values(), ppo.policy.state_dict().values()))
    assert torch.equal(best.obs_mean, ppo.policy.obs_mean.cpu())
    actor = torch.load(tmp_path / "actor_0.pt", weights_only=False)
    assert actor(batch.states[:4].cpu()).shape == (4, 12) and actor.cuda()(batch.states[:4]).shape == (4, 12)


def test_same_seed_gives_bit_identical_weights():
    """tests/test_determinism.py:79-146: two runs, same seed => torch.equal on the final weights."""
    from learninghumanoidwalking_b200.rl import PPO
    finals = []
    for _ in range(2):
        ppo = PPO(_env_fn(seed=3), _args(), seed=3)
        ppo.train(None, 2, verbose=False)
        finals.append(ppo._flat_param.clone())
        ppo.env.close()
    assert torch.equal(finals[0], finals[1])


def test_fused_exchange_kernel_single_rank_matches_oracle_clip_adam():
    """lhw_fused_allreduce_clip_adam at world = 1: three launches = clip_grad_norm_ x2 + Adam x2 (rl/algos/ppo.py:393-396),
    the Adam step number kept in device memory; an odd length exercises the scalar tail after the 16-byte loads."""
    from learninghumanoidwalking_b200.rl.comm import PeerComm
    from oracle.ppo_oracle import clip_adam
    dev = torch.device("cuda", 0)
    n_a, n = 1001, 1703
    comm = PeerComm(n, dev)
    g = torch.Generator(device="cuda").manual_seed(0)
    p = torch.randn(n, device="cuda", generator=g)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    pa, ma, va = p[:n_a].double().cpu().numpy(), np.zeros(n_a), np.zeros(n_a)
    pc, mc, vc = p[n_a:].double().cpu().numpy(), np.zeros(n - n_a), np.zeros(n - n_a)
    for step in range(1, 4):
        comm.grad.copy_(torch.randn(n, device="cuda", generator=g) * (0.3 if step == 2 else 0.001))   # clipped and unclipped cases
        gnp = comm.grad.double().cpu().numpy()
        comm.fused_step(p, m, v, n_a, 3e-4, (0.9, 0.999), 1e-5, 0.05)
        done, norms = comm.status()
        assert done == step
        pa, ma, va, na = clip_adam(pa, gnp[:n_a], ma, va, step, 3e-4, 1e-5, 0.05)
        pc, mc, vc, nc = clip_adam(pc, gnp[n_a:], mc, vc, step, 3e-4, 1e-5, 0.05)
        assert abs(norms[0] - na) < 1e-5 * max(1, na) and abs(norms[1] - nc) < 1e-5 * max(1, nc)
        assert np.abs(p[:n_a].double().cpu().numpy() - pa).max() < 2e-6 and np.abs(p[n_a:].double().cpu().numpy() - pc).max() < 2e-6
    comm.close()


def test_ppo_loss_kernel_matches_the_closed_form_oracle():
    """lhw_ppo_loss against oracle/ppo_oracle.py: ppo_loss_and_grads (itself equal to torch autograd on the reference's
    formulation, tests/test_ppo_loss_oracle.py): 8 scalars and the three gradients, with and without the mirror term."""
    from oracle.ppo_oracle import ppo_loss_and_grads
    L = _lib()
    rng = np.random.RandomState(3)
    for B, with_mirr in ((21845, True), (300, False)):
        A = 12
        stds = np.full(A, 0.223, dtype=np.float32)
        mu = (rng.normal(size=(B, A)) * 0.2).astype(np.float32)
        old_mu = (mu + rng.normal(size=(B, A)) * 0.05).astype(np.float32)
        act = (old_mu + rng.normal(size=(B, A)) * 0.223).astype(np.float32)
        adv, ret, val = (rng.normal(size=(B, 1)).astype(np.float32) for _ in range(3))
        mirr = (mu + rng.normal(size=(B, A)) * 0.05).astype(np.float32) if with_mirr else None
        d = lambda a: None if a is None else torch.as_tensor(a, device="cuda")
        g_mu, g_mirr, g_val = torch.empty(B, A, device="cuda"), torch.empty(B, A, device="cuda"), torch.empty(B, 1, device="cuda")
        part = torch.zeros(L.lib().lhw_ppo_loss_partial_words(B), dtype=torch.float64, device="cuda")
        ticket, out8 = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(8, device="cuda")
        for _ in range(2):      # twice: the ticket counter must come back to zero
            L.ops().ppo_loss(d(mu), d(old_mu), d(act), d(adv), d(ret), d(val), d(mirr), d(stds), 0.2, 0.4, 0.01, g_mu,
                             g_mirr if with_mirr else None, g_val, part, ticket, out8)
        exp = ppo_loss_and_grads(mu, old_mu, act, adv, ret, val, mirr, stds, 0.2, 0.4, 0.01)
        assert np.abs(out8.cpu().numpy() - exp[0]).max() < 2e-5 and int(ticket.item()) == 0
        assert 0.02 < exp[0][6] < 0.98
        assert np.abs(g_mu.cpu().numpy() - exp[1]).max() < 1e-6 * max(1.0, np.abs(exp[1]).max() * B)
        assert np.abs(g_mu.cpu().numpy() - exp[1]).max() < 2e-5 * np.abs(exp[1]).max()
        assert np.abs(g_val.cpu().numpy().reshape(-1) - exp[3]).max() < 2e-6 * np.abs(exp[3]).max() + 1e-12
        if with_mirr:
            assert np.abs(g_mirr.cpu().numpy() - exp[2]).max() < 2e-6 * np.abs(exp[2]).max() + 1e-12


def test_fused_loss_kernel_matches_the_torch_loss_graph(monkeypatch):
    """lhw_ppo_loss (forward + backward of the loss tail in one launch) against the torch graph it replaces
    (rl/algos/ppo.py:302-386 restated with autograd): the 7 scalars and the weights after one and two optimiser steps."""
    from learninghumanoidwalking_b200.rl import PPO
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("LHW_FUSED_LOSS", mode)
        monkeypatch.setenv("LHW_UPDATE_GRAPH", "0")
        ppo = PPO(_env_fn(seed=8), _args(), seed=8)
        ppo.make_optimizers()
        batch = ppo.sample_parallel_with_workers()
        adv = ppo.normalize_advantages(batch.returns.contiguous(), batch.values.contiguous())
        env = ppo.env
        outs = []
        for k in range(2):
            sl = slice(300 * k, 300 * k + 300)      # 300: not a multiple of the kernel's block size
            o = ppo.update_actor_critic(batch.states[sl].contiguous(), batch.actions[sl].contiguous(), batch.returns[sl].contiguous(),
                                        (adv[sl] * (3.0 if k else 1.0)).contiguous(), 1,     # larger advantages: some ratios leave the clip range
                                        mirror_observation=env.mirror_clock_observation, mirror_action=env.mirror_action)
            outs.append(torch.stack([x.float() for x in o]).cpu())
        res[mode] = (outs, ppo._flat_param.clone().cpu())
        ppo.env.close()
    for a, b in zip(res["0"][0], res["1"][0]):
        assert (a - b).abs().max().item() < 2e-5 * max(1.0, a.abs().max().item()), (a, b)
    assert (res["0"][1] - res["1"][1]).abs().max().item() < 2e-6
    assert res["1"][0][1][6] > 0 or res["1"][0][1][3].abs() > 0      # the second step really moved the ratio away from 1


def test_rollout_graph_follows_the_weights_after_make_optimizers():
    """The public sequence PPO(...); sample_parallel_with_workers(); train() (the reference's tests use it): the rollout
    graph captured by the first call holds the parameter addresses of BEFORE make_optimizers() re-homes them into the flat
    buffer.  It must be dropped then, otherwise the sampler keeps acting on weights the learner never touches."""
    from learninghumanoidwalking_b200.rl import PPO
    ppo = PPO(_env_fn(seed=6), _args(), seed=6)
    b0 = ppo.sample_parallel_with_workers(deterministic=True)
    assert b0.actions.abs().max().item() > 0
    ppo.make_optimizers()
    with torch.no_grad():
        ppo._flat_param.zero_()            # all-zero weights and biases: the deterministic action is exactly 0
    b1 = ppo.sample_parallel_with_workers(deterministic=True)
    assert b1.actions.abs().max().item() == 0 and b1.values.abs().max().item() == 0
    ppo.env.close()


def test_graph_replayed_rollout_is_bitwise_equal_to_the_eager_loop(monkeypatch):
    """DeviceRolloutWorker.sample replays one captured control step (policy + critic + lhw_sim_step + buffer writes);
    the eager loop must give bit-identical batches."""
    from learninghumanoidwalking_b200.rl import PPO
    outs = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("LHW_ROLLOUT_GRAPH", mode)
        ppo = PPO(_env_fn(seed=4), _args(), seed=4)
        b1 = ppo.sample_parallel_with_workers()
        b2 = ppo.sample_parallel_with_workers()            # second call: pure replay path
        outs[mode] = [t.clone() for b in (b1, b2) for t in (b.states, b.actions, b.rewards, b.values, b.returns, b.dones)]
        ppo.env.close()
    for a, b in zip(outs["1"], outs["0"]):
        assert torch.equal(a, b)


def test_two_stream_rollout_halves_equal_the_eager_loop_and_track_the_single_stream_rollout(monkeypatch):
    """Batches of >= 1024 environments advance as two halves on two streams (DeviceRolloutWorker._parts).  The replayed graphs
    must give bit-identical batches to the eager loop over the same halves, two calls in a row (episodes persist), and the same
    environment trajectories as the single-stream rollout up to the MLP's batch-size-dependent rounding."""
    from learninghumanoidwalking_b200.rl import PPO
    outs = {}
    for name, graph, split in (("graph", "1", "1"), ("eager", "0", "1"), ("single", "1", "0")):
        monkeypatch.setenv("LHW_ROLLOUT_GRAPH", graph)
        monkeypatch.setenv("LHW_ROLLOUT_SPLIT", split)
        ppo = PPO(_env_fn(n=2048, seed=4), _args(num_procs=2048, steps_per_env=12), seed=4)
        assert len(ppo.workers[0]._parts(2048)) == (2 if split == "1" else 1)
        b1 = ppo.sample_parallel_with_workers()
        b2 = ppo.sample_parallel_with_workers()
        outs[name] = [t.clone() for b in (b1, b2) for t in (b.states, b.actions, b.rewards, b.values, b.returns, b.dones)]
        ppo.env.close()
    for a, b in zip(outs["graph"], outs["eager"]):
        assert torch.equal(a, b)
    # first call, first few steps: the single-stream rollout sees the same environments (same seeds, same noise stream)
    st_g, st_s = outs["graph"][0].view(2048, 12, -1), outs["single"][0].view(2048, 12, -1)
    assert (st_g[:, :4] - st_s[:, :4]).abs().max().item() < 1e-3
    assert torch.equal(outs["graph"][5].view(2048, 12)[:, :4], outs["single"][5].view(2048, 12)[:, :4])


def test_two_envs_of_one_variant_with_different_constants_can_alternate_graph_replays(tmp_path):
    """The model constants of a (variant, precision) live in ONE __constant__ object per process.  Two environments of the same
    variant with different constants (here: PD gains from a YAML) whose captured rollout graphs are replayed alternately must
    each see their own constants (DeviceRolloutWorker binds the env's model before it replays): alternating gives bit-identical
    batches to running each worker alone."""
    from learninghumanoidwalking_b200.envs import BatchedHumanoidEnv
    from learninghumanoidwalking_b200.rl import DeviceRolloutWorker, FF_V, Gaussian_FF_Actor
    soft = tmp_path / "soft.yaml"
    soft.write_text("kp: [100, 100, 100, 125, 40, 40, 100, 100, 100, 125, 40, 40]\n")

    def worker(yaml):
        env = BatchedHumanoidEnv(64, precision=32, seed=3, path_to_yaml=yaml)
        torch.manual_seed(5)
        pol, cri = Gaussian_FF_Actor(37, 12, init_std=0.223).cuda(), FF_V(37).cuda()
        pol.obs_mean = cri.obs_mean = torch.tensor(env.obs_mean, dtype=torch.float32, device="cuda")
        pol.obs_std = cri.obs_std = torch.tensor(env.obs_std, dtype=torch.float32, device="cuda")
        return DeviceRolloutWorker(env, pol, cri, seed=9)

    grab = lambda b: [t.clone() for t in (b.states, b.actions, b.rewards, b.returns, b.dones)]
    alone = {}
    for name, y in (("a", None), ("b", soft)):
        w = worker(y)
        alone[name] = [grab(w.sample(0.99, 0.95, 6, 50)) for _ in range(2)]
        w.env.close()
    wa, wb = worker(None), worker(soft)
    inter = {"a": [], "b": []}
    for _ in range(2):
        inter["a"].append(grab(wa.sample(0.99, 0.95, 6, 50)))
        inter["b"].append(grab(wb.sample(0.99, 0.95, 6, 50)))
    for name in ("a", "b"):
        for x, y in zip(alone[name], inter[name]):
            assert all(torch.equal(p, q) for p, q in zip(x, y)), name
    assert not torch.equal(alone["a"][0][0], alone["b"][0][0])      # the YAML really changed the dynamics
    wa.env.close(); wb.env.close()


def test_graph_replayed_update_matches_the_eager_update(monkeypatch):
    """PPO._update_step: after three eager warm-up updates the optimiser step (losses, backward, clip + Adam with the step
    counter in device memory) is captured once and replayed; same seed, same data => the same weights as the eager loop."""
    from learninghumanoidwalking_b200.rl import PPO
    finals, logs = {}, {}
    for mode in ("0", "1"):
        monkeypatch.setenv("LHW_UPDATE_GRAPH", mode)
        # eval_batches=0: the two modes differ in the last bits of the first update (bias correction on the host vs on the device);
        # 100 deterministic control steps of evaluation between that update and the next batch would only amplify them
        ppo = PPO(_env_fn(seed=4), _args(epochs=2, eval_batches=0), seed=4)
        logs[mode] = ppo.train(None, 2, verbose=False)
        finals[mode] = ppo._flat_param.clone()
        if mode == "1":
            assert ppo._ug is not None                              # the graph was really captured and used
            assert ppo.actor_optimizer.step_count == ppo._comm.status()[0] == 20
        else:
            assert ppo._ug is None
        ppo.env.close()
    assert (finals["0"] - finals["1"]).abs().max().item() < 1e-6
    assert abs(logs["0"][-1]["critic_loss"] - logs["1"][-1]["critic_loss"]) < 1e-5
