"""Fused PPO minibatch step (csrc/ppo_update.cu, SURVEY.md s8 f.1) against PyTorch autograd / torch.optim.Adam on the same
minibatches: the oracle here is the reference's own arithmetic (ppo_continuous.py:216-239) run by PyTorch in fp32."""
import copy
import os
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _args(use_tanh=1, clip=True, K=2, mb=512, B=1500):
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=mb, max_train_steps=int(3e6),
                                 lr_a=2e-4, lr_c=2e-4, gamma=0.99, lamda=0.95, epsilon=0.1, K_epochs=K, entropy_coef=0.01,
                                 set_adam_eps=True, use_grad_clip=clip, use_lr_decay=True, use_adv_norm=True, state_dim=18,
                                 action_dim=3, hidden_width=256, use_tanh=use_tanh, use_orthogonal_init=True, chkpt_dir="/tmp")


def _pair(args, gain_boost=True):
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    torch.manual_seed(0)
    a = P.PPO_continuous(args, "pursuer")
    b = P.PPO_continuous(args, "pursuer")
    with torch.no_grad():
        if gain_boost:                      # the 0.01-gain head gives near-zero means; make the policy output matter
            a.actor.mean_layer.weight.mul_(30.0)
            a.actor.log_std.copy_(torch.tensor([[-0.3, 0.1, 0.2]]))
    b.actor.load_state_dict(a.actor.state_dict()); b.critic.load_state_dict(a.critic.state_dict())
    return a, b


def _data(agent, B, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    s = torch.randn(B, 18, device="cuda", generator=g)
    with torch.no_grad():
        dist = agent.actor.get_dist(s)
        act = torch.clamp(dist.mean + dist.stddev * torch.randn(B, 3, device="cuda", generator=g), -1.6, 1.6)
        logp = dist.log_prob(act) + 0.06 * torch.randn(B, 3, device="cuda", generator=g)      # ratios on both sides of the clip
    adv = torch.randn(B, 1, device="cuda", generator=g)
    vt = torch.randn(B, 1, device="cuda", generator=g)
    return s, act, logp, adv, vt


def _flat_grads(module, names):
    named = dict(module.named_parameters())
    return torch.cat([named[k].grad.reshape(-1) for k in names])


@pytest.fixture(params=[1, 0], ids=["tensor-cores", "ffma2"])
def fb_path(request):
    """both forward/backward implementations of the fused step: csrc/ppo_fb_tc.cu + ppo_wgrad2_tc.cu (default) and the fp32
    FFMA2 kernels of csrc/ppo_update.cu"""
    from ppo_rl_satellite_b200 import _lib as L
    lib = L.load()
    prev = lib.sat_ppo_use_tensor_cores(request.param)
    yield request.param
    lib.sat_ppo_use_tensor_cores(prev)


@pytest.mark.parametrize("use_tanh,mb", [(1, 1000), (0, 1000), (1, 64), (1, 37), (1, 300)])
def test_fused_gradients_match_autograd(use_tanh, mb, fb_path):
    from ppo_rl_satellite_b200 import engine as E
    args = _args(use_tanh=use_tanh)
    fused, eager = _pair(args)
    B = 1500
    s, act, logp, adv, vt = _data(eager, B)
    index = torch.randperm(B, device="cuda")[:mb].contiguous()
    # --- autograd (the reference's loss, :217-228 and :232-235)
    dist_now = eager.actor.get_dist(s[index])
    ent = dist_now.entropy().sum(1, keepdim=True)
    ratios = torch.exp(dist_now.log_prob(act[index]).sum(1, keepdim=True) - logp[index].sum(1, keepdim=True))
    assert ((ratios < 0.9).sum() > 0 and (ratios > 1.1).sum() > 0) or mb < 100
    surr1 = ratios * adv[index]
    surr2 = torch.clamp(ratios, 0.9, 1.1) * adv[index]
    la = (-torch.min(surr1, surr2) - 0.01 * ent).mean()
    la.backward()
    lc = torch.nn.functional.mse_loss(vt[index], eager.critic(s[index]))
    lc.backward()
    # --- fused kernels
    f = fused._fused_for(mb)
    na, nc = f["nets"]
    na.actor_grad(s, act, logp, adv.reshape(-1), index.data_ptr(), mb, 0.1, 0.01)
    nc.critic_grad(s, vt.reshape(-1), index.data_ptr(), mb)
    torch.cuda.synchronize()
    for net, module, names, loss in ((na, eager.actor, E.PpoFusedNet.ACTOR_NAMES, la), (nc, eager.critic, E.PpoFusedNet.CRITIC_NAMES, lc)):
        ref = _flat_grads(module, names)
        got = net.grads[:net.n]
        scale = ref.abs().max().item()
        assert scale > 0
        err = (got - ref).abs().max().item()
        assert err <= 2e-5 * scale + 1e-9, (err, scale)
        assert abs(net.grads[net.n].item() - loss.item()) <= 1e-5 * max(1.0, abs(loss.item()))


@pytest.mark.parametrize("use_tanh,clip", [(1, True), (0, False)])
def test_fused_optimize_tracks_torch_adam(use_tanh, clip):
    args = _args(use_tanh=use_tanh, clip=clip, K=2, mb=512)
    fused, eager = _pair(args)
    B = 1500
    s, act, logp, adv, vt = _data(eager, B)
    for it in range(2):
        torch.manual_seed(100 + it)
        eager.optimize(s, act, logp, adv, vt, mini_batch_size=512)
        torch.manual_seed(100 + it)                                   # same randperm sequence
        fused.optimize(s, act, logp, adv, vt, mini_batch_size=512, fused=True)
    torch.cuda.synchronize()
    assert int(fused._fused["nets"][0].step.item()) == 2 * 2 * 3       # 2 calls x K=2 x ceil(1500/512)
    for me, mf in ((eager.actor, fused.actor), (eager.critic, fused.critic)):
        for (k, pe), (_, pf) in zip(me.named_parameters(), mf.named_parameters()):
            d = (pe - pf).abs()
            assert d.max().item() <= 3e-5, (k, d.max().item())
            assert d.mean().item() <= 2e-6, (k, d.mean().item())
    # the parameters did move (12 Adam steps of 2e-4), so the comparison above is not vacuous
    fresh = _pair(args)[0]
    assert (fresh.actor.fc2.weight - fused.actor.fc2.weight).abs().mean().item() > 2e-4


def test_fused_step_feeds_the_sampling_kernel_and_checkpoints():
    """after a fused update the actor/critic kernels and the torch modules see the same weights"""
    args = _args(K=1, mb=512)
    fused, _ = _pair(args, gain_boost=False)
    s, act, logp, adv, vt = _data(fused, 1024)
    fused.optimize(s, act, logp, adv, vt, mini_batch_size=512, fused=True)
    assert fused._dirty is False
    obs = s[:200].contiguous()
    eps = torch.zeros(200, 3, device="cuda")
    a_k, _ = fused.actor_kernel.sample(obs=obs, eps_in=eps)
    v_k = fused.critic_kernel.value(obs)
    with torch.no_grad():
        np.testing.assert_allclose(a_k.cpu().numpy(), fused.actor(obs).cpu().numpy(), atol=2e-6)
        np.testing.assert_allclose(v_k.cpu().numpy(), fused.critic(obs).reshape(-1).cpu().numpy(), atol=5e-6)
    # loading a checkpoint into the torch views is picked up by sync_kernels (device-side repack)
    sd = {k: v.clone() for k, v in fused.actor.state_dict().items()}
    sd["mean_layer.bias"] = sd["mean_layer.bias"] + 0.25
    fused.actor.load_state_dict(sd)
    fused._dirty = True
    fused.sync_kernels()
    a_k2, _ = fused.actor_kernel.sample(obs=obs, eps_in=eps)
    with torch.no_grad():
        np.testing.assert_allclose(a_k2.cpu().numpy(), fused.actor(obs).cpu().numpy(), atol=2e-6)
    assert (a_k2 - a_k).abs().max().item() > 1e-3


def test_fused_argument_errors():
    from ppo_rl_satellite_b200 import _lib as L
    import ctypes as C
    lib = L.load()
    net = L.SatPpoNet()
    assert lib.sat_ppo_adam(C.byref(net), None, 0.9, 0.999, 1e-5, 0.5, 1.0, None, None) == -1
    assert lib.sat_ppo_workspace_floats(0) == 0 and lib.sat_ppo_workspace_floats(64) > 74 * 65536


def test_vector_trainer_fused_update_resumes_exactly(tmp_path):
    """full-run checkpoint (env state, normalisers, Philox counter, weights, fused Adam moments + step): the resumed run
    reproduces the uninterrupted one bit for bit (the fused step sums in a fixed order)"""
    from ppo_rl_satellite_b200 import engine as eng, rollout
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    n, T, mb = 256, 8, 512

    def make():
        torch.manual_seed(0)
        args = _args(K=2, mb=mb, B=n * T)
        env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=5, auto_reset=True)
        agent, opp = P.PPO_continuous(args, "pursuer"), P.PPO_continuous(args, "evader")
        return rollout.VectorTrainer(env, agent, opp, T)

    a = make()
    a.collect(); torch.manual_seed(5); a.update(mb, total_steps=1000)
    sd = copy.deepcopy(a.state_dict())            # module state_dicts alias the live parameters
    assert sd["fused_adam"] is not None and int(sd["fused_adam"][0]["step"].item()) == 2 * 4
    a.collect(); torch.manual_seed(6); a.update(mb, total_steps=2000)
    b = make().load_state_dict(sd)
    b.collect(); torch.manual_seed(6); b.update(mb, total_steps=2000)
    for pa, pb in zip(list(a.agent.actor.parameters()) + list(a.agent.critic.parameters()),
                      list(b.agent.actor.parameters()) + list(b.agent.critic.parameters())):
        assert torch.equal(pa, pb)
    assert torch.equal(a.buf.act, b.buf.act) and torch.equal(a.buf.rew64, b.buf.rew64)


# ---------------------------------------------------------------- two ranks (gloo carrying CUDA tensors, both on cuda:0)
def _rank_worker(rank, world, port, q):
    import os, sys
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        args = _args(K=3, mb=512, B=512)
        agent, _ = _pair(args)
        s, act, logp, adv, vt = _data(agent, 1024)                    # same 1024 rows on both ranks; each trains on its half
        lo = rank * 512
        agent.optimize(s[lo:lo + 512], act[lo:lo + 512], logp[lo:lo + 512], adv[lo:lo + 512], vt[lo:lo + 512],
                       mini_batch_size=512, fused=True)
        torch.cuda.synchronize()
        flat = torch.cat([p.detach().reshape(-1) for p in list(agent.actor.parameters()) + list(agent.critic.parameters())])
        q.put((rank, flat.cpu().numpy()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_ranks_average_gradients_like_one_rank_on_the_union():
    """world 2, one full-batch step per epoch: averaging the two ranks' mean-gradients == the gradient of the union batch,
    so both ranks must end on the parameters a single process reaches with the 1024-row batch."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=240) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert np.array_equal(res[0], res[1])                              # replicas stay identical
    args = _args(K=3, mb=1024, B=1024)
    agent, _ = _pair(args)
    s, act, logp, adv, vt = _data(agent, 1024)
    agent.optimize(s, act, logp, adv, vt, mini_batch_size=1024, fused=True)
    one = torch.cat([p.detach().reshape(-1) for p in list(agent.actor.parameters()) + list(agent.critic.parameters())]).cpu().numpy()
    assert np.abs(res[0] - one).max() <= 3e-5 and np.abs(res[0] - one).mean() <= 2e-6
    assert np.abs(one - torch.cat([p.detach().reshape(-1) for p in list(_pair(args)[0].actor.parameters())
                                   + list(_pair(args)[0].critic.parameters())]).cpu().numpy()).mean() > 1e-4


def _nccl_peer_worker(rank, world, port, q):
    import os, sys
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), SAT_PEER_ALLREDUCE="1")
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        from ppo_rl_satellite_b200.dropin import ppo_continuous as P
        args = _args(K=3, mb=512, B=512)
        torch.manual_seed(0)
        agent = P.PPO_continuous(args, "pursuer", device=dev)
        with torch.no_grad():
            agent.actor.mean_layer.weight.mul_(30.0)
            agent.actor.log_std.copy_(torch.tensor([[-0.3, 0.1, 0.2]], device=dev))
        g = torch.Generator(device=dev).manual_seed(1)                 # same 1024 rows on both ranks; each trains on its half
        s = torch.randn(1024, 18, device=dev, generator=g)
        with torch.no_grad():
            d_ = agent.actor.get_dist(s)
            act = torch.clamp(d_.mean + d_.stddev * torch.randn(1024, 3, device=dev, generator=g), -1.6, 1.6)
            logp = d_.log_prob(act) + 0.06 * torch.randn(1024, 3, device=dev, generator=g)
        adv = torch.randn(1024, 1, device=dev, generator=g); vt = torch.randn(1024, 1, device=dev, generator=g)
        lo = rank * 512
        agent.optimize(s[lo:lo + 512], act[lo:lo + 512], logp[lo:lo + 512], adv[lo:lo + 512], vt[lo:lo + 512], mini_batch_size=512, fused=True)
        torch.cuda.synchronize()
        peers = any(agent._fused["peers"].values())
        flat = torch.cat([p.detach().reshape(-1) for p in list(agent.actor.parameters()) + list(agent.critic.parameters())])
        # unequal per-rank batches must be refused on every rank instead of dead-locking
        refused = False
        try:
            agent.optimize(s[:512 - 64 * rank], act[:512 - 64 * rank], logp[:512 - 64 * rank], adv[:512 - 64 * rank],
                           vt[:512 - 64 * rank], mini_batch_size=128, fused=True)
        except ValueError:
            refused = True
        q.put((rank, flat.cpu().numpy(), peers, refused))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_gpus_nccl_peer_memory_gradient_exchange():
    """2 GPUs, NCCL process group: the gradient exchange fused into the Adam kernel over NVLink peer memory
    (sat_ppo_adam_peers, torch symmetric memory) gives bit-identical replicas that match one rank on the union batch."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29900 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_nccl_peer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = {r: (f, pe, rf) for r, f, pe, rf in (q.get(timeout=240) for _ in procs)}
    for p in procs:
        p.join(timeout=60)
    assert res[0][1] and res[1][1], "the peer-memory path was not taken"
    assert res[0][2] and res[1][2], "unequal per-rank batches were not refused"
    assert np.array_equal(res[0][0], res[1][0])
    args = _args(K=3, mb=1024, B=1024)
    agent, _ = _pair(args)
    s, act, logp, adv, vt = _data(agent, 1024)
    agent.optimize(s, act, logp, adv, vt, mini_batch_size=1024, fused=True)
    one = torch.cat([p.detach().reshape(-1) for p in list(agent.actor.parameters()) + list(agent.critic.parameters())]).cpu().numpy()
    assert np.abs(res[0][0] - one).max() <= 3e-5


@pytest.mark.timeout(300)
def test_tensor_core_and_ffma2_paths_agree_on_a_multi_tile_minibatch():
    """the persistent tensor-core kernels with several row tiles per CTA (148 x 128 x 2 + 37 rows: three tiles on some CTAs, a
    ragged last tile; dW2 slabs of unequal length) against the fp32 FFMA2 kernels on the same minibatch"""
    from ppo_rl_satellite_b200 import _lib as L
    lib = L.load()
    mb = 148 * 128 * 2 + 37
    args = _args(use_tanh=1, mb=mb, B=mb + 500)
    fused, eager = _pair(args)
    s, act, logp, adv, vt = _data(eager, mb + 500)
    index = torch.randperm(mb + 500, device="cuda")[:mb].contiguous()
    f = fused._fused_for(mb)
    na, nc = f["nets"]
    prev = lib.sat_ppo_use_tensor_cores(-1)
    got = {}
    try:
        for tc in (0, 1):
            lib.sat_ppo_use_tensor_cores(tc)
            na.actor_grad(s, act, logp, adv.reshape(-1), index.data_ptr(), mb, 0.1, 0.01)
            nc.critic_grad(s, vt.reshape(-1), index.data_ptr(), mb)
            torch.cuda.synchronize()
            got[tc] = (na.grads.clone(), nc.grads.clone())
    finally:
        lib.sat_ppo_use_tensor_cores(prev)
    for a, b in zip(got[0], got[1]):
        scale = a.abs().max().item()
        assert scale > 0
        assert (a - b).abs().max().item() <= 2e-6 * scale + 1e-9
