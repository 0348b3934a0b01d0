"""Training diagnostics of the fused PPO step (sat_ppo_actor_grad_stats, sat_ppo_adam_stats / _peers_stats, PpoUpdateStats) and
the epoch-granular early stop on approximate KL: the statistics against PyTorch on the same rows (the reference's formulas,
ppo_continuous.py:216-224), gradients and parameters bit-identical to the default kernels, early stop, two ranks, path
independence, rollout and self-play."""
import os
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

EPS, ENT_COEF, CLIP = 0.1, 0.01, 0.5
LOSS, SURR, ENT, KL, CLIPF, NORM, COEF, COUNT = range(8)


def _args(use_tanh=1, clip=True, K=2, mb=512, B=1500, lr=2e-4):
    return types.SimpleNamespace(policy_dist="Gaussian", max_action=1.6, batch_size=B, mini_batch_size=mb, max_train_steps=int(3e6),
                                 lr_a=lr, lr_c=lr, gamma=0.99, lamda=0.95, epsilon=EPS, K_epochs=K, entropy_coef=ENT_COEF,
                                 set_adam_eps=True, use_grad_clip=clip, use_lr_decay=True, use_adv_norm=True, state_dim=18,
                                 action_dim=3, hidden_width=256, use_tanh=use_tanh, use_orthogonal_init=True, chkpt_dir="/tmp")


def _agent(args, device="cuda"):
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    torch.manual_seed(0)
    a = P.PPO_continuous(args, "pursuer", device=device)
    with torch.no_grad():                   # the 0.01-gain head gives near-zero means; make the policy output matter
        a.actor.mean_layer.weight.mul_(30.0)
        a.actor.log_std.copy_(torch.tensor([[-0.3, 0.1, 0.2]], device=device))
    return a


def _data(agent, B, seed=1, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    s = torch.randn(B, 18, device=device, generator=g)
    with torch.no_grad():
        dist = agent.actor.get_dist(s)
        act = torch.clamp(dist.mean + dist.stddev * torch.randn(B, 3, device=device, generator=g), -1.6, 1.6)
        logp = dist.log_prob(act) + 0.06 * torch.randn(B, 3, device=device, generator=g)      # ratios on both sides of the clip
    adv = torch.randn(B, 1, device=device, generator=g)
    vt = torch.randn(B, 1, device=device, generator=g)
    return s, act, logp, adv, vt


@pytest.fixture(params=[1, 0], ids=["tensor-cores", "ffma2"])
def fb_path(request):
    from ppo_rl_satellite_b200 import _lib as L
    lib = L.load()
    prev = lib.sat_ppo_use_tensor_cores(request.param)
    yield request.param
    lib.sat_ppo_use_tensor_cores(prev)


def _torch_stats(agent, s, act, logp, adv, vt):
    """the reference's minibatch arithmetic in fp32 (autograd, clip_grad_norm_'s return value) and the KL with fp64 log-probs;
    scale: mean |term| of the surrogate (its mean can be near zero)"""
    d = agent.actor.get_dist(s)
    ent = d.entropy().sum(1, keepdim=True)
    lr = d.log_prob(act).sum(1, keepdim=True) - logp.sum(1, keepdim=True)
    ratios = torch.exp(lr)
    surr1, surr2 = ratios * adv, torch.clamp(ratios, 1 - EPS, 1 + EPS) * adv
    la = (-torch.min(surr1, surr2) - ENT_COEF * ent).mean()
    agent.actor.zero_grad(); la.backward()
    na = torch.nn.utils.clip_grad_norm_(agent.actor.parameters(), float("inf"))
    lc = torch.nn.functional.mse_loss(vt, agent.critic(s))
    agent.critic.zero_grad(); lc.backward()
    nc = torch.nn.utils.clip_grad_norm_(agent.critic.parameters(), float("inf"))
    with torch.no_grad():
        std = torch.exp(agent.actor.log_std).double()
        l64 = (torch.distributions.Normal(agent.actor(s).double(), std).log_prob(act.double()).sum(1) - logp.double().sum(1))
        return {"loss": la.item(), "surrogate": (-torch.min(surr1, surr2)).mean().item(),
                "surrogate_scale": torch.min(surr1, surr2).abs().mean().item(), "entropy": ent.mean().item(),
                "approx_kl": (torch.expm1(l64) - l64).mean().item(),
                "clip_fraction": ((ratios - 1.0).abs() > EPS).float().mean().item(),
                "value_loss": lc.item(), "actor_grad_norm": na.item(), "critic_grad_norm": nc.item()}


def _close(got, ref, rel, scale=None):
    return abs(got - ref) <= rel * max(abs(ref), scale or 0.0, 1e-12)


def _check_means(d, ref, mb, scale=None):
    """d: policy_loss, entropy, approx_kl, clip_fraction, value_loss, actor/critic_grad_norm (as_dict keys)"""
    assert _close(d["policy_loss"], ref["surrogate"], 1e-5, scale or 1e-6), (d["policy_loss"], ref["surrogate"])
    assert _close(d["entropy"], ref["entropy"], 1e-5), (d["entropy"], ref["entropy"])
    assert _close(d["value_loss"], ref["value_loss"], 1e-5), (d["value_loss"], ref["value_loss"])
    assert _close(d["approx_kl"], ref["approx_kl"], 1e-3), (d["approx_kl"], ref["approx_kl"])
    assert abs(d["clip_fraction"] - ref["clip_fraction"]) <= 2.0 / mb + 1e-4, (d["clip_fraction"], ref["clip_fraction"])
    assert _close(d["actor_grad_norm"], ref["actor_grad_norm"], 1e-4), (d["actor_grad_norm"], ref["actor_grad_norm"])
    assert _close(d["critic_grad_norm"], ref["critic_grad_norm"], 1e-4), (d["critic_grad_norm"], ref["critic_grad_norm"])


def _record_means(rec):
    """[2][8] record of one or more minibatches -> as_dict-style means"""
    a, c = rec[0] / rec[0][COUNT], rec[1] / rec[1][COUNT]
    return {"policy_loss": a[SURR], "entropy": a[ENT], "approx_kl": a[KL], "clip_fraction": a[CLIPF], "value_loss": c[LOSS],
            "actor_grad_norm": a[NORM], "critic_grad_norm": c[NORM]}


# ---------------------------------------------------------------- 1 + 2: one minibatch against PyTorch, gradient bits
@pytest.mark.parametrize("mb", [37, 1000, 65536, 148 * 128 * 2 + 37])
def test_minibatch_statistics_match_torch_and_gradients_are_unchanged(mb, fb_path):
    args = _args(mb=mb, B=mb + 500)
    fused, eager = _agent(args), _agent(args)
    B = mb + 500
    s, act, logp, adv, vt = _data(eager, B)
    index = torch.randperm(B, device="cuda")[:mb].contiguous()
    ref = _torch_stats(eager, s[index], act[index], logp[index], adv[index], vt[index])
    na, nc = fused._fused_for(mb)["nets"]
    na.actor_grad(s, act, logp, adv.reshape(-1), index.data_ptr(), mb, EPS, ENT_COEF)
    plain = na.grads[:na.n + 1].clone()
    na.actor_grad(s, act, logp, adv.reshape(-1), index.data_ptr(), mb, EPS, ENT_COEF, stats=True)
    nc.critic_grad(s, vt.reshape(-1), index.data_ptr(), mb)
    torch.cuda.synchronize()
    assert torch.equal(na.grads[:na.n + 1], plain)
    rec = torch.zeros((2, 8), dtype=torch.float64, device="cuda")
    na.adam(CLIP, 1.0, record=rec[0]); nc.adam(CLIP, 1.0, record=rec[1])
    rec = rec.cpu().numpy()
    assert rec[0][COUNT] == 1 and rec[1][COUNT] == 1
    assert _close(rec[0][LOSS], ref["loss"], 1e-5, ref["surrogate_scale"])
    _check_means(_record_means(rec), ref, mb, ref["surrogate_scale"])
    for k in (0, 1):
        norm = rec[k][NORM]
        assert _close(rec[k][COEF], min(CLIP / (norm + 1e-6), 1.0), 1e-6)
    assert (rec[1][SURR:CLIPF + 1] == 0).all()


def test_stats_argument_errors():
    import ctypes as C
    from ppo_rl_satellite_b200 import _lib as L
    lib = L.load()
    net = L.SatPpoNet()
    assert lib.sat_ppo_adam_stats(C.byref(net), None, 0.9, 0.999, 1e-5, 0.5, 1.0, None, None, None) == -1
    assert lib.sat_ppo_adam_peers_stats(C.byref(net), None, 0.9, 0.999, 1e-5, 0.5, 1.0, None, None, 1, 0, None, None) == -1
    assert lib.sat_ppo_actor_grad_stats(C.byref(net), None, None, None, None, None, 10, 0.1, 0.01, None) == -1
    args = _args()
    na, _ = _agent(args)._fused_for(64)["nets"]
    assert lib.sat_ppo_adam_stats(C.byref(na.net), na.lr.data_ptr(), 0.9, 0.999, 1e-5, 0.5, 1.0, na.step.data_ptr(), None,
                                  None) == -1                                   # the record is required


# ---------------------------------------------------------------- 3 + 4: optimisation bits, early stop
def _state(agent):
    nets = agent._fused["nets"]
    return [p.detach().clone() for p in list(agent.actor.parameters()) + list(agent.critic.parameters())] + \
           [t.clone() for n in nets for t in (n.exp_avg, n.exp_avg_sq, n.step)]


def _equal_states(x, y):
    return len(x) == len(y) and all(torch.equal(a, b) for a, b in zip(x, y))


@pytest.mark.parametrize("clip", [True, False])
def test_optimize_with_stats_is_bit_identical(clip, fb_path):
    args = _args(clip=clip, K=3, mb=512, B=1500)
    runs = []
    for stats in (False, True):
        agent = _agent(args)
        s, act, logp, adv, vt = _data(agent, 1500)
        torch.manual_seed(100)
        out = agent.optimize(s, act, logp, adv, vt, mini_batch_size=512, fused=True, stats=stats)
        torch.cuda.synchronize()
        runs.append((_state(agent), out))
    assert runs[0][1] is None
    assert _equal_states(runs[0][0], runs[1][0])
    d = runs[1][1].as_dict()
    assert d["epochs_run"] == 3 and d["early_stopped"] is False and len(d["approx_kl_per_epoch"]) == 3
    rec = runs[1][1].records.cpu().numpy()
    assert (rec[:, :, COUNT] == 3).all()
    assert all(np.isfinite(v) for k, v in d.items() if isinstance(v, float))


def test_early_stop_on_target_kl():
    s = None
    results = {}
    for name, K, target in (("stop", 3, 1e-12), ("k1", 1, None), ("loose", 3, 1e9), ("none", 3, None)):
        agent = _agent(_args(K=K, mb=512, B=1500))
        if s is None:
            s, act, logp, adv, vt = _data(agent, 1500)
        torch.manual_seed(100)
        out = agent.optimize(s, act, logp, adv, vt, mini_batch_size=512, fused=True, target_kl=target)
        torch.cuda.synchronize()
        results[name] = (_state(agent), out)
    stop = results["stop"][1].as_dict()
    assert stop["epochs_run"] == 1 and stop["early_stopped"] is True and len(stop["approx_kl_per_epoch"]) == 1
    assert _equal_states(results["stop"][0], results["k1"][0])
    assert results["k1"][1] is None and results["none"][1] is None
    loose = results["loose"][1].as_dict()
    assert loose["epochs_run"] == 3 and loose["early_stopped"] is False
    assert _equal_states(results["loose"][0], results["none"][0])
    # the reference interface: args.target_kl applies by default and the stats are kept
    args = _args(K=3, mb=512, B=1500)
    args.target_kl = 1e-12
    agent = _agent(args)
    out = agent.optimize(s, act, logp, adv, vt, mini_batch_size=512, fused=True)
    assert out.as_dict()["epochs_run"] == 1


# ---------------------------------------------------------------- 7: the PyTorch step reports the same statistics
@pytest.mark.parametrize("use_graph", [True, False])
def test_pytorch_path_statistics_agree_with_fused(use_graph):
    mb = 1000
    args = _args(K=1, mb=mb, B=mb)
    out = {}
    for fused in (True, False):
        agent = _agent(args)
        s, act, logp, adv, vt = _data(agent, mb)
        ref = _torch_stats(_agent(args), s, act, logp, adv, vt)
        torch.manual_seed(3)
        st = agent.optimize(s, act, logp, adv, vt, mini_batch_size=mb, fused=fused, use_graph=use_graph, stats=True)
        out[fused] = st.as_dict()
    assert set(out[True]) == set(out[False])
    _check_means(out[False], ref, mb, ref["surrogate_scale"])
    _check_means(out[True], ref, mb, ref["surrogate_scale"])
    assert out[False]["epochs_run"] == out[True]["epochs_run"] == 1


# ---------------------------------------------------------------- 5 + 6: two ranks
def _union_and_target():
    """single process on the union batch (1024 rows, one minibatch per epoch): per-epoch KL and a target that stops after
    the second epoch when the KL grows, else after the first"""
    agent = _agent(_args(K=3, mb=1024, B=1024, lr=3e-3))
    s, act, logp, adv, vt = _data(agent, 1024)
    torch.manual_seed(7)
    kl = agent.optimize(s, act, logp, adv, vt, mini_batch_size=1024, fused=True, stats=True).as_dict()["approx_kl_per_epoch"]
    target = 0.5 * (kl[0] + kl[1]) if kl[1] > kl[0] else 0.5 * kl[0]
    agent = _agent(_args(K=3, mb=1024, B=1024, lr=3e-3))
    torch.manual_seed(7)
    st = agent.optimize(s, act, logp, adv, vt, mini_batch_size=1024, fused=True, target_kl=target)
    return target, st.records.cpu().numpy(), st.epochs_run


def _rank_body(rank, q, target, device):
    args = _args(K=3, mb=512, B=512, lr=3e-3)
    agent = _agent(args, device=device)
    s, act, logp, adv, vt = _data(agent, 1024, device=device)        # same 1024 rows on both ranks; each trains on its half
    lo = rank * 512
    torch.manual_seed(7)
    st = agent.optimize(s[lo:lo + 512], act[lo:lo + 512], logp[lo:lo + 512], adv[lo:lo + 512], vt[lo:lo + 512],
                        mini_batch_size=512, fused=True, stats=True, target_kl=target)
    torch.cuda.synchronize()
    peers = any(agent._fused.get("peers", {}).values())
    q.put((rank, st.records.cpu().numpy(), st.epochs_run, peers))


def _gloo_worker(rank, world, port, q, target):
    import os, sys
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        _rank_body(rank, q, target, "cuda")
    finally:
        dist.destroy_process_group()


def _nccl_worker(rank, world, port, q, target):
    import os, sys
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), SAT_PEER_ALLREDUCE="1")
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        _rank_body(rank, q, target, dev)
    finally:
        dist.destroy_process_group()


def _run_two_ranks(worker, port_base, target):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = port_base + (os.getpid() % 2000)
    procs = [ctx.Process(target=worker, args=(r, 2, port, q, target)) for r in range(2)]
    for p in procs:
        p.start()
    res = {r: (rec, e, pe) for r, rec, e, pe in (q.get(timeout=240) for _ in procs)}
    for p in procs:
        p.join(timeout=60)
    return res


def _check_two_ranks(res, ref_rec, ref_epochs):
    assert np.array_equal(res[0][0], res[1][0])                      # bit-identical statistics on both ranks
    assert res[0][1] == res[1][1] == ref_epochs
    for e in range(ref_epochs):
        got, ref = _record_means(res[0][0][e]), _record_means(ref_rec[e])
        ref = dict(ref, surrogate=ref["policy_loss"])
        _check_means(got, ref, 1024)


@pytest.mark.timeout(300)
def test_two_ranks_gloo_statistics_and_early_stop_agree():
    target, ref_rec, ref_epochs = _union_and_target()
    assert ref_epochs in (1, 2)
    res = _run_two_ranks(_gloo_worker, 31700, target)
    _check_two_ranks(res, ref_rec, ref_epochs)


@pytest.mark.timeout(300)
def test_two_gpus_nccl_peer_memory_statistics_and_early_stop_agree():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    target, ref_rec, ref_epochs = _union_and_target()
    res = _run_two_ranks(_nccl_worker, 33700, target)
    assert res[0][2] and res[1][2], "the peer-memory path was not taken"
    _check_two_ranks(res, ref_rec, ref_epochs)


# ---------------------------------------------------------------- 8: rollout and self-play
def _trainer(n=256, T=8, mb=512):
    from ppo_rl_satellite_b200 import engine as eng, rollout
    from ppo_rl_satellite_b200.dropin import ppo_continuous as P
    torch.manual_seed(0)
    args = _args(K=2, mb=mb, B=n * T)
    env = eng.EnvBatch(n, mode="cw", d_capture=20000.0, max_episode_steps=5, auto_reset=True)
    return env, P.PPO_continuous(args, "pursuer"), P.PPO_continuous(args, "evader")


def test_vector_trainer_and_self_play_report_statistics():
    from ppo_rl_satellite_b200 import rollout
    env, agent, opp = _trainer()
    agent.use_adv_norm = False                    # keep buf.adv as the GAE produced it, for the explained-variance check
    tr = rollout.VectorTrainer(env, agent, opp, 8)
    tr.collect()
    d = tr.update(512, stats=True).as_dict()
    keys = {"policy_loss", "entropy", "approx_kl", "clip_fraction", "value_loss", "actor_grad_norm", "critic_grad_norm",
            "epochs_run", "early_stopped", "approx_kl_per_epoch", "explained_variance"}
    assert set(d) == keys
    assert all(np.isfinite(d[k]) for k in keys - {"early_stopped", "approx_kl_per_epoch", "epochs_run"})
    assert d["epochs_run"] == 2 and all(np.isfinite(d["approx_kl_per_epoch"]))
    adv, vt = tr.buf.adv.double().cpu().numpy(), tr.buf.v_target.double().cpu().numpy()
    ev = 1.0 - np.var(adv) / np.var(vt)
    assert abs(d["explained_variance"] - ev) <= 1e-6 * max(1.0, abs(ev)), (d["explained_variance"], ev)
    tr.collect()
    assert tr.update(512) is None                 # stats off: nothing returned, as before

    env, agent, opp = _trainer()
    sp = rollout.SelfPlay(env, agent, opp, 8, 512)
    recs = sp.run_phase(0, 2, stats=True) + sp.run_phase(1, 1)
    assert len(recs) == 3
    for r in recs[:2]:
        assert {"flag", "iteration", "mean_reward", "episodes_finished"} | keys <= set(r)
    assert set(recs[2]) == {"flag", "iteration", "mean_reward", "episodes_finished"}
