"""ppo_continuous -- drop-in for the reference's ppo_continuous.py with the hot parts on CUDA kernels.

Same classes, parameter names and checkpoint files as the reference, so model_file/one_layer/agent_pursuer_* load
unchanged (ppo_continuous.py:61-134, 252-258):
  choose_action -> fused Gaussian-actor kernel (forward + Philox sampling + log-prob), batch 1 or [N, 18]
  update        -> critic values, sat_gae_flat reverse scan, advantage normalisation kernel; the K-epoch clipped-PPO
                   minibatch loop runs on the fused forward/backward/Adam kernels of csrc/ppo_update.cu (fused_update=True,
                   SURVEY s8 f.1) or as the PyTorch step (SURVEY a19), with a gradient all-reduce when torch.distributed is
                   initialised (one flat bucket per network, NCCL over NVLink).
Only the Gaussian policy is on the CUDA path (policy_dist == "Beta" is out of the north star's scope).
"""
import os
import zlib

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.distributions import Normal

try:
    from ._boot import engine as _eng
except ImportError:
    from _boot import engine as _eng
_L = _eng.L


def orthogonal_init(layer, gain=1.0):
    nn.init.orthogonal_(layer.weight, gain=gain)
    nn.init.constant_(layer.bias, 0)


class Actor_Gaussian(nn.Module):
    def __init__(self, args, agent_idx):
        super().__init__()
        self.agent_name = 'agent_%s' % agent_idx
        self.chkpt_file = os.path.join(args.chkpt_dir, self.agent_name + '_actor_Gaussian')
        self.max_action = args.max_action
        self.fc1 = nn.Linear(args.state_dim, args.hidden_width)
        self.fc2 = nn.Linear(args.hidden_width, args.hidden_width)
        self.mean_layer = nn.Linear(args.hidden_width, args.action_dim)
        self.log_std = nn.Parameter(torch.zeros(1, args.action_dim))
        self.activate_func = [nn.ReLU(), nn.Tanh()][args.use_tanh]
        if args.use_orthogonal_init:
            orthogonal_init(self.fc1)
            orthogonal_init(self.fc2)
            orthogonal_init(self.mean_layer, gain=0.01)

    def forward(self, s):
        s = self.activate_func(self.fc1(s))
        s = self.activate_func(self.fc2(s))
        return self.max_action * torch.tanh(self.mean_layer(s))

    def get_dist(self, s):
        mean = self.forward(s)
        # validate_args=False: the default argument check synchronises the stream (illegal inside a CUDA-graph capture)
        return Normal(mean, torch.exp(self.log_std.expand_as(mean)), validate_args=False)

    def save_checkpoint(self):
        torch.save(self.state_dict(), self.chkpt_file)

    def load_checkpoint(self):
        self.load_state_dict(torch.load(self.chkpt_file, map_location="cpu"))


class Critic(nn.Module):
    def __init__(self, args, agent_idx):
        super().__init__()
        self.agent_name = 'agent_%s' % agent_idx
        self.chkpt_file = os.path.join(args.chkpt_dir, self.agent_name + '_critic')
        self.fc1 = nn.Linear(args.state_dim, args.hidden_width)
        self.fc2 = nn.Linear(args.hidden_width, args.hidden_width)
        self.fc3 = nn.Linear(args.hidden_width, 1)
        self.activate_func = [nn.ReLU(), nn.Tanh()][args.use_tanh]
        if args.use_orthogonal_init:
            orthogonal_init(self.fc1)
            orthogonal_init(self.fc2)
            orthogonal_init(self.fc3)

    def forward(self, s):
        s = self.activate_func(self.fc1(s))
        s = self.activate_func(self.fc2(s))
        return self.fc3(s)

    def save_checkpoint(self):
        torch.save(self.state_dict(), self.chkpt_file)

    def load_checkpoint(self):
        self.load_state_dict(torch.load(self.chkpt_file, map_location="cpu"))


def allreduce_grads_(module, group=None):
    """Average gradients across ranks with ONE flat all-reduce per network (286 KB actor / 284 KB critic)."""
    dist = torch.distributed
    if group is False or not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    grads = [p.grad for p in module.parameters() if p.grad is not None]
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, group=group)
    flat /= dist.get_world_size(group)
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()


_FROM_ARGS = object()


class PpoUpdateStats:
    """Training diagnostics of one PPO_continuous.optimize call.

    `records` is an fp64 tensor [K][2][PPO_STATS_DOUBLES] (layout _lib.PPO_STAT_*) on the training device: for every epoch and
    network (0 actor, 1 critic) the sums over that epoch's minibatches of the global minibatch means, with COUNT the number of
    minibatches. Nothing is read back until as_dict(), except one fp64 per epoch when target_kl is set."""

    def __init__(self, records, minibatches: int, target_kl=None):
        self.records, self.minibatches, self.target_kl = records, int(minibatches), target_kl
        self.epochs_run, self.early_stopped = 0, False
        self.extra = {}                 # further device scalars reported by as_dict(), e.g. explained_variance

    def end_epoch(self, e: int) -> bool:
        """Called once epoch e is enqueued on the current stream; True when the remaining epochs must not run: the mean over
        epoch e's minibatches of the global approximate KL is above target_kl (one fp64 read, synchronising the stream)."""
        self.epochs_run = e + 1
        if self.target_kl is None or e + 1 >= self.records.shape[0]:
            return False
        kl = float(self.records[e, 0, _L.PPO_STAT_APPROX_KL].item()) / self.minibatches
        self.early_stopped = kl > self.target_kl
        return self.early_stopped

    def as_dict(self) -> dict:
        """Means over all minibatches that ran (one device synchronisation)."""
        names = sorted(self.extra)
        flat = torch.cat([self.records.reshape(-1)] + [self.extra[k].reshape(1).to(self.records) for k in names]).cpu()
        rec = flat[:self.records.numel()].view(self.records.shape)[:self.epochs_run]
        act, cri = rec.sum(0)
        n = _L.PPO_STAT_COUNT

        def mean(r, k):
            return float(r[k] / r[n]) if r[n] > 0 else float("nan")
        out = {"policy_loss": mean(act, _L.PPO_STAT_SURROGATE), "entropy": mean(act, _L.PPO_STAT_ENTROPY),
               "approx_kl": mean(act, _L.PPO_STAT_APPROX_KL), "clip_fraction": mean(act, _L.PPO_STAT_CLIP_FRAC),
               "value_loss": mean(cri, _L.PPO_STAT_LOSS), "actor_grad_norm": mean(act, _L.PPO_STAT_GRAD_NORM),
               "critic_grad_norm": mean(cri, _L.PPO_STAT_GRAD_NORM), "epochs_run": self.epochs_run,
               "early_stopped": self.early_stopped,
               "approx_kl_per_epoch": [mean(r[0], _L.PPO_STAT_APPROX_KL) for r in rec]}
        for i, k in enumerate(names):
            out[k] = float(flat[self.records.numel() + i])
        return out


class PPO_continuous:
    def __init__(self, args, agent_idx, device="cuda", seed=0, fused_update=True):
        if getattr(args, "policy_dist", "Gaussian") != "Gaussian":
            raise NotImplementedError("only the Gaussian policy is on the CUDA path")
        self.device = torch.device(device)
        self.policy_dist = args.policy_dist
        self.max_action, self.batch_size, self.mini_batch_size = args.max_action, args.batch_size, args.mini_batch_size
        self.max_train_steps, self.lr_a, self.lr_c = args.max_train_steps, args.lr_a, args.lr_c
        self.gamma, self.lamda, self.epsilon, self.K_epochs = args.gamma, args.lamda, args.epsilon, args.K_epochs
        self.entropy_coef, self.set_adam_eps = args.entropy_coef, args.set_adam_eps
        self.use_grad_clip, self.use_lr_decay, self.use_adv_norm = args.use_grad_clip, args.use_lr_decay, args.use_adv_norm
        self.target_kl = getattr(args, "target_kl", None)
        self.last_update_stats = None
        self.actor = Actor_Gaussian(args, agent_idx).to(self.device)
        self.critic = Critic(args, agent_idx).to(self.device)
        eps = dict(eps=1e-5) if self.set_adam_eps else {}
        # capturable Adam with a device-resident learning rate: the whole optimiser step can live in a CUDA graph
        cap = dict(capturable=True) if self.device.type == "cuda" else {}
        self.optimizer_actor = torch.optim.Adam(self.actor.parameters(), lr=torch.tensor(float(self.lr_a), device=self.device), **eps, **cap)
        self.optimizer_critic = torch.optim.Adam(self.critic.parameters(), lr=torch.tensor(float(self.lr_c), device=self.device), **eps, **cap)
        self._graph = None
        self._stats_acc = None
        self._fused = None
        self.fused_update = bool(fused_update)        # update(): fused CUDA minibatch step instead of autograd + torch Adam
        self._use_tanh = bool(args.use_tanh)
        self.actor_kernel = _eng.GaussianActorKernel(max_action=self.max_action, use_tanh=self._use_tanh, device=self.device)
        self.critic_kernel = _eng.GaussianActorKernel(use_tanh=self._use_tanh, device=self.device, critic=True)
        # per-agent Philox key offset; crc32 (not hash()) so that it is the same in every process and run
        self.seed, self._step = int(seed) + (zlib.crc32(str(agent_idx).encode()) & 0xffff), 0
        self._dirty = True

    # ---- kernel-side weight image follows the torch parameters
    def sync_kernels(self):
        if self._fused is not None and all(n.adopted() for n in self._fused["nets"]):
            for n in self._fused["nets"]:            # device-side repack of the flat parameters
                n.pack()
        else:
            self.actor_kernel.load_state_dict(self.actor.state_dict())
            self.critic_kernel.load_state_dict(self.critic.state_dict())
        self._dirty = False

    # ---- fused CUDA minibatch step (csrc/ppo_update.cu): flat parameter buffers the torch modules hold views of
    def _fused_for(self, mb):
        f = self._fused
        if f is None or not all(n.adopted() for n in f["nets"]):
            eps = 1e-5 if self.set_adam_eps else 1e-8
            na = _eng.PpoFusedNet(self.actor, False, self._use_tanh, self.max_action, self.optimizer_actor.param_groups[0]["lr"],
                                  packed=self.actor_kernel.packed, eps=eps)
            nc = _eng.PpoFusedNet(self.critic, True, self._use_tanh, 0.0, self.optimizer_critic.param_groups[0]["lr"],
                                  packed=self.critic_kernel.packed, eps=eps)
            if f is not None:                         # parameters were moved (e.g. module.to()): keep the Adam moments
                na.load_state_dict(f["nets"][0].state_dict()); nc.load_state_dict(f["nets"][1].state_dict())
            f = self._fused = {"nets": (na, nc), "mb": 0, "streams": (torch.cuda.Stream(self.device), torch.cuda.Stream(self.device))}
            self.actor_kernel.w, self.critic_kernel.w = na.actor_weights(), nc.actor_weights()
            self._graph = None                        # a captured graph holds the old parameter addresses
        # torch's Optimizer.load_state_dict replaces the lr tensors: always read the live ones
        f["nets"][0].lr = self.optimizer_actor.param_groups[0]["lr"]
        f["nets"][1].lr = self.optimizer_critic.param_groups[0]["lr"]
        if f["mb"] < mb:
            f["mb"] = mb
            for n in f["nets"]:                       # one workspace per network: the two chains run concurrently
                n.bind(_eng.ppo_workspace(mb, self.device))
        return f

    def _peer_allreduce(self, f, group):
        """True when the gradient all-reduce runs inside the Adam kernel over NVLink peer memory (NCCL process group on
        CUDA, torch symmetric memory available, SAT_PEER_ALLREDUCE != 0); otherwise the step calls dist.all_reduce.
        The decision is collective: a rank whose rendezvous failed would otherwise take the NCCL path while its peers wait in
        the symmetric-memory barrier, so the local outcome is MIN-reduced over the group before anyone commits. Cached per
        process group."""
        cache = f.setdefault("peers", {})
        key = id(group) if group is not None else None
        if key not in cache:
            dist = torch.distributed
            ok = os.environ.get("SAT_PEER_ALLREDUCE", "1") != "0" and dist.get_backend(group) == "nccl"
            err = None
            if ok:
                try:
                    for n in f["nets"]:
                        n.enable_peer_allreduce(group)
                except Exception as exc:          # no peer access / symmetric memory on this system
                    ok, err = False, exc
            if dist.get_backend(group) == "nccl":
                flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
                all_ok = bool(flag.item())
            else:
                all_ok = ok
            if not all_ok:
                for n in f["nets"]:
                    n.disable_peer_allreduce()     # private gradient buffer again on every rank
                if err is not None or ok:
                    import warnings
                    warnings.warn(f"symmetric-memory gradient exchange unavailable on at least one rank ({err!r}); using NCCL all-reduce")
            cache[key] = all_ok
        return cache[key]

    @staticmethod
    def _require_equal_batches(B, group, device):
        """Every rank must bring the same number of samples: the ranks issue one gradient exchange per minibatch, so
        different ceil(B / mb) would dead-lock, and the exchange averages per-rank means with equal weights. Collective."""
        dist = torch.distributed
        t = torch.tensor([B, -B], dtype=torch.int64, device=device if dist.get_backend(group) == "nccl" else "cpu")
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        if int(t[0]) != -int(t[1]):
            raise ValueError(f"PPO update with unequal per-rank batches (min {-int(t[1])}, max {int(t[0])} samples): shard the envs "
                             f"evenly (n_total % world == 0) or trim the rollout to a common size")

    def _optimize_fused(self, s, a, a_logprob, adv, v_target, mb, group, out=None):
        """The actor chain and the critic chain are independent (ppo_continuous.py:216-239 shares only s[index]), so each
        runs on its own stream: one network's short kernels (partial sums, Adam) hide under the other's GEMM kernels.
        out (PpoUpdateStats): the stats variants of the kernels add every minibatch to out.records; the diagnostics ride in the
        gradient buffer's tail, so the same exchange makes them global."""
        dist = torch.distributed
        if group is False:                            # explicit "no gradient exchange" (single-rank use inside a job)
            world, group = 1, None
        else:
            world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        B = s.shape[0]
        f = self._fused_for(min(mb, B))
        na, nc = f["nets"]
        peers = False
        if world > 1:
            self._require_equal_batches(B, group, self.device)
            peers = self._peer_allreduce(f, group)
        s, a, a_logprob = s.contiguous(), a.contiguous(), a_logprob.contiguous()
        adv, v_target = adv.reshape(-1).contiguous(), v_target.reshape(-1).contiguous()
        clip = 0.5 if self.use_grad_clip else 0.0
        main = torch.cuda.current_stream(self.device)
        sa, sc = f["streams"]
        stats = out is not None
        for e in range(self.K_epochs):
            perm = torch.randperm(B, device=s.device)
            sa.wait_stream(main); sc.wait_stream(main)
            perm.record_stream(sa); perm.record_stream(sc)
            rec_a, rec_c = (out.records[e, 0], out.records[e, 1]) if stats else (None, None)
            for lo in range(0, B, mb):
                m = min(mb, B - lo)
                index = perm.data_ptr() + 8 * lo
                with torch.cuda.stream(sa):
                    na.actor_grad(s, a, a_logprob, adv, index, m, self.epsilon, self.entropy_coef, stats=stats)
                    if world > 1 and not peers:
                        dist.all_reduce(na.grads_stats if stats else na.grads, group=group)
                    na.adam(clip, 1.0 / world, record=rec_a)
                with torch.cuda.stream(sc):
                    nc.critic_grad(s, v_target, index, m)
                    if world > 1 and not peers:
                        dist.all_reduce(nc.grads, group=group)
                    nc.adam(clip, 1.0 / world, record=rec_c)
            if stats:
                with torch.cuda.stream(sa):
                    if out.end_epoch(e):
                        break
        main.wait_stream(sa); main.wait_stream(sc)
        self._dirty = False                           # the Adam kernel rewrites the packed weight images itself

    def _obs(self, s):
        a = np.asarray(s, dtype=np.float32)
        return torch.as_tensor(np.ascontiguousarray(a.reshape(-1, a.shape[-1])), device=self.device), a.ndim == 1

    def evaluate(self, s):
        x, one = self._obs(s)
        with torch.no_grad():
            a = self.actor(x).cpu().numpy()
        return a.flatten() if one else a

    def choose_action(self, s):
        """(a, a_logprob) as float32 numpy, flattened for a single observation (ppo_continuous.py:176-189)."""
        if self._dirty:
            self.sync_kernels()
        x, one = self._obs(s)
        a, lp = self.actor_kernel.sample(obs=x, seed=self.seed, step=self._step)
        self._step += 1
        out = torch.cat([a, lp], dim=1).cpu().numpy()
        a, lp = out[:, :a.shape[1]], out[:, a.shape[1]:]
        return (a.flatten(), lp.flatten()) if one else (a, lp)

    # ---- PPO update
    def update(self, replay_buffer, total_steps):
        s, a, a_logprob, r, s_, dw, done = (t.to(self.device) for t in replay_buffer.numpy_to_tensor())
        with torch.no_grad():                                              # :198-210
            vs, vs_ = self.critic(s), self.critic(s_)
            adv, v_target = _eng.gae_flat(r, vs, vs_, dw, done, self.gamma, self.lamda)
            adv, v_target = adv.view(-1, 1), v_target.view(-1, 1)
            if self.use_adv_norm:
                _eng.adv_normalize_(adv, group=False)
        self.last_update_stats = self.optimize(s, a, a_logprob, adv, v_target, fused=self.fused_update)
        if self.use_lr_decay:
            self.lr_decay(total_steps)

    def _minibatch_step(self, s, a, a_logprob, adv, v_target, group, acc=None):
        """one clipped-PPO actor step + one critic step on a minibatch (ppo_continuous.py:216-239); acc: fp64 [2][8] device
        accumulator the minibatch's statistics are added to (PpoUpdateStats layout)"""
        dist_now = self.actor.get_dist(s)
        dist_entropy = dist_now.entropy().sum(1, keepdim=True)
        a_logprob_now = dist_now.log_prob(a)
        ratios = torch.exp(a_logprob_now.sum(1, keepdim=True) - a_logprob.sum(1, keepdim=True))
        surr1 = ratios * adv
        surr2 = torch.clamp(ratios, 1 - self.epsilon, 1 + self.epsilon) * adv
        actor_loss = -torch.min(surr1, surr2) - self.entropy_coef * dist_entropy
        self.optimizer_actor.zero_grad(set_to_none=False)
        actor_loss.mean().backward()
        allreduce_grads_(self.actor, group)
        norms = []
        if self.use_grad_clip:
            norms.append(torch.nn.utils.clip_grad_norm_(self.actor.parameters(), 0.5))
        elif acc is not None:
            norms.append(torch.nn.utils.get_total_norm([p.grad for p in self.actor.parameters()]))
        self.optimizer_actor.step()
        v_s = self.critic(s)
        critic_loss = F.mse_loss(v_target, v_s)
        self.optimizer_critic.zero_grad(set_to_none=False)
        critic_loss.backward()
        allreduce_grads_(self.critic, group)
        if self.use_grad_clip:
            norms.append(torch.nn.utils.clip_grad_norm_(self.critic.parameters(), 0.5))
        elif acc is not None:
            norms.append(torch.nn.utils.get_total_norm([p.grad for p in self.critic.parameters()]))
        self.optimizer_critic.step()
        if acc is not None:
            with torch.no_grad():
                log_ratio = a_logprob_now.sum(1, keepdim=True) - a_logprob.sum(1, keepdim=True)
                one, zero = critic_loss.new_ones(()), critic_loss.new_zeros(())
                coef = [torch.clamp(0.5 / (nm + 1e-6), max=1.0) if self.use_grad_clip else one for nm in norms]
                acc[0] += torch.stack([actor_loss.mean(), (-torch.min(surr1, surr2)).mean(), dist_entropy.mean(),
                                       (torch.expm1(log_ratio) - log_ratio).mean(),
                                       ((ratios - 1.0).abs() > self.epsilon).float().mean(), norms[0], coef[0], one]).double()
                acc[1] += torch.stack([critic_loss, zero, zero, zero, zero, norms[1], coef[1], one]).double()

    def _graph_for(self, tensors, mb, group, acc=None):
        """CUDA graph of (gather minibatch by a static index buffer -> _minibatch_step), keyed by the buffer addresses"""
        key = (tuple(t.data_ptr() for t in tensors), tuple(t.shape for t in tensors), mb, acc is not None)
        if self._graph is not None and self._graph["key"] == key:
            return self._graph
        idx = torch.zeros(mb, dtype=torch.long, device=self.device)

        def body():
            self._minibatch_step(*(t.index_select(0, idx) for t in tensors), group, acc)
        # warm-up on a side stream (allocator, cuBLAS handles, lazily created Adam state), then capture; weights and
        # optimiser state are restored IN PLACE afterwards so the captured addresses stay valid
        params = list(self.actor.parameters()) + list(self.critic.parameters())
        saved = [p.detach().clone() for p in params]
        opts = (self.optimizer_actor, self.optimizer_critic)
        opt_saved = [{p: {k: v.detach().clone() for k, v in st.items() if torch.is_tensor(v)} for p, st in o.state.items()}
                     for o in opts]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(3):
                body()
        torch.cuda.current_stream(self.device).wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            body()
        with torch.no_grad():
            for p, q in zip(params, saved):
                p.copy_(q)
            for o, snap in zip(opts, opt_saved):
                for p, st in o.state.items():
                    for k, v in st.items():
                        if torch.is_tensor(v):
                            if p in snap and k in snap[p]:
                                v.copy_(snap[p][k])
                            else:
                                v.zero_()             # state created during the warm-up: back to a fresh optimiser
            if acc is not None:
                acc.zero_()
        self._graph = {"key": key, "graph": g, "idx": idx}
        return self._graph

    def optimize(self, s, a, a_logprob, adv, v_target, mini_batch_size=None, group=None, use_graph=False, fused=False,
                 stats=False, target_kl=_FROM_ARGS):
        """K epochs of clipped-PPO minibatch steps (ppo_continuous.py:213-239) on device tensors.
        fused: the hand-written forward/backward/Adam kernels (own Adam moments, independent of the torch optimisers);
        use_graph: replay one captured CUDA graph of the PyTorch step per minibatch (static buffers, full minibatches only).
        stats: return a PpoUpdateStats (policy / value loss, entropy, approximate KL, clip fraction, gradient norms) with the
        same keys on every path; otherwise None, unless target_kl is set.
        target_kl (default: args.target_kl, else None): early stop at epoch granularity. After each epoch the mean over its
        minibatches of the global approximate KL is read back (one fp64, the only added host synchronisation); above
        target_kl, the remaining epochs of both networks do not run. Unlike SB3's per-minibatch 1.5 x target_kl test, the
        epoch that crossed the target completes, which keeps the actor / critic streams overlapped within the epoch."""
        B = s.shape[0]
        mb = mini_batch_size or self.mini_batch_size
        if target_kl is _FROM_ARGS:
            target_kl = self.target_kl
        out = None
        if stats or target_kl is not None:
            out = PpoUpdateStats(torch.zeros((self.K_epochs, 2, _L.PPO_STATS_DOUBLES), dtype=torch.float64, device=s.device),
                                 -(-B // mb), target_kl)
        if fused:
            self._optimize_fused(s, a, a_logprob, adv, v_target, mb, group, out)
            return out
        dist = torch.distributed
        multi = group is not False and dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        if multi:
            self._require_equal_batches(B, group, self.device)
        acc = None
        if out is not None:                               # static accumulator: a captured graph adds into it
            if self._stats_acc is None or self._stats_acc.device != s.device:
                self._stats_acc = torch.zeros((2, _L.PPO_STATS_DOUBLES), dtype=torch.float64, device=s.device)
            acc = self._stats_acc
            acc.zero_()
        tensors = (s, a, a_logprob, adv, v_target)
        graph = None
        if use_graph and B >= mb:
            try:
                graph = self._graph_for(tensors, mb, group, acc)
            except Exception as exc:                      # capture not possible here: stay eager, say so once
                import warnings
                warnings.warn(f"CUDA-graph capture of the PPO step failed ({exc!r}); running eagerly")
                graph = None
        for e in range(self.K_epochs):
            perm = torch.randperm(B, device=s.device)
            for lo in range(0, B, mb):
                index = perm[lo:lo + mb]
                if graph is not None and index.numel() == mb:
                    graph["idx"].copy_(index)
                    graph["graph"].replay()
                else:
                    self._minibatch_step(*(t[index] for t in tensors), group, acc)
            if out is not None:
                if multi:                                 # per-rank minibatch means -> global means, the same on every rank
                    dist.all_reduce(acc, group=group)
                    acc /= dist.get_world_size(group)
                out.records[e].copy_(acc)
                acc.zero_()
                if out.end_epoch(e):
                    break
        self._dirty = True
        return out

    def lr_decay(self, total_steps):
        lr_a_now = self.lr_a * (1 - total_steps / self.max_train_steps)
        lr_c_now = self.lr_c * (1 - total_steps / self.max_train_steps)
        for p in self.optimizer_actor.param_groups:
            if torch.is_tensor(p['lr']):
                p['lr'].fill_(lr_a_now)           # device-resident: visible to a captured graph
            else:
                p['lr'] = lr_a_now
        for p in self.optimizer_critic.param_groups:
            if torch.is_tensor(p['lr']):
                p['lr'].fill_(lr_c_now)
            else:
                p['lr'] = lr_c_now

    def save_checkpoint(self):
        self.actor.save_checkpoint()
        self.critic.save_checkpoint()

    def load_checkpoint(self):
        self.actor.load_checkpoint()
        self.critic.load_checkpoint()
        self.actor.to(self.device)
        self.critic.to(self.device)
        self._dirty = True
