"""PPO update for the DS-RNN policy (SURVEY.md 8(f) row N1), the reference's `PPO`
(pytorchBaselines/a2c_ppo_acktr/algo/ppo.py:7-118) with the same constructor, the same `update(rollouts)` return value
and the same arithmetic: advantage normalisation with the unbiased std + 1e-5, clipped surrogate, clipped value loss,
`value_loss * value_loss_coef + action_loss - entropy * entropy_coef`, grad-norm clipping, Adam(lr, eps).

Added for the sharded rollout (BASELINE.json configs[4]: envs sharded over 1/2/4/8 GPUs):

* data parallel over `torch.distributed` (NCCL on GPUs, gloo in the CPU tests): every rank owns the rollouts of its own
  envs; the advantage mean/std are computed over ALL ranks' samples (one float64 all-reduce of sum / sum-of-squares /
  count) and the gradients of each minibatch are averaged with ONE all-reduce of a flat bucket before clipping, so a
  W-rank update of W*n envs is the single-process update of the union minibatch;
* `max_envs_per_pass`: a minibatch is processed in sub-chunks of whole env trajectories with gradient accumulation
  (same gradient, bounded activation memory: T=30 steps x 21 edges x 768 gate columns per env are kept for backward).

`deterministic=True` (the reference's training.cuda_deterministic) makes the native update bit-reproducible: its split-K
weight gradients and edge-encoder gradient are summed in a fixed order instead of with atomics (native.ordered).  The
other update paths are reproducible already.  With several ranks every rank runs the same ordered kernels; whether two
multi-GPU runs then agree bit for bit also depends on the order of NCCL's all-reduce, which this does not control.

The rollout forward (`Policy.act`) is the CUDA hot path.  The differentiable sequence forward used here is
`Policy.evaluate_actions` (model.py): the recurrent units run as masked GRU sequences -- one autograd node each, cuBLAS
GEMMs (fp32, `tf32=True`, or split-bf16 3-pass with `bf16x3=True`) around the library's hand-written gate kernels
(csrc/dsrnn_train.cu) -- and everything without a recurrence is evaluated for the whole [T, n] chunk in one batch.
"""
import torch
import torch.distributed as dist
import torch.nn as nn
import torch.optim as optim


def _world(group=None):
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group)
    return 1


def normalized_advantages(rollouts, group=None):
    """ppo.py:37-38 -- (A - mean) / (std + 1e-5) with torch's unbiased std, statistics taken over every rank."""
    adv = rollouts.returns[:-1] - rollouts.value_preds[:-1]
    if _world(group) == 1:
        return (adv - adv.mean()) / (adv.std() + 1e-5)
    a64 = adv.double()
    stats = torch.stack([a64.sum(), (a64 * a64).sum(), torch.tensor(float(adv.numel()), dtype=torch.float64, device=adv.device)])
    dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    total, sq, count = stats[0], stats[1], stats[2]
    mean = total / count
    var = (sq - count * mean * mean).clamp_min(0.0) / (count - 1.0)
    return ((a64 - mean) / (var.sqrt() + 1e-5)).float()


class PPO:
    def __init__(self, actor_critic, clip_param, ppo_epoch, num_mini_batch, value_loss_coef, entropy_coef, lr=None, eps=None,
                 max_grad_norm=None, use_clipped_value_loss=True, group=None, max_envs_per_pass=None, tf32=False, bf16x3=False,
                 native=False, deterministic=False):
        self.actor_critic = actor_critic
        self.clip_param = clip_param
        self.ppo_epoch = ppo_epoch
        self.num_mini_batch = num_mini_batch
        self.value_loss_coef = value_loss_coef
        self.entropy_coef = entropy_coef
        self.max_grad_norm = max_grad_norm
        self.use_clipped_value_loss = use_clipped_value_loss
        self.group = group
        self.max_envs_per_pass = max_envs_per_pass
        self.tf32 = bool(tf32)         # TF32 tensor cores for the fp32 GEMMs of the update's forward + backward
        self.bf16x3 = bool(bf16x3)     # split-bf16 3-pass tensor-core GEMMs (fp32-level accuracy) for the recurrent products
        self.native = bool(native)     # every contraction of the update on the library's own tcgen05 kernels (native.py), CUDA only
        self.deterministic = bool(deterministic)   # native path: reductions in a fixed order, same gradients bit for bit
        self.optimizer = optim.Adam(actor_critic.parameters(), lr=lr, eps=eps)
        self.perm_fn = None            # tests / reproducibility: callable(num_processes) -> env permutation
        self.allreduce_calls = 0
        self.overlap_allreduce = True  # start the all-reduce of the early gradient bucket while backward is still running
        self._early = None             # overlap state: parameters of the early bucket, hooks, pending handle

    # ------------------------------------------------------------------ pieces
    def _losses(self, sample, weight):
        obs, hx, actions, value_preds, returns, masks, old_log_probs, adv = sample
        values, log_probs, entropy, _ = self.actor_critic.evaluate_actions(obs, hx, masks, actions)
        ratio = torch.exp(log_probs - old_log_probs)
        surr1 = ratio * adv
        surr2 = torch.clamp(ratio, 1.0 - self.clip_param, 1.0 + self.clip_param) * adv
        action_loss = -torch.min(surr1, surr2).mean()
        if self.use_clipped_value_loss:
            clipped = value_preds + (values - value_preds).clamp(-self.clip_param, self.clip_param)
            value_loss = 0.5 * torch.max((values - returns).pow(2), (clipped - returns).pow(2)).mean()
        else:
            value_loss = 0.5 * (returns - values).pow(2).mean()
        total = value_loss * self.value_loss_coef + action_loss - entropy * self.entropy_coef
        (total * weight).backward()
        return value_loss.detach() * weight, action_loss.detach() * weight, entropy.detach() * weight

    # Gradient exchange (SURVEY 8(e)): the 3.9 MB of gradients are averaged once per minibatch, in two flat buckets.  Backward
    # reaches the heads, the node RNN and the attention first and the two edge GRUs -- by far its longest part -- last, so
    # the bucket of everything BUT the edge-GRU parameters is complete early: its all-reduce is started from a gradient
    # hook (asynchronously, on NCCL's stream) and runs over NVLink while the edge-GRU backward is still computing; only
    # the edge-GRU bucket (0.26 M of the 0.97 M elements) is exchanged after backward.
    def _is_late(self, name):
        return "humanhumanEdgeRNN" in name

    def _arm_early_bucket(self):
        """Called before the LAST backward of a minibatch (gradient accumulation keeps earlier passes local)."""
        if _world(self.group) == 1 or not self.overlap_allreduce:
            return
        if self._early is None:
            self._early = {"params": None, "hooks": [], "pending": None, "ready": 0, "armed": False}
        st = self._early
        if st["params"] is None:
            # parameters that actually receive gradients are only known after one backward: the first minibatch of the
            # first update runs without overlap and records them
            return
        st["ready"], st["armed"] = 0, True

    def _early_hook(self, _param):
        st = self._early
        if st is None or not st["armed"]:
            return
        st["ready"] += 1
        if st["ready"] == len(st["params"]):
            st["armed"] = False
            flat = torch.cat([p.grad.reshape(-1) for p in st["params"]])
            work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            st["pending"] = (flat, work)
            self.allreduce_calls += 1

    def _average_gradients(self):
        world = _world(self.group)
        if world == 1:
            return
        named = [(n, p) for n, p in self.actor_critic.named_parameters() if p.grad is not None]
        st = self._early
        pending = st["pending"] if st is not None else None
        if pending is not None:
            st["pending"] = None
            early_ids = {id(p) for p in st["params"]}
            rest = [p for _, p in named if id(p) not in early_ids]
        else:
            rest = [p for _, p in named]
        flat = torch.cat([p.grad.reshape(-1) for p in rest])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        self.allreduce_calls += 1
        buckets = [(rest, flat)]
        if pending is not None:
            pending[1].wait()
            buckets.append((st["params"], pending[0]))
        for params, buf in buckets:
            buf.div_(world)
            offset = 0
            for p in params:
                p.grad.copy_(buf[offset:offset + p.numel()].view_as(p.grad))
                offset += p.numel()
        if st is not None and st["params"] is None and self.overlap_allreduce:
            st["params"] = [p for n, p in named if not self._is_late(n)]
            st["hooks"] = [p.register_post_accumulate_grad_hook(self._early_hook) for p in st["params"]]

    # ------------------------------------------------------------------ reference interface
    def update(self, rollouts, sync=True):
        """`sync=False` returns the three averaged losses as a device tensor instead of Python floats (no host synchronisation)."""
        from . import model as _model
        from . import native as _native

        prev, prev_gemm, prev_det = torch.backends.cuda.matmul.allow_tf32, _model.SEQUENCE_GEMM, _native.DETERMINISTIC
        prev_impl = getattr(self.actor_critic, "sequence_impl", "batched")
        torch.backends.cuda.matmul.allow_tf32 = prev or self.tf32
        if self.bf16x3:
            _model.SEQUENCE_GEMM = "bf16x3"
        if self.native and rollouts.device.type == "cuda":
            self.actor_critic.sequence_impl = "native"
        if self.deterministic:
            _native.DETERMINISTIC = True
        try:
            return self._update(rollouts, sync)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
            _model.SEQUENCE_GEMM = prev_gemm
            _native.DETERMINISTIC = prev_det
            self.actor_critic.sequence_impl = prev_impl

    def _update(self, rollouts, sync=True):
        advantages = normalized_advantages(rollouts, self.group)
        N = rollouts.num_processes
        n = N // self.num_mini_batch
        per_pass = n if not self.max_envs_per_pass else max(1, min(n, int(self.max_envs_per_pass)))
        sums = torch.zeros(3, device=advantages.device)
        for _ in range(self.ppo_epoch):
            perm = self.perm_fn(N) if self.perm_fn is not None else torch.randperm(N)
            perm = torch.as_tensor(perm, dtype=torch.int64).to(advantages.device)
            for start in range(0, n * self.num_mini_batch, n):
                self.optimizer.zero_grad()
                for a in range(0, n, per_pass):
                    ind = perm[start + a:start + min(a + per_pass, n)]
                    if a + per_pass >= n:
                        self._arm_early_bucket()
                    parts = self._losses(rollouts.gather(ind, advantages), ind.numel() / float(n))
                    sums += torch.stack(parts)
                self._average_gradients()
                nn.utils.clip_grad_norm_(self.actor_critic.parameters(), self.max_grad_norm)
                self.optimizer.step()
        sums /= float(self.ppo_epoch * self.num_mini_batch)
        if _world(self.group) > 1:
            dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=self.group)
            sums /= _world(self.group)
        if not sync:
            return sums
        value_loss, action_loss, entropy = sums.tolist()
        return value_loss, action_loss, entropy


def update_linear_schedule(optimizer, epoch, total_num_epochs, initial_lr):
    """pytorchBaselines/a2c_ppo_acktr/utils.py:46-50."""
    lr = initial_lr - (initial_lr * (epoch / float(total_num_epochs)))
    for group in optimizer.param_groups:
        group["lr"] = lr
