"""MGProto with a B200-native prototype head -- the drop-in boundary (SURVEY.md section 8b).

Same constructor, methods, attributes and state-dict keys as the reference's ``model.MGProto``
(``/root/reference/model.py:77-482``), so the reference's ``train_and_test.py`` / ``push.py`` /
``main.py`` loops drive it unchanged.  Differences a caller can observe (also listed in INTEGRATION.md):
``memory_updated_cls`` is a read-only snapshot of device flags; ``proto_layer_rf_info`` is computed for the
torchvision backbones by ``backbones.proto_layer_rf_info`` (the reference's receptive-field walk) and is ``None`` for
custom ``features``; ``construct_MGProto(pretrained=True)`` loads weights from ``$MGPROTO_PRETRAINED_DIR`` if set and
otherwise warns and keeps the random initialisation (no network on the target boxes).  The backbone, add-on convs, embedding and losses are
ordinary PyTorch; everything between the add-on output ``[B,D,H,W]`` and the log mixture
evidences ``[B,C,T]`` -- plus the memory bank and its EM update -- runs in the hand-written
sm_100a kernels of ``libmgproto_b200.so``.  There is no CPU path: tensors must be on a CUDA
device when the hot methods are called.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from ._lib import MGP_OUT_LOGP_BPHW, MGP_OUT_LOGP_NP, MGP_OUT_NEGP_BPHW
from .backbones import base_architecture_to_features, out_channels
from .memory import MemoryBank


def l2_normalize(x, dim):
    """ref model.py:40-41."""
    return F.normalize(x, p=2, dim=dim)


def momentum_update(old_value, new_value, momentum, debug=False):
    """ref model.py:44-50."""
    return momentum * old_value + (1 - momentum) * new_value


class NonNegLinear(nn.Module):
    """ref model.py:54-74: the pi mixing layer.  ``weight [C, C*K]`` is block-diagonal and
    non-negative; the fused head reads its class-diagonal blocks directly (no GEMM, no
    host-synchronising asserts).  ``forward`` is kept for API parity."""

    def __init__(self, in_features, out_features, prototype_class_identity=None, device=None, dtype=None):
        super().__init__()
        self.in_features = in_features
        self.out_features = out_features
        self.prototype_class_identity = prototype_class_identity
        self.weight = nn.Parameter(torch.ones((out_features, in_features), device=device, dtype=dtype),
                                   requires_grad=False)

    def forward(self, input, prototypes_to_keep_with_negative=None):
        return F.linear(input, self.weight, bias=None)


class MGProto(nn.Module):
    def __init__(self, features, img_size, prototype_shape, proto_layer_rf_info, num_classes, init_weights=True,
                 prototype_activation_function="log", add_on_layers_type="bottleneck", sz_embedding=32,
                 mem_capacity=800, mine_K=20):
        super().__init__()
        self.img_size = img_size
        self.prototype_shape = prototype_shape
        self.num_prototypes = prototype_shape[0]
        self.num_classes = num_classes
        self.epsilon = 1e-4
        self.prototype_activation_function = prototype_activation_function
        assert self.num_prototypes % self.num_classes == 0                        # ref :95
        self.num_prototypes_per_class = self.num_prototypes // self.num_classes
        C, K, D = num_classes, self.num_prototypes_per_class, prototype_shape[1]
        ident = torch.zeros(self.num_prototypes, C)
        ident[torch.arange(self.num_prototypes), torch.arange(self.num_prototypes) // K] = 1
        self.prototype_class_identity = ident                                     # CPU attribute, as in the reference
        self.proto_layer_rf_info = proto_layer_rf_info
        self.features = features
        cin = out_channels(features)

        if add_on_layers_type == "bottleneck":                                    # ref :117-135
            layers, cur = [], cin
            while cur > D or not layers:
                nxt = max(D, cur // 2)
                layers += [nn.Conv2d(cur, nxt, kernel_size=1), nn.ReLU(), nn.Conv2d(nxt, nxt, kernel_size=1)]
                if nxt > D:
                    layers.append(nn.ReLU())
                else:
                    assert nxt == D
                    layers.append(nn.Sigmoid())
                cur = cur // 2
            self.add_on_layers = nn.Sequential(*layers)
        else:                                                                     # 'regular', ref :137-143
            self.add_on_layers = nn.Sequential(nn.Conv2d(cin, D, kernel_size=1), nn.Conv2d(D, D, kernel_size=1))

        self.gap = nn.AdaptiveAvgPool2d(1)
        self.embedding = nn.Linear(cin, sz_embedding)

        mu = torch.rand(C, K, D)
        self.prototype_means = nn.Parameter(l2_normalize(mu, dim=2), requires_grad=True)          # ref :148-149
        self.init_sigma = 1 / math.sqrt(2 * math.pi)
        self.prototype_covs = nn.Parameter(torch.ones(C, K, D) * self.init_sigma, requires_grad=False)  # std, ref :151-152
        self.last_layer = NonNegLinear(self.num_prototypes, C, prototype_class_identity=self.prototype_class_identity)
        if init_weights:
            self.initialize_weights()

        self.mine_T = mine_K
        self.capacity_pc = mem_capacity
        self.queue = MemoryBank(C, D, self.capacity_pc * C, mode="all")
        self.iteration_counter = nn.Parameter(torch.zeros(1), requires_grad=False)
        self.prototype_optimizer = None

        self.update_interval = 1
        self.num_em_loop = 3
        self.alpha = 0.1
        self.tau = 0.990

        # B200 knobs (not in the reference)
        self.math_mode = "auto"          # 'fp32' exact SIMT | 'tc' tcgen05 fp16x3 | 'auto'
        self.em_n_split = 2              # row splits of the EM statistics reduction
        self.em_group = None             # torch.distributed process group of the batch-sharded replicas (parallel.py)
        self.em_shard = False            # True: shard bank rows over the ranks + all-reduce the EM statistics per loop
        self.overlap_enqueue = False     # multi-GPU: True = all-gather + enqueue on a side stream behind the backward (measured
                                         # slower on 2 x B200: 707 vs 640 us/step, profiles/r2_mgpu_breakdown.txt: the NCCL kernel
                                         # and the backward kernels delay each other), False = inline on the main stream
        self._side_stream = None
        self._em_status = None           # int32[1] on the device: set by the tensor-core EM kernel if sigma was not isotropic
        self._adam_step_dev = None       # int32[1] on the device: Adam step count, advanced by update_GMM's planner
        self._adam_step_seen = None      # host value the device counter was seeded from / last folded back to
        self._em_dirty = False           # device counter ahead of prototype_optimizer.state[...]['step']

    # -- reference attribute: CPU bool flags ----------------------------------------------------
    @property
    def memory_updated_cls(self):
        """The reference's CPU bool tensor (model.py:167), here a read-only snapshot of the device flags
        ``queue.updated`` (this read synchronises; the training path never needs it -- write through
        ``queue.updated``)."""
        return self.queue.updated.bool().cpu()

    # -- backbone side (stock PyTorch) ----------------------------------------------------------
    def conv_features(self, x):
        """ref model.py:176-186."""
        x = self.features(x)
        x_add = self.add_on_layers(x)
        x_embed = l2_normalize(self.embedding(self.gap(x).flatten(1)), dim=1)
        return x_add, x_embed

    # -- hot path ---------------------------------------------------------------------------------
    def head(self, x_add, gt):
        """Add-on features [B,D,H,W] (+ labels) -> log mixture evidences [B,C,T]; enqueues the mined
        patches when labels are given.  This is forward() without the backbone (ref :210-254)."""
        logits, xhat, idx = ops.head_forward(x_add, self.prototype_means, self.prototype_covs,
                                             self.last_layer.weight, gt, self.mine_T, self.math_mode)
        if gt is not None:
            with torch.no_grad():
                q = self.queue
                gt = gt.contiguous()
                HWn, Kn = x_add.shape[2] * x_add.shape[3], self.num_prototypes_per_class
                if self.em_group is not None:
                    # batch-sharded replicas: the gather kernel writes packed per-image records, ONE all-gather exchanges
                    # them, the enqueue kernels read the gathered buffer in place (no packing / unpacking copies)
                    from .parallel import all_gather_records
                    rec, _, _ = ops.mined_gather(xhat, idx, gt, HWn, self.num_classes, Kn, packed=True)
                    Dn = xhat.shape[1]
                    if self.overlap_enqueue:
                        # exchange + enqueue on a side stream, overlapping this step's loss / backward (nothing there
                        # reads the bank).  The inputs stay referenced until a later access waits (no record_stream:
                        # that would park their blocks in the allocator's deferred-free list).
                        self.wait_enqueue()
                        cur = torch.cuda.current_stream()
                        if self._side_stream is None:
                            self._side_stream = torch.cuda.Stream(device=x_add.device)
                        side = self._side_stream
                        side.wait_stream(cur)
                        with torch.cuda.stream(side):
                            buf = all_gather_records(rec, self.em_group)
                            r1, t1, g1 = ops._rec_views(buf, Kn, Dn)
                            ops.bank_enqueue(q.bank, q.mem_len, q.head, q.updated, r1, t1, g1, shadow=q.shadow_if_valid())
                            done = torch.cuda.Event()
                            done.record(side)
                            del buf, r1, t1, g1                                   # side-stream blocks: reused in stream order
                        # the bank remembers the event: every later access to its tensors (mem_len in the training loop,
                        # state_dict, push, update_GMM) first makes its stream wait for this enqueue
                        q.set_pending(done, (rec,))
                    else:
                        buf = all_gather_records(rec, self.em_group)
                        r1, t1, g1 = ops._rec_views(buf, Kn, Dn)
                        ops.bank_enqueue(q.bank, q.mem_len, q.head, q.updated, r1, t1, g1, shadow=q.shadow_if_valid())
                else:
                    top1, rows = ops.mined_gather(xhat, idx, gt, HWn, self.num_classes, Kn)
                    ops.bank_enqueue(q.bank, q.mem_len, q.head, q.updated, rows, top1, gt, shadow=q.shadow_if_valid())
                self.iteration_counter += 1                                       # ref :252
        return logits

    @torch.no_grad()
    def head_level0(self, x_add):
        """[B,C] level-0 log evidences = head(x_add, None)[:, :, 0]: what the reference's test / OoD loop uses
        (train_and_test.py:182-199), without mining the other T-1 levels or materialising log p."""
        return ops.head_level0(x_add, self.prototype_means, self.prototype_covs, self.last_layer.weight, self.math_mode)

    def forward(self, x, gt):
        """ref model.py:208-254 -> (log_probs [B,C,T], x_embed [B,sz_embedding])."""
        x_add, x_embed = self.conv_features(x)
        return self.head(x_add, gt), x_embed

    def compute_log_prob(self, _fea, n_block=4, c_block=1, eps=0e-10):
        """ref model.py:256-275: [N,D] (already normalised) -> [N,C,K].  The reference's row/class
        chunking only bounds its [N/4,P,D] temporaries; the fused kernel has none."""
        C, K, D = self.prototype_means.shape
        out = ops.logprob(_fea.contiguous(), self.prototype_means.detach().reshape(C * K, D),
                          self.prototype_covs.detach().reshape(C * K, D), MGP_OUT_LOGP_NP, eps=eps, eps_log=0.0,
                          math=self.math_mode)
        return out.view(-1, C, K)

    def push_forward(self, x):
        """ref model.py:429-438 -> (normalised features [B,D,H,W], -p [B,P,H,W])."""
        x_add, _ = self.conv_features(x)
        return self.push_forward_features(x_add)

    def push_forward_features(self, x_add):
        C, K, D = self.prototype_means.shape
        B, _, H, W = x_add.shape
        xhat, _, nchw = ops.normalize_fwd(x_add.contiguous(), want_nchw=True)
        dist = ops.logprob(xhat, self.prototype_means.detach().reshape(C * K, D),
                           self.prototype_covs.detach().reshape(C * K, D), MGP_OUT_NEGP_BPHW, B=B, HW=H * W,
                           math=self.math_mode)
        return nchw, dist.view(B, C * K, H, W)

    def push_search(self, x_add, labels):
        """Device-side half of push.py:104-158: per image, for the K prototypes of its class, the
        flat argmin of -p over HW and the value; the 401 MB map never leaves the GPU.
        -> (arg [B,K] int32, val [B,K], xhat [N,D])."""
        C, K, D = self.prototype_means.shape
        B, _, H, W = x_add.shape
        mu = self.prototype_means.detach().reshape(C * K, D)
        sg = self.prototype_covs.detach().reshape(C * K, D)
        # the max / arg-max epilogue of the tensor-core kernel already is the per-prototype search: no [B,P,HW] map at all
        stage = ops._stage_for_top1(B, H * W, C * K, D, sg, self.math_mode)
        if stage is not None:
            xhat, _, _, ws = ops.normalize_fwd(x_add.contiguous(), stage=stage)
            best = ops.logprob_top1(xhat, mu, sg, B, H * W, self.math_mode, ws=ws, staged=stage)
        else:
            xhat, _, _ = ops.normalize_fwd(x_add.contiguous())
            best = ops.logprob_top1(xhat, mu, sg, B, H * W, self.math_mode)
        if best is not None:
            arg, val = ops.push_argmin_top1(best, labels.contiguous(), C, K)
            return arg, val, xhat
        lp = ops.logprob(xhat, mu, sg, MGP_OUT_LOGP_BPHW, B=B, HW=H * W, math=self.math_mode)
        arg, val = ops.push_argmin(lp, labels.contiguous(), C, K)
        return arg, val, xhat

    # -- EM ---------------------------------------------------------------------------------------
    def _adam_config(self):
        """The fused sequential path needs the plain torch.optim.Adam that main.py:223-228 builds."""
        opt = self.prototype_optimizer
        if opt is None:
            raise RuntimeError("update_GMM needs model.prototype_optimizer (ref main.py:223-228)")
        if type(opt) is not torch.optim.Adam or len(opt.param_groups) != 1:
            return None
        g = opt.param_groups[0]
        if (len(g["params"]) != 1 or g["params"][0] is not self.prototype_means or g.get("weight_decay", 0) != 0
                or g.get("amsgrad", False) or g.get("maximize", False) or g.get("capturable", False)
                or g.get("differentiable", False)):
            return None
        return g

    def wait_enqueue(self):
        """Make the current stream wait for a bank enqueue still running on the side stream (multi-GPU path).
        update_GMM and the next enqueue call it; call it before reading ``queue`` tensors on another stream."""
        self.queue.wait_pending()

    def sync_optimizer_state(self):
        """Fold the Adam step count kept on the device (advanced by every update_GMM without touching the host)
        into ``prototype_optimizer.state[...]['step']``.  Synchronises; call it before inspecting or saving the
        optimiser.  update_GMM itself never waits for the device."""
        if self._em_status is not None and int(self._em_status.item()) != 0:
            raise RuntimeError("mgproto_b200: update_GMM's tensor-core kernel found anisotropic sigma after the host check "
                               "said isotropic (prototype_covs was modified in place without a version bump?)")
        if self._em_dirty:
            v = int(self._adam_step_dev.item())
            st = self.prototype_optimizer.state[self.prototype_means]
            if torch.is_tensor(st["step"]):
                st["step"].fill_(float(v))
            else:
                st["step"] = v
            self._adam_step_seen = v
            self._em_dirty = False

    def _hook_optimizer(self):
        """optimizer.state_dict() (checkpointing in the reference's loop) must see the Adam step count update_GMM keeps
        on the device: fold it in right before the state is read.  optimizer.load_state_dict() replaces the state:
        fold first (a state dict that aliases the live tensors then loads the current step), and reseed the device
        counter from the loaded step afterwards."""
        opt = self.prototype_optimizer
        if getattr(opt, "_mgp_hooked", None) is not self:
            opt.register_state_dict_pre_hook(lambda o: self.sync_optimizer_state() if o is self.prototype_optimizer else None)
            opt.register_load_state_dict_pre_hook(
                lambda o, sd: self.sync_optimizer_state() if o is self.prototype_optimizer else None)
            opt.register_load_state_dict_post_hook(lambda o: self._reseed_after_load(o))
            opt._mgp_hooked = self

    def _reseed_after_load(self, opt):
        if opt is self.prototype_optimizer and self._adam_step_dev is not None:
            st = opt.state.get(self.prototype_means, {})
            self._seed_adam_step(int(st["step"]) if "step" in st else 0)

    def _seed_adam_step(self, step):
        """Set the device counter to `step` (in place when it exists: a captured CUDA graph keeps reading it)."""
        dev = self.prototype_means.device
        if self._adam_step_dev is not None and self._adam_step_dev.device == dev:
            self._adam_step_dev.fill_(step)
        else:
            self._adam_step_dev = torch.tensor([step], dtype=torch.int32, device=dev)
        self._adam_step_seen = step
        self._em_dirty = False

    def _adam_state(self):
        opt, p = self.prototype_optimizer, self.prototype_means
        st = opt.state[p]
        if len(st) == 0:
            st["step"] = torch.tensor(0.0, dtype=torch.float32)
            st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        return st

    def _prepare_adam(self):
        """(param group, state) of prototype_optimizer for the fused update_GMM, or (None, None) for the generic path.
        Creates the Adam state and (re)seeds the device step counter: host-side work that a CUDA-graph capture of
        update_GMM must not contain, so GraphedStep calls this before capturing."""
        group = self._adam_config()
        if group is None:
            return None, None
        opt = self.prototype_optimizer
        fresh = getattr(opt, "_mgp_hooked", None) is not self        # first call, or a new optimiser object
        st = self._adam_state()
        self._hook_optimizer()
        host_step = int(st["step"])
        if fresh or self._adam_step_dev is None or self._adam_step_dev.device != self.prototype_means.device or \
                self._adam_step_seen is None or host_step != self._adam_step_seen:
            # the optimiser state was stepped elsewhere: keep the steps not folded back yet -- unless the optimiser is
            # a new object (they were the old optimiser's)
            if not fresh and self._em_dirty and self._adam_step_dev is not None and self._adam_step_seen is not None:
                host_step += int(self._adam_step_dev.item()) - self._adam_step_seen
                st["step"] = torch.tensor(float(host_step)) if torch.is_tensor(st["step"]) else host_step
            self._seed_adam_step(host_step)
        return group, st

    @torch.no_grad()
    def update_GMM(self):
        """ref model.py:277-301 with identical sequential semantics (one Adam step on the whole
        mean tensor per updated class and EM loop) in 4 + 2*num_em_loop launches and no host
        synchronisation.  With ``em_group`` set, bank rows are sharded over the ranks and the packed
        sufficient statistics are all-reduced once per EM loop (parallel.py)."""
        q = self.queue
        self.wait_enqueue()
        C, K, D = self.prototype_means.shape
        cap = q.cap_cls
        dev = self.prototype_means.device
        L = self.num_em_loop
        group, st = self._prepare_adam()
        order = torch.empty(C, dtype=torch.int32, device=dev)
        sched = torch.empty(2, dtype=torch.int32, device=dev)
        world, rank = 1, 0
        if self.em_group is not None and self.em_shard:
            import torch.distributed as dist
            world, rank = dist.get_world_size(self.em_group), dist.get_rank(self.em_group)
        n_split = self.em_n_split if world == 1 else 1
        rows_per = (cap + world - 1) // world
        r0, r1 = min(cap, rank * rows_per), min(cap, (rank + 1) * rows_per)
        stride = ops.em_stat_stride(K, D)
        stats = torch.zeros((C, n_split, stride), dtype=torch.float32, device=dev) if (world > 1) else \
            torch.empty((C, n_split, stride), dtype=torch.float32, device=dev)
        mu, sg, wt = self.prototype_means.data, self.prototype_covs.data, self.last_layer.weight.data

        if group is None:
            return self._update_GMM_generic(order, sched, stats, n_split, r0, r1, world)

        lr, (b1, b2), eps = group["lr"], group["betas"], group["eps"]
        if world == 1:
            # tensor-core path (csrc/em_tc.cu): K <= 16, D in {128, 256}, sigma constant over d inside every prototype
            # (one cached host check: prototype_covs never changes in the reference's loop) -- needs the bank's shadow
            shadow, iso = None, False
            if 2 <= K <= 16 and D in (128, 256) and ops.sigma_is_isotropic(self.prototype_covs):
                shadow, iso = q.ensure_shadow(), True
                if self._em_status is None or self._em_status.device != dev:
                    self._em_status = torch.zeros(1, dtype=torch.int32, device=dev)
            ops.update_gmm(q.bank, q.updated, q.mem_len, mu, sg, wt, st["exp_avg"], st["exp_avg_sq"], self._adam_step_dev,
                           order, sched, stats, n_split, L, self.alpha, lr, b1, b2, eps, self.tau, shadow=shadow,
                           sigma_iso=iso, status=self._em_status)
            self._em_dirty = True
            self._bump_versions()
            return
        ops.em_plan(q.updated, q.mem_len, order, sched, 0, cap, L, adam_step=self._adam_step_dev)
        ops.em_update(None, n_split, cap, order, sched, mu, sg, wt, st["exp_avg"], st["exp_avg_sq"], 0, L, 0,
                      lr, b1, b2, eps, self.tau)
        for i in range(L):
            if r1 > r0:
                ops.em_stats(q.bank, order, mu, sg, wt, self.alpha, stats, n_split, r0, r1)
            else:
                stats.zero_()
            if world > 1:
                import torch.distributed as dist
                dist.all_reduce(stats, group=self.em_group)
            ops.em_update(stats, n_split, cap, order, sched, mu, sg, wt, st["exp_avg"], st["exp_avg_sq"], i, L, 1,
                          lr, b1, b2, eps, self.tau)
        ops.em_update(None, n_split, cap, order, sched, mu, sg, wt, st["exp_avg"], st["exp_avg_sq"], 0, L, 2,
                      lr, b1, b2, eps, self.tau)
        self._em_dirty = True
        self._bump_versions()

    def _bump_versions(self):
        """The EM kernels write the means and the mixture weights through raw pointers: tell torch (autograd's
        saved-tensor checks, and the caches keyed on the version counter such as ops.logprob's prototype operands)."""
        torch.autograd.graph.increment_version(self.prototype_means)
        torch.autograd.graph.increment_version(self.last_layer.weight)

    def _update_GMM_generic(self, order, sched, stats, n_split, r0, r1, world):
        """Any other optimiser: same order of operations as the reference, one optimiser.step()
        per (class, EM loop), fed with the fused gradient.  Host-synchronous (needs the class list)."""
        q = self.queue
        C, K, D = self.prototype_means.shape
        cap, L = q.cap_cls, self.num_em_loop
        mu, sg, wt = self.prototype_means.data, self.prototype_covs.data, self.last_layer.weight.data
        ops.em_plan(q.updated, q.mem_len, order, sched, 0, cap, L)
        active = torch.nonzero(order >= 0).flatten().tolist()
        for c in active:
            one = torch.full_like(order, -1)
            one[c] = 0
            for i in range(L):
                if world > 1:
                    stats.zero_()
                if r1 > r0:
                    ops.em_stats(q.bank, one, mu, sg, wt, self.alpha, stats, n_split, r0, r1)
                if world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(stats, group=self.em_group)
                grad = torch.zeros_like(mu)
                ops.em_update(stats, n_split, cap, one, sched, mu, sg, wt, None, None, i, L, 1, 0.0, 0.9, 0.999,
                              1e-8, self.tau, grad_out=grad, only_class=c)
                self.prototype_optimizer.zero_grad()
                self.prototype_means.grad = grad
                self.prototype_optimizer.step()

    def _check_size(self, x):
        return x.unsqueeze(1) if x.dim() == 2 else x                               # ref :423-427

    def _estimate_log_prob(self, x, mu, var, eps=1e-10):
        """ref model.py:323-336: x [n,D] | [n,1,D], mu/var [1,K,D] -> [n,K,1]."""
        x2 = self._check_size(x).squeeze(1).contiguous()
        out = ops.logprob(x2, mu.detach().reshape(-1, x2.shape[-1]).contiguous(),
                          var.detach().reshape(-1, x2.shape[-1]).contiguous(), MGP_OUT_LOGP_NP, eps=eps, eps_log=eps,
                          math="fp32")
        return out.unsqueeze(-1)

    def _e_step(self, x, mu, var, pi, eps=1e-10):
        """ref model.py:303-321 -> (mean log-likelihood, log_resp [n,K,1])."""
        x2 = self._check_size(x).squeeze(1)
        D = x2.shape[-1]
        log_resp, score = ops.em_estep(x2, mu.detach().reshape(-1, D), var.detach().reshape(-1, D),
                                       pi.detach().reshape(-1))
        return score.mean(), log_resp.unsqueeze(-1)

    def _m_step(self, x, log_resp, eps=1e-10):
        """ref model.py:338-365 -> (pi [1,K,1], mu [1,K,D], var [1,K,D])."""
        x2 = self._check_size(x).squeeze(1)
        pi, mu, var = ops.em_mstep_closed(x2, log_resp.reshape(x2.shape[0], -1), self.alpha)
        return pi.view(1, -1, 1), mu.unsqueeze(0), var.unsqueeze(0)

    def _class_of_view(self, mu_old):
        """The class whose slice of ``prototype_means`` ``mu_old`` views (the reference's autograd finds it through
        the indexing op ``self.prototype_means[_c]``, model.py:295)."""
        p = self.prototype_means
        C, K, D = p.shape
        off = mu_old.data_ptr() - p.data_ptr()
        step = K * D * p.element_size()
        if mu_old.numel() != K * D or off < 0 or off % step != 0 or off // step >= C or \
                mu_old.untyped_storage().data_ptr() != p.untyped_storage().data_ptr():
            raise RuntimeError("_m_step_diversified: mu_old must be a view prototype_means[c] of the parameter the "
                               "prototype optimiser owns (ref model.py:295): the gradient goes to that class")
        return off // step

    def _m_step_diversified(self, x, log_resp, mu_old, var_old, pi_old, eps=1e-10, lamda=1.0):
        """ref model.py:367-401: one diversified M-step = gradient of the GMM loss w.r.t. the class's means (fused
        kernel, equal to the reference's autograd gradient: SURVEY KA6) + ``prototype_optimizer.step()`` on the whole
        mean tensor (zero gradient outside the class, as the reference's backward leaves it).
        -> (pi [1,K,1], mu_old, var_old); sigma untouched, exactly like the reference."""
        if abs(eps - 1e-10) > 1e-16:
            raise RuntimeError("_m_step_diversified: the kernels are built for the reference's eps = 1e-10")
        if self.prototype_optimizer is None:
            raise RuntimeError("_m_step_diversified needs model.prototype_optimizer (ref main.py:223-228)")
        x2 = self._check_size(x).squeeze(1)
        n, D = x2.shape
        c = self._class_of_view(mu_old)
        K = self.num_prototypes_per_class
        with torch.no_grad():
            pi, grad = ops.em_mstep_div(x2.detach(), log_resp.detach().reshape(n, K), mu_old.detach().reshape(K, D),
                                        var_old.detach().reshape(K, D), self.alpha, lamda)
            self.sync_optimizer_state()                      # fold update_GMM's device-side step count in first
            self.prototype_optimizer.zero_grad()
            full = torch.zeros_like(self.prototype_means)
            full[c].copy_(grad)
            self.prototype_means.grad = full
            self.prototype_optimizer.step()
            self._adam_step_seen = None                      # the optimiser stepped outside update_GMM: reseed next time
        return pi.view(1, K, 1), mu_old, var_old

    def global_max_pooling_gmm_topT(self, similarities, conv_features, mine_T=20):
        """ref model.py:188-206: ``similarities`` [B,C,K,H,W] (probabilities), ``conv_features`` [B,D,H,W] ->
        (values [B,P,T] sorted descending, features [B,C,K,D,T], indices [B,C,K,T] int64).  forward() does not call
        this (the fused head mines inside the kernels and never builds the 5 GB feature gather); it exists for code
        written against the reference's method."""
        B, C, K, H, W = similarities.shape
        vals, idx, feats = ops.topt_pool(similarities.detach().reshape(B, C * K, H * W), conv_features.detach(),
                                         int(mine_T), C, K)
        D = conv_features.shape[1]
        return vals, feats.view(B, C, K, D, int(mine_T)), idx.view(B, C, K, int(mine_T)).long()

    def _score(self, x, mu, var, pi, as_average=True, eps=1e-10):
        """ref model.py:403-421."""
        x2 = self._check_size(x).squeeze(1)
        D = x2.shape[-1]
        _, score = ops.em_estep(x2, mu.detach().reshape(-1, D), var.detach().reshape(-1, D), pi.detach().reshape(-1),
                                want_log_resp=False)
        return score.mean() if as_average else score

    # -- reference utilities ------------------------------------------------------------------------
    def set_last_layer_incorrect_connection(self, incorrect_strength):
        """ref model.py:440-447."""
        pos = torch.t(self.prototype_class_identity).to(self.last_layer.weight.device)
        self.last_layer.weight.data.copy_((1.0 / self.num_prototypes_per_class) * pos + incorrect_strength * (1 - pos))

    def initialize_weights(self):
        """ref model.py:449-465."""
        for m in self.add_on_layers.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
        nn.init.kaiming_normal_(self.embedding.weight, mode="fan_out")
        nn.init.constant_(self.embedding.bias, 0)
        self.set_last_layer_incorrect_connection(incorrect_strength=0.0)

    def prune_prototypes_topM(self, top_M=1):
        """ref model.py:467-482: keep, per class, the top_M prototypes by prior; zero the rest of
        last_layer.weight in place (the fused head then ignores them: their pi is 0)."""
        w = self.last_layer.weight
        pos = torch.t(self.prototype_class_identity).to(w.device)
        prior = w[pos == 1].view(self.num_classes, -1)
        thr = torch.topk(prior, top_M, dim=1)[0][:, -1:]
        self.prototypes_to_keep = prior >= thr
        self.prototypes_to_keep_with_negative = w >= thr
        assert (self.prototypes_to_keep.sum(1) >= 1).all()
        w.data[~self.prototypes_to_keep_with_negative] = 0.0


def construct_MGProto(base_architecture, pretrained=True, img_size=224, prototype_shape=(2000, 128, 1, 1),
                      num_classes=200, prototype_activation_function="log", add_on_layers_type="bottleneck",
                      sz_embedding=32, mem_capacity=1000, mine_K=10):
    """ref model.py:485-510."""
    from .backbones import conv_info, proto_layer_rf_info
    features = base_architecture_to_features[base_architecture](pretrained=pretrained)
    ks, st, pd = conv_info(features)
    rf = proto_layer_rf_info(img_size, ks, st, pd, prototype_shape[2])
    return MGProto(features=features, img_size=img_size, prototype_shape=prototype_shape, proto_layer_rf_info=rf,
                   num_classes=num_classes, init_weights=True,
                   prototype_activation_function=prototype_activation_function,
                   add_on_layers_type=add_on_layers_type, sz_embedding=sz_embedding, mem_capacity=mem_capacity,
                   mine_K=mine_K)
