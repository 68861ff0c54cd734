"""Tensor-level wrappers over the C ABI (include/mgproto_b200.h).

PyTorch is plumbing here: it owns device memory and streams; every function validates its
tensors (CUDA, fp32, contiguous) and enqueues hand-written sm_100a kernels on the current
stream through ctypes.  Nothing falls back to ATen or to the CPU.
"""
from __future__ import annotations

import os

import torch

from . import _lib
from ._lib import (MGP_MATH_AUTO, MGP_MATH_FP32, MGP_MATH_TC, MGP_MATH_TC_ISO, MGP_MATH_TC_ISO_REUSE, MGP_MATH_TC_REUSE,
                   MGP_MATH_X_STAGED, MGP_MATH_X_STAGED_ISO,
                   MGP_OUT_LOGP_BPHW,
                   MGP_OUT_LOGP_NP, MGP_OUT_NEGP_BPHW, MGP_OUT_TOP1_BP, check)

__all__ = ["normalize_fwd", "logprob", "logprob_top1", "head_select", "head_select_top1", "head_level0", "head_forward", "HeadFunction", "mined_gather", "bank_enqueue",
           "bank_linearize", "bank_shadow_sync", "em_plan", "em_stats", "em_update", "update_gmm", "em_estep", "em_mstep_closed", "em_mstep_div", "topt_pool", "ood_score", "push_argmin", "push_argmin_top1", "mine_cross_entropy",
           "MATH_MODES"]

MATH_MODES = {"fp32": MGP_MATH_FP32, "tc": MGP_MATH_TC, "auto": MGP_MATH_AUTO, "tc_reuse": MGP_MATH_TC_REUSE,
              "tc_iso": MGP_MATH_TC_ISO, "tc_iso_reuse": MGP_MATH_TC_ISO_REUSE}

_iso_cache = {}


def sigma_is_isotropic(sigma: torch.Tensor) -> bool:
    """True if sigma is constant over the feature dim inside every prototype.  One tiny device reduction + host
    read, cached per (storage, version): sigma never changes in the reference's training loop.  A write that does
    not bump the version (through ``.data``) is not seen."""
    # ([C,K,D] and its [P,D] view are the same question: the key leaves the leading shape out)
    key = (sigma.data_ptr(), sigma._version, sigma.numel(), sigma.shape[-1], str(sigma.device))
    hit = _iso_cache.get(key)
    if hit is None:
        if len(_iso_cache) >= 8:
            _iso_cache.clear()
        # the entry keeps sigma alive: a freed block handed to a new tensor (version 0 again) would match the key
        hit = (bool((sigma == sigma[..., :1]).all().item()), sigma)
        _iso_cache[key] = hit
    return hit[0]

_launches = 0          # kernels launched through this module (bench.py reports it as gpu_launches)


def launch_count() -> int:
    return _launches


def _count(n: int):
    global _launches
    _launches += n


_op_device = None      # device of the op being issued: every tensor argument of one op must live on it
_CHECK_ALL = os.environ.get("MGP_CHECK_DEVICES", "0") == "1"


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """Raw handle of the current stream OF THE OP'S DEVICE (not of whatever device happens to be current)."""
    if _raw_stream is not None and _op_device is not None and _op_device.index is not None:
        return _raw_stream(_op_device.index)                 # (no Stream object: ~10x cheaper, called once per launch)
    return torch.cuda.current_stream(_op_device).cuda_stream


class _on_device:
    """Wraps an op: all tensor arguments must share one CUDA device, and the op runs with that device current (the C
    library launches on the current context; a model on cuda:1 called from a thread whose current device is cuda:0
    must not dereference foreign pointers)."""

    def __init__(self, fn):
        self.fn = fn
        self.__name__ = getattr(fn, "__name__", "op")
        self.__doc__ = fn.__doc__

    def __call__(self, *args, **kw):
        global _op_device
        # fast path (one attribute read + one comparison per op): the first tensor argument's device is the current
        # device.  Only when it is not -- or when MGP_CHECK_DEVICES=1 asks for it -- are all tensor arguments checked.
        t0 = args[0] if args else None
        dev = t0.device if isinstance(t0, torch.Tensor) else None
        if dev is not None and not _CHECK_ALL and dev.type == "cuda" and dev.index == torch.cuda.current_device():
            prev, _op_device = _op_device, dev
            try:
                return self.fn(*args, **kw)
            finally:
                _op_device = prev
        dev = None
        for a in list(args) + list(kw.values()):
            if isinstance(a, (tuple, list)):
                cand = [t for t in a if isinstance(t, torch.Tensor)]
            else:
                cand = [a] if isinstance(a, torch.Tensor) else []
            for t in cand:
                if t.is_cuda:
                    if dev is None:
                        dev = t.device
                    elif t.device != dev:
                        raise RuntimeError("mgproto_b200: %s got tensors on %s and %s" % (self.__name__, dev, t.device))
        prev = _op_device
        if dev is None or dev.index == torch.cuda.current_device():
            _op_device = dev
            try:
                return self.fn(*args, **kw)
            finally:
                _op_device = prev
        with torch.cuda.device(dev):
            _op_device = dev
            try:
                return self.fn(*args, **kw)
            finally:
                _op_device = prev


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("mgproto_b200: %s must be a CUDA tensor (there is no CPU path)" % name)
    if t.dtype != dtype:
        raise RuntimeError("mgproto_b200: %s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise RuntimeError("mgproto_b200: %s must be contiguous" % name)
    return t


def _p(t):
    return 0 if t is None else t.data_ptr()


def _math(math) -> int:
    return MATH_MODES[math] if isinstance(math, str) else int(math)


# ----------------------------------------------------------------------------------- a1
@_on_device
def normalize_fwd(x_bdhw: torch.Tensor, want_nchw: bool = False, stage=None):
    """ref model.py:210-211.  -> (xhat [N,D], inv_norm [N], xhat_nchw [B,D,H,W] | None).
    stage = (P, aniso): also write the patch-side operands of the tensor-core log-likelihood kernels in the same pass
    (mgp_normalize_fwd_stage) -> a 4th return value: the workspace to hand to logprob_top1(..., staged=...)."""
    x = _req(x_bdhw, torch.float32, "x")
    B, D, H, W = x.shape
    HW = H * W
    xhat = torch.empty((B * HW, D), device=x.device, dtype=torch.float32)
    inv = torch.empty((B * HW,), device=x.device, dtype=torch.float32)
    nchw = torch.empty_like(x) if want_nchw else None
    lib = _lib.load()
    if stage is not None:
        P, aniso = stage
        nbytes = lib.mgp_logprob_ws_bytes(B, HW, int(P), D, MGP_MATH_TC)
        ws = torch.empty((max(16, nbytes),), device=x.device, dtype=torch.uint8)
        check(lib.mgp_normalize_fwd_stage(x.data_ptr(), xhat.data_ptr(), inv.data_ptr(), _p(nchw), ws.data_ptr(), nbytes,
                                          B, D, HW, int(P), 1 if aniso else 0, _stream()), "mgp_normalize_fwd_stage")
        _count(1)
        return xhat, inv, nchw, ws
    check(lib.mgp_normalize_fwd(x.data_ptr(), xhat.data_ptr(), inv.data_ptr(), _p(nchw), B, D, HW, _stream()),
          "mgp_normalize_fwd")
    _count(1)
    return xhat, inv, nchw


def _stage_for_top1(B, HW, P, D, sg, math):
    """(P, aniso) if the labelled head's max / arg-max kernel will read staged patch operands for this shape and math
    mode (tensor-core path, D <= 128: csrc/logprob_tc.cu), else None."""
    m = _math(math)
    if m not in (MGP_MATH_AUTO, MGP_MATH_TC, MGP_MATH_TC_ISO) or D not in (64, 128) or HW < 32 or HW > 256:
        return None
    if not _lib.load().mgp_has_tensor_core_path():
        return None
    return (P, not sigma_is_isotropic(sg))


# ----------------------------------------------------------------------------------- a2/a3/a16
@_on_device
def logprob(xhat_nd, mu_pd, sigma_pd, layout=MGP_OUT_LOGP_NP, B=None, HW=None, eps=0.0, eps_log=0.0,
            math="auto", ws=None, out=None, return_ws=False):
    """ref model.py:256-275 / :323-336.  xhat [N,D], mu/sigma [P,D] ->
    layout NP: [N,P] log p;  BPHW: [B,P,HW] log p;  NEGP: [B,P,HW] -exp(log p)."""
    x = _req(xhat_nd, torch.float32, "xhat")
    mu = _req(mu_pd, torch.float32, "mu")
    sg = _req(sigma_pd, torch.float32, "sigma")
    N, D = x.shape
    P = mu.shape[0]
    if mu.shape != (P, D) or sg.shape != (P, D):
        raise RuntimeError("mgproto_b200: mu/sigma must be [P, D]")
    if layout == MGP_OUT_LOGP_NP:
        B_, HW_ = N, 1
        shape = (N, P)
    else:
        if B is None or HW is None or B * HW != N:
            raise RuntimeError("mgproto_b200: BPHW layouts need B*HW == N")
        B_, HW_ = B, HW
        shape = (B, P, HW)
    if out is None:
        out = torch.empty(shape, device=x.device, dtype=torch.float32)
    elif tuple(out.shape) != shape:
        raise RuntimeError("mgproto_b200: out has the wrong shape")
    lib = _lib.load()
    m = _math(math)
    if m == MGP_MATH_AUTO:
        # one cached host check (sigma never changes in the reference's loop): isotropic sigma lets the [N,P] layout
        # take the TMEM-resident kernel with the fused operand split (D <= 128) and D = 256 fit the tensor-core tiles
        iso = sigma_is_isotropic(sg)
        if D > 128:
            m = MGP_MATH_TC_ISO if (D == 256 and iso) else MGP_MATH_FP32
        elif iso and D in (64, 128):
            m = MGP_MATH_TC_ISO
    nbytes = lib.mgp_logprob_ws_bytes(B_, HW_, P, D, m)
    # Every call rebuilds the prototype-side operands: mu can be written without a version bump (the reference's
    # push writes through `.data`), so nothing here can tell that cached operands are still current.  A caller that
    # keeps mu / sigma fixed passes math="tc_iso_reuse" and the workspace of a return_ws=True call instead.
    if ws is None:
        ws = torch.empty((max(16, nbytes),), device=x.device, dtype=torch.uint8)
    elif ws.numel() < nbytes:
        raise RuntimeError("mgproto_b200: workspace too small")
    check(lib.mgp_logprob_fwd(x.data_ptr(), mu.data_ptr(), sg.data_ptr(), float(eps), float(eps_log), out.data_ptr(),
                              int(layout), B_, HW_, P, D, m, ws.data_ptr(), nbytes, _stream()), "mgp_logprob_fwd")
    _count(1 if m in (MGP_MATH_TC_REUSE, MGP_MATH_TC_ISO_REUSE) else (3 if nbytes > (P * D + P) * 4 else 2))
    return (out, ws) if return_ws else out


@_on_device
def logprob_top1(xhat_nd, mu_pd, sigma_pd, B, HW, math="auto", ws=None, return_ws=False, staged=None):
    """Per (image, prototype) max / arg-max of log p over the patches, computed in the tensor-core kernel's
    epilogue without writing log p (MGP_OUT_TOP1_BP).  -> packed int64 [B,P] (see include/mgproto_b200.h), or None
    when the tensor-core path does not cover the shape / math mode (the caller then materialises log p).
    staged = (P, aniso) as given to normalize_fwd(stage=...), with its workspace in `ws`: the patch pre-pass is skipped."""
    x = _req(xhat_nd, torch.float32, "xhat")
    mu = _req(mu_pd, torch.float32, "mu")
    sg = _req(sigma_pd, torch.float32, "sigma")
    N, D = x.shape
    P = mu.shape[0]
    if B * HW != N or mu.shape != (P, D) or sg.shape != (P, D):
        raise RuntimeError("mgproto_b200: shape mismatch in logprob_top1")
    m = _math(math)
    if m == MGP_MATH_AUTO and D > 128:
        m = MGP_MATH_TC_ISO if (D == 256 and sigma_is_isotropic(sg)) else MGP_MATH_FP32
    if m == MGP_MATH_FP32 or (m == MGP_MATH_TC_REUSE and ws is None):
        return None
    lib = _lib.load()
    nbytes = lib.mgp_logprob_ws_bytes(B, HW, P, D, m)
    if ws is None:
        ws = torch.empty((max(16, nbytes),), device=x.device, dtype=torch.uint8)
    elif ws.numel() < nbytes:
        raise RuntimeError("mgproto_b200: workspace too small")
    best = torch.empty((B, P), device=x.device, dtype=torch.int64)
    flag = 0
    if staged is not None and ws is not None:
        flag = MGP_MATH_X_STAGED if staged[1] else MGP_MATH_X_STAGED_ISO
    rc = lib.mgp_logprob_fwd(x.data_ptr(), mu.data_ptr(), sg.data_ptr(), 0.0, 0.0, best.data_ptr(), MGP_OUT_TOP1_BP,
                             B, HW, P, D, m | flag, ws.data_ptr(), nbytes, _stream())
    if rc == -2:                                      # MGP_ERR_UNSUPPORTED: no tensor-core path for this shape
        return None
    check(rc, "mgp_logprob_fwd(top1)")
    _count(1 if m == MGP_MATH_TC_REUSE else (2 if flag else 3))
    return (best, ws) if return_ws else best


@_on_device
def head_select_top1(best, xhat_nd, mu_pd, sigma_pd, weight_cp, gt, T, C, K, HW):
    """Labelled head from the packed level-0 results (ref model.py:188-206, :218-222, :254): full top-T only for
    every image's own class (exact fp32 log p of its K prototypes).  -> (logits [B,C,T], vals, idx [B,P,T]);
    of vals/idx only level 0 and the own-class rows are written."""
    B, P = best.shape
    x = _req(xhat_nd, torch.float32, "xhat")
    D = x.shape[1]
    gt = _req(gt, torch.int64, "gt")
    logits = torch.empty((B, C, T), device=x.device, dtype=torch.float32)
    vals = torch.empty((B, P, T), device=x.device, dtype=torch.float32)
    idx = torch.empty((B, P, T), device=x.device, dtype=torch.int32)
    check(_lib.load().mgp_head_select_top1(best.data_ptr(), x.data_ptr(), mu_pd.data_ptr(), sigma_pd.data_ptr(),
                                           weight_cp.data_ptr(), gt.data_ptr(), logits.data_ptr(), vals.data_ptr(),
                                           idx.data_ptr(), B, HW, C, K, D, T, _stream()), "mgp_head_select_top1")
    _count(1)
    return logits, vals, idx


# ----------------------------------------------------------------------------------- a4-a7
@_on_device
def head_select(logp, weight_cp, gt, T, C, K, B=None, HW=None):
    """ref model.py:188-206, :218-222, :254 -> (logits [B,C,T], vals [B,P,T], idx [B,P,T] int32).
    logp is [B,P,HW], or [N,P] (then pass B and HW)."""
    lp = _req(logp, torch.float32, "logp")
    w = _req(weight_cp, torch.float32, "last_layer.weight")
    from_np = lp.dim() == 2
    if from_np:
        N, P = lp.shape
        if B is None or HW is None or B * HW != N:
            raise RuntimeError("mgproto_b200: head_select on [N,P] needs B*HW == N")
    else:
        B, P, HW = lp.shape
    if P != C * K or w.shape != (C, P):
        raise RuntimeError("mgproto_b200: shape mismatch in head_select")
    if gt is not None:
        gt = _req(gt, torch.int64, "gt")
        if gt.shape != (B,):
            raise RuntimeError("mgproto_b200: gt must be [B]")
    logits = torch.empty((B, C, T), device=lp.device, dtype=torch.float32)
    vals = torch.empty((B, P, T), device=lp.device, dtype=torch.float32)
    idx = torch.empty((B, P, T), device=lp.device, dtype=torch.int32)
    fn = _lib.load().mgp_head_select_np if from_np else _lib.load().mgp_head_select
    check(fn(lp.data_ptr(), w.data_ptr(), _p(gt), logits.data_ptr(), vals.data_ptr(), idx.data_ptr(), B, HW, C, K, T,
             _stream()), "mgp_head_select")
    _count(1)
    return logits, vals, idx


class HeadFunction(torch.autograd.Function):
    """features [B,D,H,W] -> log mixture evidences [B,C,T] (ref model.py:210-222, :254).

    Forward = normalise + log-likelihood + top-T + pi-mix, all in the CUDA library.  Backward
    differentiates w.r.t. the features only (mu/sigma are detached in the reference,
    model.py:264-265; last_layer.weight has requires_grad=False) by re-differentiating the T
    selected patches per (image, prototype) instead of saving the N*P*D autograd tape.
    Also returns (non-differentiable) xhat [N,D] and idx [B,P,T] for the bank enqueue.
    """

    @staticmethod
    def forward(ctx, x_add, mu_ckd, sigma_ckd, weight_cp, gt, T, math):
        C, K, D = mu_ckd.shape
        B, _, H, W = x_add.shape
        HW = H * W
        x_add = x_add.contiguous()
        mu = mu_ckd.detach().reshape(C * K, D).contiguous()
        sg = sigma_ckd.detach().reshape(C * K, D).contiguous()
        wt = weight_cp.detach().contiguous()
        # the labelled fast path needs the tensor-core kernel and head_top1_kernel's shared-memory layout to fit
        top1_smem = (2 * C * K + K * T + K * (HW + 1) + 2 * K * D + 2 * K + 4) * 4
        use_top1 = gt is not None and T <= min(32, HW) and HW <= 1024 and top1_smem <= 200 * 1024
        stage = _stage_for_top1(B, HW, C * K, D, sg, math) if use_top1 else None
        if stage is not None:       # one pass: normalise + the fp16 hi/lo operands the max / arg-max kernel reads
            xhat, inv, _, ws1 = normalize_fwd(x_add, stage=stage)
            best = logprob_top1(xhat, mu, sg, B, HW, math, ws=ws1, staged=stage)
        else:
            xhat, inv, _ = normalize_fwd(x_add)
            best = logprob_top1(xhat, mu, sg, B, HW, math) if use_top1 else None
        if best is not None:
            # labelled step: log p never reaches HBM (wrong-class prototypes only need their max, ref model.py:218-221)
            logits, vals, idx = head_select_top1(best, xhat, mu, sg, wt, _req(gt, torch.int64, "gt"), T, C, K, HW)
        else:
            lp = logprob(xhat, mu, sg, MGP_OUT_LOGP_BPHW, B=B, HW=HW, math=math)   # [B,P,HW]: contiguous rows for the mining
            logits, vals, idx = head_select(lp, wt, gt, T, C, K)
        ctx.save_for_backward(logits, vals, idx, wt, gt if gt is not None else torch.empty(0), xhat, inv, mu, sg)
        ctx.has_gt = gt is not None
        ctx.dims = (B, HW, C, K, D, T, H, W)
        ctx.mark_non_differentiable(xhat, idx)
        ctx.set_materialize_grads(False)      # no zero-filled "gradients" for xhat [N,D] / idx [B,P,T] (67 MB of fills)
        return logits, xhat, idx

    @staticmethod
    def backward(ctx, g_logits, _g_xhat, _g_idx):
        if g_logits is None:
            return (None,) * 7
        logits, vals, idx, wt, gt, xhat, inv, mu, sg = ctx.saved_tensors
        B, HW, C, K, D, T, H, W = ctx.dims
        gx = head_backward(g_logits, logits, vals, idx, wt, gt if ctx.has_gt else None, xhat, inv, mu, sg, ctx.dims)
        return gx, None, None, None, None, None, None


@_on_device
def head_backward(g_logits, logits, vals, idx, wt, gt, xhat, inv, mu, sg, dims):
    """d logits / d features through the selected patches only (mgp_head_bwd): -> grad of the add-on features [B,D,H,W]."""
    B, HW, C, K, D, T, H, W = dims
    g = _req(g_logits.contiguous(), torch.float32, "grad_logits")
    lib = _lib.load()
    nbytes = lib.mgp_head_bwd_ws_bytes(B, HW, C * K, D)
    ws = torch.empty((nbytes,), device=g.device, dtype=torch.uint8)
    gx = torch.empty((B, D, H, W), device=g.device, dtype=torch.float32)
    check(lib.mgp_head_bwd(g.data_ptr(), logits.data_ptr(), vals.data_ptr(), idx.data_ptr(), wt.data_ptr(), _p(gt),
                           xhat.data_ptr(), inv.data_ptr(), mu.data_ptr(), sg.data_ptr(), ws.data_ptr(), nbytes,
                           gx.data_ptr(), B, HW, C, K, D, T, _stream()), "mgp_head_bwd")
    _count(3)
    return gx


def head_level0(x_add, mu_ckd, sigma_ckd, weight_cp, math="auto"):
    """Level 0 of the unlabelled head, [B,C] = head_forward(..., gt=None)[0][:, :, 0] -- all the reference's test /
    OoD loop reads (train_and_test.py:182-199: output[:, :, 0]).  Uses the max/arg-max epilogue (no log p matrix, no
    top-T) when the tensor-core path covers the shape; no gradient."""
    C, K, D = mu_ckd.shape
    B, _, H, W = x_add.shape
    HW = H * W
    with torch.no_grad():
        mu = mu_ckd.detach().reshape(C * K, D).contiguous()
        sg = sigma_ckd.detach().reshape(C * K, D).contiguous()
        wt = weight_cp.detach().contiguous()
        fits = HW <= 1024 and (2 * C * K + 2 * K + K * (HW + 1) + 2 * K * D + 2 * K + 4) * 4 <= 200 * 1024
        stage = _stage_for_top1(B, HW, C * K, D, sg, math) if fits else None
        if stage is not None:
            xhat, _, _, ws1 = normalize_fwd(x_add.detach().contiguous(), stage=stage)
            best = logprob_top1(xhat, mu, sg, B, HW, math, ws=ws1, staged=stage)
        else:
            xhat, _, _ = normalize_fwd(x_add.detach().contiguous())
            best = logprob_top1(xhat, mu, sg, B, HW, math) if fits else None
        if best is None:
            lp = logprob(xhat, mu, sg, MGP_OUT_LOGP_BPHW, B=B, HW=HW, math=math)
            return head_select(lp, wt, None, 1, C, K)[0][:, :, 0]
        none = torch.full((B,), -1, dtype=torch.int64, device=x_add.device)     # no own class: every class keeps level 0 only
        return head_select_top1(best, xhat, mu, sg, wt, none, 1, C, K, HW)[0][:, :, 0]


def head_forward(x_add, mu_ckd, sigma_ckd, weight_cp, gt, T, math="auto"):
    return HeadFunction.apply(x_add, mu_ckd, sigma_ckd, weight_cp, gt, int(T), math)


# ----------------------------------------------------------------------------------- a8/a9
def _rec_stride(K, D):
    """fp32 words of one packed per-image record [rows K*D | top1 K (int32 bits) | gt (int64 bits) | pad]: a multiple
    of 4 (16-byte row alignment for the vector loads) with the int64 on an 8-byte boundary."""
    return ((K * D + K + 1) // 2 * 2 + 2 + 3) // 4 * 4


def _rec_views(rec, K, D):
    """(rows [b, K*D] fp32, top1 [b, K] int32, gt [b] int64) views into packed records [b, stride]."""
    off = (K * D + K + 1) // 2 * 2
    rows = rec[:, :K * D]
    top1 = rec.view(torch.int32)[:, K * D:K * D + K]
    gt = rec.view(torch.int64)[:, off // 2]
    return rows, top1, gt


@_on_device
def mined_gather(xhat_nd, idx, gt, HW, C, K, packed=False):
    """ref model.py:225-226: (top1 [B,K] int32, rows [B,K,D]) of every image's GT-class prototypes.  packed=True: the
    kernel writes them straight into per-image records [B, _rec_stride(K, D)] (+ the label), the unit a batch-sharded run
    all-gathers (parallel.py); returns (records, top1 view, rows view)."""
    _req(xhat_nd, torch.float32, "xhat")
    _req(idx, torch.int32, "idx")
    _req(gt, torch.int64, "gt")
    B, P, T = idx.shape
    D = xhat_nd.shape[1]
    lib = _lib.load()
    if packed:
        rs = _rec_stride(K, D)
        rec = torch.empty((B, rs), device=idx.device, dtype=torch.float32)
        rows, top1, gtv = _rec_views(rec, K, D)
        gtv.copy_(gt)
        check(lib.mgp_mined_gather(xhat_nd.data_ptr(), idx.data_ptr(), gt.data_ptr(), top1.data_ptr(), rows.data_ptr(), rs, rs,
                                   B, HW, C, K, D, T, _stream()), "mgp_mined_gather")
        _count(1)
        return rec, top1, rows
    top1 = torch.empty((B, K), device=idx.device, dtype=torch.int32)
    rows = torch.empty((B, K, D), device=idx.device, dtype=torch.float32)
    check(lib.mgp_mined_gather(xhat_nd.data_ptr(), idx.data_ptr(), gt.data_ptr(), top1.data_ptr(), rows.data_ptr(), 0, 0,
                               B, HW, C, K, D, T, _stream()), "mgp_mined_gather")
    _count(1)
    return top1, rows


@_on_device
def bank_enqueue(bank, mem_len, head, updated, rows, top1, gt, shadow=None):
    """ref model.py:228-250 + utils/memory.py:31-73, in place on (bank, mem_len, head, updated); ``shadow`` =
    (shadow_h, shadow_l, shadow_xx) keeps the tensor-core operand copy of the bank in step (MemoryBank.ensure_shadow).
    rows / top1 / gt may be the strided views of packed records (`_rec_views`): they are read in place."""
    bank = _req(bank, torch.float32, "bank")
    C, cap, D = bank.shape
    B, K = top1.shape
    _req(mem_len, torch.int64, "mem_len")
    _req(head, torch.int32, "head")
    _req(updated, torch.uint8, "updated")
    for t, dt, nm in ((rows, torch.float32, "rows"), (top1, torch.int32, "top1"), (gt, torch.int64, "gt")):
        if not t.is_cuda or t.dtype != dt:
            raise RuntimeError("mgproto_b200: %s must be a CUDA %s tensor" % (nm, dt))
    if rows.numel() != B * K * D or gt.shape != (B,) or rows.stride(-1) != 1 or top1.stride(-1) != 1:
        raise RuntimeError("mgproto_b200: enqueue shape mismatch")
    rs = rows.stride(0) if B > 1 else 0
    ts = top1.stride(0) if B > 1 else 0
    gs = gt.stride(0) if B > 1 else 0
    lib = _lib.load()
    plan = torch.empty((int(lib.mgp_bank_enqueue_plan_ints(B, C, K)),), device=bank.device, dtype=torch.int32)
    sh = shadow if shadow is not None else (None, None, None)
    check(lib.mgp_bank_enqueue(bank.data_ptr(), mem_len.data_ptr(), head.data_ptr(), updated.data_ptr(),
                                       rows.data_ptr(), top1.data_ptr(), gt.data_ptr(), int(rs), int(ts), int(gs),
                                       plan.data_ptr(), _p(sh[0]), _p(sh[1]), _p(sh[2]), B, C, K, D, cap, _stream()),
          "mgp_bank_enqueue")
    _count(3)


@_on_device
def bank_shadow_sync(bank, shadow_h, shadow_l, shadow_xx):
    """(Re)build the fp16 hi/lo + |row|^2 shadow of the whole bank (include/mgproto_b200.h: mgp_bank_shadow_sync)."""
    bank = _req(bank, torch.float32, "bank")
    C, cap, D = bank.shape
    _req(shadow_h, torch.float16, "shadow_h")
    _req(shadow_l, torch.float16, "shadow_l")
    _req(shadow_xx, torch.float32, "shadow_xx")
    check(_lib.load().mgp_bank_shadow_sync(bank.data_ptr(), shadow_h.data_ptr(), shadow_l.data_ptr(), shadow_xx.data_ptr(),
                                           C, cap, D, _stream()), "mgp_bank_shadow_sync")
    _count(1)


@_on_device
def bank_linearize(bank, mem_len, head):
    bank = _req(bank, torch.float32, "bank")
    C, cap, D = bank.shape
    lin = torch.empty_like(bank)
    check(_lib.load().mgp_bank_linearize(bank.data_ptr(), mem_len.data_ptr(), head.data_ptr(), lin.data_ptr(), C, cap,
                                         D, _stream()), "mgp_bank_linearize")
    _count(1)
    return lin


# ----------------------------------------------------------------------------------- a10-a14
def em_stat_stride(K, D, with_s2=False) -> int:
    return int(_lib.load().mgp_em_stat_stride(K, D, 1 if with_s2 else 0))


@_on_device
def em_plan(updated, mem_len, order, sched, step0, cap, num_em_loop, adam_step=None):
    C = updated.numel()
    check(_lib.load().mgp_em_plan(updated.data_ptr(), mem_len.data_ptr(), order.data_ptr(), sched.data_ptr(),
                                  _p(adam_step), int(step0), C, int(cap), int(num_em_loop), _stream()), "mgp_em_plan")
    _count(1)


@_on_device
def em_stats(bank, order, mu_ckd, sigma_ckd, weight_cp, alpha, stats, n_split, row_begin=0, row_end=None,
             with_s2=False):
    C, cap, D = bank.shape
    K = mu_ckd.shape[1]
    if row_end is None:
        row_end = cap
    check(_lib.load().mgp_em_stats(bank.data_ptr(), order.data_ptr(), mu_ckd.data_ptr(), sigma_ckd.data_ptr(),
                                   weight_cp.data_ptr(), float(alpha), int(row_begin), int(row_end), int(n_split),
                                   1 if with_s2 else 0, stats.data_ptr(), C, K, D, cap, _stream()), "mgp_em_stats")
    _count(1)


@_on_device
def em_update(stats, n_split, n_rows_total, order, sched, mu_ckd, sigma_ckd, weight_cp, exp_avg, exp_avg_sq, em_loop,
              num_em_loop, phase, lr, beta1, beta2, adam_eps, tau, lamda=1.0, grad_out=None, only_class=-1,
              with_s2=False):
    C, K, D = mu_ckd.shape
    check(_lib.load().mgp_em_update(_p(stats), int(n_split), 1 if with_s2 else 0, int(n_rows_total), order.data_ptr(),
                                    sched.data_ptr(), mu_ckd.data_ptr(), sigma_ckd.data_ptr(), weight_cp.data_ptr(),
                                    _p(exp_avg), _p(exp_avg_sq), int(em_loop), int(num_em_loop), int(phase), float(lr),
                                    float(beta1), float(beta2), float(adam_eps), float(tau), float(lamda),
                                    _p(grad_out), int(only_class), C, K, D, _stream()), "mgp_em_update")
    _count(1)


@_on_device
def update_gmm(bank, updated, mem_len, mu_ckd, sigma_ckd, weight_cp, exp_avg, exp_avg_sq, adam_step, order, sched, stats,
               n_split, num_em_loop, alpha, lr, beta1, beta2, adam_eps, tau, lamda=1.0, shadow=None, sigma_iso=False,
               status=None):
    """ref model.py:277-301, single replica: plan + zero-gradient replays + num_em_loop x (stats, step) in one call.
    With ``shadow`` (MemoryBank.ensure_shadow()), ``sigma_iso`` and a device int32 ``status`` word the supported
    shapes run on the tensor cores (csrc/em_tc.cu)."""
    C, cap, D = bank.shape
    K = mu_ckd.shape[1]
    sh = shadow if shadow is not None else (None, None, None)
    tc = shadow is not None and sigma_iso and status is not None
    check(_lib.load().mgp_update_gmm(bank.data_ptr(), _p(sh[0]), _p(sh[1]), _p(sh[2]), 1 if sigma_iso else 0, _p(status),
                                     updated.data_ptr(), mem_len.data_ptr(), mu_ckd.data_ptr(),
                                     sigma_ckd.data_ptr(), weight_cp.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                     adam_step.data_ptr(), order.data_ptr(), sched.data_ptr(), stats.data_ptr(),
                                     int(n_split), int(num_em_loop), float(alpha), float(lr), float(beta1), float(beta2),
                                     float(adam_eps), float(tau), float(lamda), C, K, D, cap, _stream()), "mgp_update_gmm")
    _count(int(_lib.load().mgp_update_gmm_launches(K, D, cap, int(num_em_loop), 1 if tc else 0)))


@_on_device
def em_estep(x_nd, mu_kd, sigma_kd, pi_k, want_log_resp=True, want_score=True):
    """ref model.py:303-321 / :403-421 -> (log_resp [n,K] | None, score [n] | None)."""
    x = _req(x_nd.contiguous(), torch.float32, "x")
    mu = _req(mu_kd.contiguous(), torch.float32, "mu")
    sg = _req(sigma_kd.contiguous(), torch.float32, "sigma")
    pi = _req(pi_k.contiguous(), torch.float32, "pi")
    n, D = x.shape
    K = mu.shape[0]
    lr = torch.empty((n, K), device=x.device, dtype=torch.float32) if want_log_resp else None
    sc = torch.empty((n,), device=x.device, dtype=torch.float32) if want_score else None
    check(_lib.load().mgp_em_estep(x.data_ptr(), mu.data_ptr(), sg.data_ptr(), pi.data_ptr(), _p(lr), _p(sc), n, K, D,
                                   _stream()), "mgp_em_estep")
    _count(1)
    return lr, sc


@_on_device
def em_mstep_closed(x_nd, log_resp_nk, alpha):
    """ref model.py:338-365 -> (pi [K], mu [K,D], sigma [K,D])."""
    x = _req(x_nd.contiguous(), torch.float32, "x")
    lr = _req(log_resp_nk.contiguous(), torch.float32, "log_resp")
    n, D = x.shape
    K = lr.shape[1]
    pi = torch.empty((K,), device=x.device, dtype=torch.float32)
    mu = torch.empty((K, D), device=x.device, dtype=torch.float32)
    sg = torch.empty((K, D), device=x.device, dtype=torch.float32)
    check(_lib.load().mgp_em_mstep_closed(x.data_ptr(), lr.data_ptr(), float(alpha), pi.data_ptr(), mu.data_ptr(),
                                          sg.data_ptr(), n, K, D, _stream()), "mgp_em_mstep_closed")
    _count(1)
    return pi, mu, sg


@_on_device
def em_mstep_div(x_nd, log_resp_nk, mu_kd, sigma_kd, alpha, lamda=1.0):
    """ref model.py:367-401 on explicit rows -> (pi_new [K], grad [K,D] = d gmm_loss / d mu)."""
    x = _req(x_nd.contiguous(), torch.float32, "x")
    lr = _req(log_resp_nk.contiguous(), torch.float32, "log_resp")
    mu = _req(mu_kd.contiguous(), torch.float32, "mu")
    sg = _req(sigma_kd.contiguous(), torch.float32, "sigma")
    n, D = x.shape
    K = mu.shape[0]
    if lr.shape != (n, K) or mu.shape != (K, D) or sg.shape != (K, D):
        raise RuntimeError("mgproto_b200: shape mismatch in em_mstep_div")
    ws = torch.empty((n, K), device=x.device, dtype=torch.float32)
    pi = torch.empty((K,), device=x.device, dtype=torch.float32)
    grad = torch.empty((K, D), device=x.device, dtype=torch.float32)
    check(_lib.load().mgp_em_mstep_div(x.data_ptr(), lr.data_ptr(), mu.data_ptr(), sg.data_ptr(), float(alpha),
                                       float(lamda), ws.data_ptr(), pi.data_ptr(), grad.data_ptr(), n, K, D, _stream()),
          "mgp_em_mstep_div")
    _count(2)
    return pi, grad


@_on_device
def topt_pool(sims_bphw, x_nchw, T, C, K, want_feats=True):
    """ref model.py:188-206 on probabilities [B,P,HW] -> (vals [B,P,T], idx [B,P,T] int32, feats [B,P,D,T] | None)."""
    sm = _req(sims_bphw.contiguous(), torch.float32, "similarities")
    B, P, HW = sm.shape
    if P != C * K:
        raise RuntimeError("mgproto_b200: shape mismatch in topt_pool")
    vals = torch.empty((B, P, T), device=sm.device, dtype=torch.float32)
    idx = torch.empty((B, P, T), device=sm.device, dtype=torch.int32)
    feats, xp, D = None, 0, 1
    if want_feats:
        x = _req(x_nchw.contiguous(), torch.float32, "conv_features")
        D = x.shape[1]
        if x.shape[0] != B or x.numel() != B * D * HW:
            raise RuntimeError("mgproto_b200: conv_features must be [B,D,H,W] with H*W == HW")
        feats = torch.empty((B, P, D, T), device=sm.device, dtype=torch.float32)
        xp = x.data_ptr()
    check(_lib.load().mgp_topt_pool(sm.data_ptr(), xp, vals.data_ptr(), idx.data_ptr(), _p(feats), B, HW, C, K, D, int(T),
                                    _stream()), "mgp_topt_pool")
    _count(2 if want_feats else 1)
    return vals, idx, feats


@_on_device
def ood_score(out0):
    """ref train_and_test.py:184-199, :212-213 on level-0 log evidences [B,C] (any strides): -> (p_sum [B], p_mean [B],
    pred [B] int64)."""
    if not out0.is_cuda or out0.dtype != torch.float32 or out0.dim() != 2:
        raise RuntimeError("mgproto_b200: out0 must be a CUDA fp32 [B, C] tensor")
    B, C = out0.shape
    ps = torch.empty((B,), device=out0.device, dtype=torch.float32)
    pm = torch.empty((B,), device=out0.device, dtype=torch.float32)
    pred = torch.empty((B,), device=out0.device, dtype=torch.int64)
    check(_lib.load().mgp_ood_score(out0.data_ptr(), out0.stride(0), out0.stride(1), ps.data_ptr(), pm.data_ptr(),
                                    pred.data_ptr(), B, C, _stream()), "mgp_ood_score")
    _count(1)
    return ps, pm, pred


# ----------------------------------------------------------------------------------- a17 (optional)
@_on_device
def _mine_ce(out, gt, mine_coef):
    o = _req(out.contiguous(), torch.float32, "output")
    g = _req(gt.contiguous(), torch.int64, "target")
    B, C, T = o.shape
    loss_b = torch.empty((B,), device=o.device, dtype=torch.float32)
    grad = torch.empty_like(o)
    check(_lib.load().mgp_mine_ce(o.data_ptr(), g.data_ptr(), loss_b.data_ptr(), grad.data_ptr(), B, C, T,
                                  float(mine_coef), _stream()), "mgp_mine_ce")
    _count(1)
    return loss_b, grad


class MineCEFunction(torch.autograd.Function):
    """loss = CE(out[:,:,0], gt) + mine_coef * mean_{t>=1} CE(out[:,:,t], gt) (ref train_and_test.py:37-41,:55)
    with value and gradient from one kernel."""

    @staticmethod
    def forward(ctx, out, gt, mine_coef):
        loss_b, grad = _mine_ce(out, gt, mine_coef)
        ctx.save_for_backward(grad)
        return loss_b.sum()

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return grad * g, None, None


def mine_cross_entropy(out, gt, mine_coef=0.2):
    return MineCEFunction.apply(out, gt, float(mine_coef))


# ----------------------------------------------------------------------------------- f1
@_on_device
def push_argmin_top1(best_bp, labels, C, K):
    """ref push.py:125-158 from the packed top-1 results of logprob_top1 -> (arg [B,K] int32, val [B,K] = -p there)."""
    best = _req(best_bp, torch.int64, "best")
    lab = _req(labels, torch.int64, "labels")
    B = best.shape[0]
    arg = torch.empty((B, K), device=best.device, dtype=torch.int32)
    val = torch.empty((B, K), device=best.device, dtype=torch.float32)
    check(_lib.load().mgp_push_argmin_top1(best.data_ptr(), lab.data_ptr(), arg.data_ptr(), val.data_ptr(), B, C, K,
                                           _stream()), "mgp_push_argmin_top1")
    _count(1)
    return arg, val


@_on_device
def push_argmin(logp_bphw, labels, C, K):
    """ref push.py:125-158 -> (arg [B,K] int32 flat HW index, val [B,K] = -p at the argmin)."""
    lp = _req(logp_bphw, torch.float32, "logp")
    lab = _req(labels, torch.int64, "labels")
    B, P, HW = lp.shape
    arg = torch.empty((B, K), device=lp.device, dtype=torch.int32)
    val = torch.empty((B, K), device=lp.device, dtype=torch.float32)
    check(_lib.load().mgp_push_argmin(lp.data_ptr(), lab.data_ptr(), arg.data_ptr(), val.data_ptr(), B, HW, C, K,
                                      _stream()), "mgp_push_argmin")
    _count(1)
    return arg, val
