"""GPU parity at the HEADLINE shapes (-m gpu) -- the kernels and code paths bench.py times, against
(1) tests/golden/headline.npz: outputs of the UNMODIFIED reference for these seeded inputs, and
(2) the numpy oracle in float64,
through the reference-facing API over the C ABI: labelled head (tensor-core max/arg-max epilogue over 16 prototype
tiles with classes straddling tile boundaries + head_top1_kernel + head_bwd_kernel), unlabelled head, enqueue into
full ring banks, and update_GMM with ~150 active classes on a pre-seeded Adam state (5 row batches per CTA, the
zero-gradient replay beyond its 131-step cutoff), fused and multi-launch.

Tolerance: 1e-4 (the north star's bound), element-wise relative for logits / log p / pi, norm-wise (max |err| over
max |ref|) for tensors with cancellation (feature gradient, mu, Adam moments); the reference's own fp32 results sit
2e-7 .. 8e-6 norm-wise from the fp64 oracle on these cases (tests/test_oracle_headline.py prints it).  Indices are
bit-exact wherever the reference's top-2 values are separated by more than the fp16x3 log p error."""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

import headline_case as HC

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "headline.npz")
GT_FIXED = (12, 25, 199, 0, 38, 12)
TOL = 1e-4


def _dev():
    return torch.device("cuda:0")


def _t(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=_dev())


def normwise(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / np.abs(b).max())


@pytest.fixture(scope="module")
def hl():
    z = np.load(GOLD)
    g = {k: z[k] for k in z.files}
    C, K, D = (int(g[k]) for k in "C K D".split())
    g["mu"], g["sg"], g["wt"] = HC.mixture(C, K, D)
    g["x"], gt = HC.head_batch(int(g["B"]), C, K, D, int(g["H"]), int(g["W"]), g["mu"], gt_fixed=GT_FIXED)
    assert (gt == g["gt"]).all()
    return g


def _net(C, K, D, T, cap, mu, sg, wt, math, lr=3e-3):
    import mgproto_b200 as M
    net = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 8, 1)), img_size=224, prototype_shape=(C * K, D, 1, 1),
                    proto_layer_rf_info=None, num_classes=C, add_on_layers_type="regular", sz_embedding=8,
                    mem_capacity=cap, mine_K=T).to(_dev())
    net.prototype_means.data.copy_(_t(mu))
    net.prototype_covs.data.copy_(_t(sg))
    net.last_layer.weight.data.copy_(_t(wt))
    net.prototype_optimizer = torch.optim.Adam([{"params": net.prototype_means, "lr": lr}])
    net.math_mode = math
    net.train()
    return net


def _fill_bank(net, rows, short, short_len):
    q = net.queue
    q.bank.copy_(_t(rows))
    q.mem_len.fill_(q.cap_cls)
    q.head.zero_()
    for s in short:
        q.mem_len[int(s)] = short_len
        q.bank[int(s), short_len:] = 0


def _seed_adam(net, am, av, step0):
    p = net.prototype_means
    net.prototype_optimizer.state[p] = {"step": torch.tensor(float(step0)), "exp_avg": _t(am).clone(),
                                        "exp_avg_sq": _t(av).clone()}


def _loss(out, gt):
    import torch.nn.functional as F
    ce0 = F.cross_entropy(out[:, :, 0], gt)
    mine = sum(F.cross_entropy(out[:, :, k], gt) for k in range(1, out.shape[2])) / (out.shape[2] - 1)
    return ce0 + 0.2 * mine                                                  # train_and_test.py:37-41, :55


# ------------------------------------------------------------------------------------------------ head
@pytest.mark.parametrize("math", ["auto", "fp32"])
def test_headline_labelled_step_vs_reference(hl, math):
    """forward(+enqueue) + backward of one labelled batch at P = 2000 (16 prototype tiles), vs the reference's
    logits / loss / feature gradient / own-class and level-0 indices, and the bank rows it pushed."""
    g = hl
    C, K, D, T, cap, B, H, W = (int(g[k]) for k in "C K D T cap B H W".split())
    net = _net(C, K, D, T, cap, g["mu"], g["sg"], g["wt"], math)
    am, av, flags, short, step0 = HC.em_state(C, K, D)
    _fill_bank(net, HC.bank_rows(C, K, D, cap, g["mu"]), short, int(g["short_len"]))
    from mgproto_b200 import ops
    x = _t(g["x"]).requires_grad_(True)
    gt = _t(g["gt"], torch.int64)
    logits, xhat, idx = ops.head_forward(x, net.prototype_means, net.prototype_covs, net.last_layer.weight, gt, T, math)
    loss = _loss(logits, gt)
    loss.backward()
    np.testing.assert_allclose(logits.detach().cpu().numpy(), g["logits"], rtol=TOL, atol=1e-5)
    np.testing.assert_allclose(float(loss), float(g["loss"]), rtol=TOL)
    err = normwise(x.grad.cpu().numpy()[HC.GRAD_X], g["grad_x"])
    print("grad_x norm-wise error vs reference (%s): %.2e" % (math, err))
    assert err < TOL
    # per image too (an image whose gradient is small must not hide behind a large one)
    gx, rx = x.grad.cpu().numpy()[HC.GRAD_X], g["grad_x"]
    for b in range(B):
        assert normwise(gx[b], rx[b]) < 2 * TOL, b
    # indices: level 0 of every prototype, all T levels of the own class
    ix = idx.cpu().numpy()
    sep0 = (np.log(g["top1_val"]) - np.log(g["top2_val"])) > 1e-3
    assert sep0.mean() > 0.9
    assert (ix[:, :, 0][sep0] == g["top1_idx"][sep0]).all()
    for b in range(B):
        c = int(g["gt"][b])
        lv = np.log(g["own_val"][b].astype(np.float64))                       # [K,T] descending
        gap_hi = np.r_["1", np.full((K, 1), np.inf), lv[:, :-1] - lv[:, 1:]]
        gap_lo = np.r_["1", lv[:, :-1] - lv[:, 1:], np.full((K, 1), np.inf)]
        ok = (gap_hi > 1e-3) & (gap_lo > 1e-3)
        ok[:, -1] = False                                                     # the gap below level T-1 is not recorded
        assert ok.mean() > 0.5
        assert (ix[b, c * K:(c + 1) * K][ok] == g["own_idx"][b][ok]).all(), b
    # the model-level call enqueues: bank tails and lengths as the reference left them
    net.head(_t(g["x"]), gt)
    np.testing.assert_array_equal(net.queue.mem_len.cpu().numpy(), g["mem_len_after_enqueue"])
    np.testing.assert_array_equal(net.memory_updated_cls.numpy(), g["updated_after_enqueue"])
    lin = net.queue.linear().cpu().numpy()
    for i, c in enumerate(g["touched"]):
        np.testing.assert_allclose(lin[int(c), -HC.BANK_TAIL:], g["bank_tail"][i], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("math", ["auto", "fp32"])
def test_headline_unlabelled_and_logprob_vs_reference(hl, math):
    g = hl
    C, K, D, T, cap, B, H, W = (int(g[k]) for k in "C K D T cap B H W".split())
    net = _net(C, K, D, T, cap, g["mu"], g["sg"], g["wt"], math)
    from mgproto_b200 import ops
    x = _t(g["x"])
    with torch.no_grad():
        lg0, _, idx0 = ops.head_forward(x, net.prototype_means, net.prototype_covs, net.last_layer.weight, None, T, math)
        l0 = net.head_level0(x)
        xhat, _, _ = ops.normalize_fwd(x)
        lp = net.compute_log_prob(xhat).reshape(-1, C * K)
    np.testing.assert_allclose(lg0.cpu().numpy(), g["logits_nogt"], rtol=TOL, atol=1e-5)
    np.testing.assert_allclose(l0.cpu().numpy(), g["logits_nogt"][:, :, 0], rtol=TOL, atol=1e-5)
    np.testing.assert_allclose(lp[HC.LOGP_ROWS].cpu().numpy(), g["logp_rows"], rtol=TOL, atol=3e-5)
    sep0 = (np.log(g["top1_val"]) - np.log(g["top2_val"])) > 1e-3
    assert (idx0.cpu().numpy()[:, :, 0][sep0] == g["top1_idx"][sep0]).all()


def test_headline_head_vs_fp64_oracle_batch16():
    """A different 16-image batch (other seed, labels on other tile-straddling classes) against the fp64 oracle:
    logits, gradient (oracle.head_backward) and indices."""
    from mgproto_b200 import ops
    from oracle import mgproto_oracle as O
    C, K, D, T, B, H, W = 200, 10, 128, 20, 16, 14, 14
    mu, sg, wt = HC.mixture(C, K, D, seed=12)
    x, gt = HC.head_batch(B, C, K, D, H, W, mu, seed=13, gt_fixed=(51, 63, 64, 76, 89, 102, 115, 127, 140, 153, 166, 179, 191, 198))
    f64 = lambda a: a.astype(np.float64)                                        # noqa: E731
    fw = O.head_forward(f64(x), f64(mu), f64(sg), f64(wt), gt, T)
    gl = np.random.default_rng(3).standard_normal(fw["logits"].shape) / B
    for math in ("auto", "fp32"):
        xd = _t(x).requires_grad_(True)
        logits, _, idx = ops.head_forward(xd, _t(mu), _t(sg), _t(wt), _t(gt, torch.int64), T, math)
        logits.backward(_t(gl))
        np.testing.assert_allclose(logits.detach().cpu().numpy(), fw["logits"], rtol=TOL, atol=1e-5)
        # the gradient goes through the patches the kernel selected; they must be valid top-k picks (value within
        # 1e-4 of the oracle's t-th largest: near-ties may be broken differently, torch.topk's order is undefined)
        gx_ref, dev = O.head_backward(f64(x), f64(mu), f64(sg), f64(wt), gt, T, gl, idx=idx.cpu().numpy())
        assert dev < TOL, dev
        err = normwise(xd.grad.cpu().numpy(), gx_ref)
        print("B=16 grad_x norm-wise error vs fp64 oracle (%s): %.2e (pick deviation %.1e)" % (math, err, dev))
        assert err < TOL
        lpv = np.log(fw["vals"])                                               # after the wrong-class rule; level 0 intact
        srt = -np.sort(-fw["logp"].reshape(B, H * W, C * K).transpose(0, 2, 1), axis=2)
        sep0 = (srt[:, :, 0] - srt[:, :, 1]) > 1e-3
        assert (idx.cpu().numpy()[:, :, 0][sep0] == fw["idx"][:, :, 0][sep0]).all()
        del lpv


# ------------------------------------------------------------------------------------------------ EM
# (em_tc, em_fused, em_pipe) switches of mgp_set_option
EM_PATHS = {"tc": (1, 1, 1), "tc_serial": (1, 1, 0), "fused": (0, 1, 1), "multilaunch": (0, 0, 1)}


class em_path:
    """Select which update_GMM implementation the library takes: tensor-core kernel (csrc/em_tc.cu; pipelined, or one
    tile at a time), fp32 cluster kernel, or the multi-launch path (identical semantics; the tests cross-check them)."""

    def __init__(self, name):
        self.want = EM_PATHS[name]

    def __enter__(self):
        from mgproto_b200 import _lib
        lib = _lib.load()
        self.prev = (lib.mgp_set_option(b"em_tc", self.want[0]), lib.mgp_set_option(b"em_fused", self.want[1]),
                     lib.mgp_set_option(b"em_pipe", self.want[2]))

    def __exit__(self, *a):
        from mgproto_b200 import _lib
        lib = _lib.load()
        lib.mgp_set_option(b"em_tc", self.prev[0])
        lib.mgp_set_option(b"em_fused", self.prev[1])
        lib.mgp_set_option(b"em_pipe", self.prev[2])


def _run_em(g, math, path):
    C, K, D, T, cap = (int(g[k]) for k in "C K D T cap".split())
    net = _net(C, K, D, T, cap, g["mu"], g["sg"], g["wt"], math, lr=float(g["lr"]))
    am, av, flags, short, step0 = HC.em_state(C, K, D)
    _fill_bank(net, HC.bank_rows(C, K, D, cap, g["mu"]), short, int(g["short_len"]))
    _seed_adam(net, am, av, step0)
    with em_path(path):
        with torch.no_grad():
            net.head(_t(g["x"]), _t(g["gt"], torch.int64))                    # the labelled step's enqueue
        outs = []
        for it in range(2):
            net.queue.updated |= _t(flags[it], torch.uint8)
            np.testing.assert_array_equal(net.memory_updated_cls.numpy(), g["flags%d" % it])
            v0 = net.prototype_means._version
            net.update_GMM()
            assert net.prototype_means._version > v0                  # raw-pointer writes are announced to torch
            assert int(net.memory_updated_cls.sum()) == 0
            w = net.last_layer.weight.detach().cpu().numpy()
            outs.append((net.prototype_means.detach().cpu().numpy().copy(),
                         np.stack([w[i, i * K:(i + 1) * K] for i in range(C)])))
        net.sync_optimizer_state()
    return net, outs


@pytest.mark.parametrize("path", ["tc", "tc_serial", "fused", "multilaunch"])
@pytest.mark.parametrize("math", ["auto", "fp32"])
def test_headline_update_gmm_vs_reference(hl, math, path):
    """Two update_GMM calls (156 + 137 active classes, 5 flagged-but-short classes, Adam at step 1000) after the
    labelled step's enqueue: mu, pi, Adam moments and step vs the unmodified reference."""
    g = hl
    net, outs = _run_em(g, math, path)
    (mu0, pi0), (mu1, pi1) = outs
    mu1 = mu1[HC.MU_AFTER1]                                      # the stored samples of the reference's results
    e0, e1 = normwise(mu0[HC.MU_AFTER0], g["mu_after0"]), normwise(mu1, g["mu_after1"])
    print("mu norm-wise error vs reference (%s, %s): %.2e / %.2e" % (math, path, e0, e1))
    assert e0 < TOL and e1 < TOL
    # per class (a class that barely moved must still be right): error relative to that class's largest |mu|
    d = np.abs(mu1.astype(np.float64) - g["mu_after1"]).reshape(mu1.shape[0], -1).max(1)
    s = np.abs(g["mu_after1"]).reshape(mu1.shape[0], -1).max(1)
    assert (d / s).max() < TOL
    # ... and the MOVEMENT itself (mu_after - mu_before), the quantity the update computes
    mv_ref = g["mu_after1"].astype(np.float64) - g["mu"][HC.MU_AFTER1]
    mv_got = mu1.astype(np.float64) - g["mu"][HC.MU_AFTER1]
    assert normwise(mv_got, mv_ref) < 2e-3, normwise(mv_got, mv_ref)
    np.testing.assert_allclose(pi0, g["pi_after0"], rtol=TOL)
    np.testing.assert_allclose(pi1, g["pi_after1"], rtol=TOL)
    st = net.prototype_optimizer.state[net.prototype_means]
    assert int(st["step"]) == int(g["adam_step"])
    em, ev = normwise(st["exp_avg"].cpu().numpy()[HC.ADAM], g["adam_m"]), normwise(st["exp_avg_sq"].cpu().numpy()[HC.ADAM], g["adam_v"])
    print("Adam moments norm-wise error vs reference: %.2e / %.2e" % (em, ev))
    assert em < TOL and ev < TOL


# ---------------------------------------------------------------------------- variants: D = 256, K = 20 / 40
@pytest.mark.parametrize("C,K,D,sigma_mode", [(200, 10, 256, "iso"), (200, 10, 256, "init"), (100, 20, 128, "init"),
                                              (50, 40, 128, "init"), (40, 10, 256, "diag"), (40, 5, 512, "init"),
                                              (40, 10, 64, "diag")])
def test_variant_shapes_head_and_em_vs_fp64_oracle(C, K, D, sigma_mode):
    """BASELINE configs[2]/[3] mixtures: labelled head (fwd + bwd) and one update_GMM against the fp64 oracle."""
    from mgproto_b200 import ops
    from oracle import mgproto_oracle as O
    T, B, H, W, cap = 20, 6, 14, 14, 200
    mu, sg, wt = HC.mixture(C, K, D, seed=20 + K + D, sigma_mode=sigma_mode)
    x, gt = HC.head_batch(B, C, K, D, H, W, mu, seed=21, gt_fixed=(C - 1, 0, min(C - 1, 128 // K), min(C - 1, 256 // K)))
    f64 = lambda a: a.astype(np.float64)                                        # noqa: E731
    fw = O.head_forward(f64(x), f64(mu), f64(sg), f64(wt), gt, T)
    gl = np.random.default_rng(4).standard_normal(fw["logits"].shape) / B
    net = _net(C, K, D, T, cap, mu, sg, wt, "auto")
    xd = _t(x).requires_grad_(True)
    logits, _, idx = ops.head_forward(xd, net.prototype_means, net.prototype_covs, net.last_layer.weight,
                                      _t(gt, torch.int64), T, "auto")
    logits.backward(_t(gl))
    np.testing.assert_allclose(logits.detach().cpu().numpy(), fw["logits"], rtol=TOL, atol=1e-5)
    gx_ref, dev = O.head_backward(f64(x), f64(mu), f64(sg), f64(wt), gt, T, gl, idx=idx.cpu().numpy())
    assert dev < TOL, dev
    assert normwise(xd.grad.cpu().numpy(), gx_ref) < TOL
    with torch.no_grad():
        lg0 = ops.head_forward(_t(x), net.prototype_means, net.prototype_covs, net.last_layer.weight, None, T, "auto")[0]
    fw0 = O.head_forward(f64(x), f64(mu), f64(sg), f64(wt), None, T)
    np.testing.assert_allclose(lg0.cpu().numpy(), fw0["logits"], rtol=TOL, atol=1e-5)
    # EM: all classes flagged, Adam pre-seeded
    rows = HC.bank_rows(C, K, D, cap, mu, seed=22)
    am, av, flags, short, step0 = HC.em_state(C, K, D, seed=23, n_active=(C,), n_short=2, step0=(5000 if D == 256 else 500))
    bank = O.MemoryBankOracle(C, D, cap, dtype=np.float64)
    bank.data[:] = rows
    bank.mem_len[:] = cap
    for s in short:
        bank.mem_len[s] = cap - 11
    adam = O.AdamOracle((C, K, D), lr=3e-3)
    adam.m, adam.v, adam.t = f64(am), f64(av), step0
    mu_ref, wt_ref, _ = O.update_gmm(bank, flags[0], f64(mu), f64(sg), f64(wt), adam)
    for path in ("tc", "tc_serial", "multilaunch"):           # (tc falls through to the fp32 kernels where it does not apply)
        net = _net(C, K, D, T, cap, mu, sg, wt, "auto")
        _fill_bank(net, rows, short, cap - 11)
        _seed_adam(net, am, av, step0)
        net.queue.updated |= _t(flags[0], torch.uint8)
        with em_path(path):
            net.update_GMM()
            net.sync_optimizer_state()
        got = net.prototype_means.detach().cpu().numpy()
        e_mu, e_mv = normwise(got, mu_ref), normwise(got.astype(np.float64) - mu, mu_ref - mu)
        print("variant C%d K%d D%d %s [%s]: mu %.2e movement %.2e" % (C, K, D, sigma_mode, path, e_mu, e_mv))
        assert e_mu < TOL and e_mv < 1e-3, (path, e_mu, e_mv)
        np.testing.assert_allclose(net.last_layer.weight.cpu().numpy(), wt_ref, rtol=TOL, atol=1e-9)
        st = net.prototype_optimizer.state[net.prototype_means]
        assert int(st["step"]) == adam.t
        assert normwise(st["exp_avg"].cpu().numpy(), adam.m) < TOL
        assert normwise(st["exp_avg_sq"].cpu().numpy(), adam.v) < TOL
