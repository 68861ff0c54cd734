"""GPU parity tests proper (-m gpu): the CUDA path, called through the C ABI, against
(1) the committed golden fixtures produced by the unmodified reference and (2) the numpy
oracle on seeded inputs.  Tolerance: 1e-4 relative on fp32 results (the north-star bound),
indices bit-exact wherever the reference's adjacent top-T values are separated."""
import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

RTOL = 1e-4


def _dev():
    return torch.device("cuda:0")


def _t(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=_dev())


def _model_from(g, math="fp32"):
    import mgproto_b200 as M
    C, K, D, T, cap = (int(g[k]) for k in "C K D T cap".split())
    net = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 16, 1)), img_size=14, prototype_shape=(C * K, D, 1, 1),
                    proto_layer_rf_info=None, num_classes=C, add_on_layers_type="regular", sz_embedding=8,
                    mem_capacity=cap, mine_K=T).to(_dev())
    net.prototype_means.data.copy_(_t(g["mu0"]))
    net.prototype_covs.data.copy_(_t(g["sigma"]))
    net.last_layer.weight.data.copy_(_t(g["weight0"]))
    net.prototype_optimizer = torch.optim.Adam([{"params": net.prototype_means, "lr": float(g["lr"])}])
    net.math_mode = math
    net.train()
    return net


def _loss(out, gt):
    ce0 = F.cross_entropy(out[:, :, 0], gt)
    mine = sum(F.cross_entropy(out[:, :, k], gt) for k in range(1, out.shape[2])) / (out.shape[2] - 1)
    return ce0 + 0.2 * mine


def _separated(v):
    v = v.astype(np.float64)
    rel = np.abs(np.diff(v, axis=-1)) > 1e-5 * np.abs(v[..., :-1])
    a = np.ones_like(v, dtype=bool)
    b = np.ones_like(v, dtype=bool)
    a[..., 1:] = rel
    b[..., :-1] = rel
    return a & b


def test_library_loaded_and_abi():
    from mgproto_b200 import _lib
    lib = _lib.load()
    assert lib.mgp_abi_version() == 2


def test_normalize(golden):
    from mgproto_b200 import ops
    from oracle import mgproto_oracle as O
    x = golden["it0_x_add"]
    xhat, inv, nchw = ops.normalize_fwd(_t(x), want_nchw=True)
    ref = O.l2_normalize(x.astype(np.float64), axis=1)
    np.testing.assert_allclose(nchw.cpu().numpy(), ref, rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(xhat.cpu().numpy(), O.features_to_rows(ref), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(nchw.cpu().numpy()[golden["sample"]], golden["it0_push_feat"], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("math", ["fp32", "auto"])
def test_compute_log_prob_golden(golden, math):
    g = golden
    net = _model_from(g, math)
    net.prototype_means.data.copy_(_t(g["it0_mu"]))
    from mgproto_b200 import ops
    xhat, _, _ = ops.normalize_fwd(_t(g["it0_x_add"]))
    lp = net.compute_log_prob(xhat)
    np.testing.assert_allclose(lp.cpu().numpy(), g["it0_logp"], rtol=RTOL, atol=1e-5)


@pytest.mark.parametrize("math", ["fp32", "auto"])
def test_push_forward_golden(golden, math):
    g = golden
    net = _model_from(g, math)
    net.prototype_means.data.copy_(_t(g["it0_mu"]))
    feat, dist = net.push_forward_features(_t(g["it0_x_add"]))
    np.testing.assert_allclose(feat.cpu().numpy()[g["sample"]], g["it0_push_feat"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(dist.cpu().numpy(), g["it0_push_dist"], rtol=RTOL, atol=1e-9)
    # f1: device-side projection search == argmin over the reference's distance map
    from oracle import mgproto_oracle as O
    arg, val, _ = net.push_search(_t(g["it0_x_add"]), _t(g["it0_gt"], torch.int64))
    oi, ov = O.push_argmin(g["it0_push_dist"], g["it0_gt"], int(g["K"]))
    np.testing.assert_allclose(val.cpu().numpy(), ov, rtol=RTOL, atol=1e-9)
    d = g["it0_push_dist"]
    B, P, H, W = d.shape
    got = arg.cpu().numpy()
    for b in range(B):
        c = int(g["it0_gt"][b])
        for k in range(int(g["K"])):
            row = d[b, c * int(g["K"]) + k].reshape(-1)
            assert row[got[b, k]] <= row.min() * (1 - 1e-5) or got[b, k] == oi[b, k]


@pytest.mark.parametrize("math", ["fp32", "auto"])
def test_head_forward_golden(golden, math):
    g = golden
    net = _model_from(g, math)
    net.prototype_means.data.copy_(_t(g["it0_mu"]))
    from mgproto_b200 import ops
    x = _t(g["it0_x_add"])
    gt = _t(g["it0_gt"], torch.int64)
    with torch.no_grad():
        lg, xhat, idx = ops.head_forward(x, net.prototype_means, net.prototype_covs, net.last_layer.weight, gt,
                                         net.mine_T, math)
        lg0, _, idx0 = ops.head_forward(x, net.prototype_means, net.prototype_covs, net.last_layer.weight, None,
                                        net.mine_T, math)
    np.testing.assert_allclose(lg.cpu().numpy(), g["it0_logits"], rtol=RTOL, atol=1e-6)
    np.testing.assert_allclose(lg0.cpu().numpy(), g["it0_logits_nogt"], rtol=RTOL, atol=1e-6)
    sep = _separated(g["it0_topk_vals"])
    assert sep.mean() > 0.5
    assert (idx0.cpu().numpy()[sep] == g["it0_topk_idx"][sep]).all()          # bit-exact indices
    # KA4: with gt, wrong-class columns of levels t>=1 equal level 0
    L = lg.cpu().numpy()
    B, C, T = L.shape
    for b in range(B):
        for c in range(C):
            if c != int(g["it0_gt"][b]):
                np.testing.assert_array_equal(L[b, c, 1:], np.repeat(L[b, c, :1], T - 1))
            else:
                assert (np.diff(L[b, c]) <= 1e-6).all()


def test_head_values_and_indices_vs_oracle(golden):
    g = golden
    from mgproto_b200 import ops
    from oracle import mgproto_oracle as O
    C, K, D, T = (int(g[k]) for k in "C K D T".split())
    B, _, H, W = g["it0_x_add"].shape
    xhat, _, _ = ops.normalize_fwd(_t(g["it0_x_add"]))
    lp = ops.logprob(xhat, _t(g["it0_mu"]).view(C * K, D), _t(g["sigma"]).view(C * K, D), 1, B=B, HW=H * W,
                     math="fp32")
    _, vals, idx = ops.head_select(lp, _t(g["it0_weight"]), None, T, C, K)
    np.testing.assert_allclose(vals.cpu().numpy(), g["it0_topk_vals"], rtol=RTOL, atol=1e-12)
    fw = O.head_forward(g["it0_x_add"].astype(np.float64), g["it0_mu"].astype(np.float64),
                        g["sigma"].astype(np.float64), g["it0_weight"].astype(np.float64), None, T)
    sep = _separated(fw["vals"])
    assert (idx.cpu().numpy()[sep] == fw["idx"][sep]).all()


@pytest.mark.parametrize("math", ["fp32", "auto"])
def test_head_backward_golden(golden, math):
    g = golden
    net = _model_from(g, math)
    for it in range(int(g["iters"])):
        pre = "it%d_" % it
        net.prototype_means.data.copy_(_t(g[pre + "mu"]))
        net.last_layer.weight.data.copy_(_t(g[pre + "weight"]))
        x = _t(g[pre + "x_add"]).requires_grad_(True)
        gt = _t(g[pre + "gt"], torch.int64)
        out = net.head(x, gt)
        loss = _loss(out, gt)
        loss.backward()
        np.testing.assert_allclose(out.detach().cpu().numpy(), g[pre + "logits"], rtol=RTOL, atol=1e-6)
        np.testing.assert_allclose(float(loss), float(g[pre + "loss"]), rtol=RTOL)
        ref = g[pre + "grad_x"]
        np.testing.assert_allclose(x.grad.cpu().numpy()[g["sample"]], ref, rtol=2e-3, atol=2e-4 * np.abs(ref).max())


@pytest.mark.parametrize("math", ["fp32", "auto"])
@pytest.mark.parametrize("em_path", ["fused", "generic"])
def test_training_sequence_bank_and_em(golden, em_path, math):
    """forward -> enqueue -> update_GMM over the fixture's iterations: bank contents, mem_len,
    update flags, mu, pi and the Adam state follow the reference step for step (KA7 included)."""
    g = golden
    net = _model_from(g, math)
    C, K, D, cap = (int(g[k]) for k in "C K D cap".split())
    if em_path == "generic":
        class AdamSub(torch.optim.Adam):      # not `type is Adam` -> host-driven generic path
            pass
        net.prototype_optimizer = AdamSub([{"params": net.prototype_means, "lr": float(g["lr"])}])
    for it in range(int(g["iters"])):
        pre = "it%d_" % it
        np.testing.assert_allclose(net.prototype_means.detach().cpu().numpy(), g[pre + "mu"], rtol=RTOL, atol=2e-6)
        np.testing.assert_allclose(net.last_layer.weight.detach().cpu().numpy(), g[pre + "weight"], rtol=RTOL,
                                   atol=1e-7)
        x = _t(g[pre + "x_add"])
        gt = _t(g[pre + "gt"], torch.int64)
        with torch.no_grad():
            net.head(x, gt)
        np.testing.assert_array_equal(net.queue.mem_len.cpu().numpy(), g[pre + "mem_len"])
        np.testing.assert_array_equal(net.memory_updated_cls.numpy(), g[pre + "updated"])
        sd = net.state_dict()
        for c in range(C):
            n = int(g[pre + "mem_len"][c])
            np.testing.assert_allclose(sd["queue.cls%d" % c].cpu().numpy()[:n], g[pre + "bank"][c, :n], rtol=1e-5,
                                       atol=1e-6)
        if int(net.queue.mem_len.sum()) > 0:                                   # train_and_test.py:61-63
            net.update_GMM()
        assert int(net.memory_updated_cls.sum()) == 0                          # ref model.py:301
        np.testing.assert_allclose(net.prototype_means.detach().cpu().numpy(), g[pre + "mu_after"], rtol=RTOL,
                                   atol=2e-6)
        np.testing.assert_allclose(net.last_layer.weight.detach().cpu().numpy(), g[pre + "weight_after"], rtol=RTOL,
                                   atol=1e-7)
        assert float(net.iteration_counter) == it + 1
    if em_path == "fused":
        net.sync_optimizer_state()
    st = net.prototype_optimizer.state[net.prototype_means]
    assert int(st["step"]) == int(g["adam_step"])
    np.testing.assert_allclose(st["exp_avg"].cpu().numpy(), g["adam_m"], rtol=1e-3, atol=1e-7)
    np.testing.assert_allclose(st["exp_avg_sq"].cpu().numpy(), g["adam_v"], rtol=1e-3, atol=1e-10)
    # KA2: every class's pi row sums to 1
    w = net.last_layer.weight.detach().cpu().numpy()
    np.testing.assert_allclose(w.sum(1), 1.0, rtol=1e-5)


def test_em_building_blocks(golden):
    g = golden
    net = _model_from(g, "fp32")
    K = int(g["K"])
    x, mu, sg, pi = _t(g["em_x"]), _t(g["em_mu"]), _t(g["em_sigma"]), _t(g["em_pi"])
    ll, log_resp = net._e_step(x, mu, sg, pi)
    np.testing.assert_allclose(float(ll), float(g["em_loglik"]), rtol=1e-5)
    np.testing.assert_allclose(log_resp.cpu().numpy(), g["em_log_resp"], rtol=RTOL, atol=1e-5)
    p, m, v = net._m_step(x, _t(g["em_log_resp"]))
    np.testing.assert_allclose(p.cpu().numpy(), g["em_mstep_pi"], rtol=1e-5)
    np.testing.assert_allclose(m.cpu().numpy(), g["em_mstep_mu"], rtol=RTOL, atol=1e-6)
    np.testing.assert_allclose(v.cpu().numpy(), g["em_mstep_var"], rtol=2e-3, atol=2e-5)
    sc = net._score(x.unsqueeze(1), mu, sg, pi, as_average=False)
    np.testing.assert_allclose(sc.cpu().numpy(), g["em_score"], rtol=1e-5)
    elp = net._estimate_log_prob(x, mu, sg)
    np.testing.assert_allclose(elp.cpu().numpy(), g["em_est_log_prob"], rtol=1e-5)


def test_em_gradient_ka6(golden):
    """The fused M-step gradient equals the reference's autograd gradient (KA6)."""
    g = golden
    from mgproto_b200 import ops
    C, K, D, cap = (int(g[k]) for k in "C K D cap".split())
    c = int(g["em_class"])
    x = g["em_x"]
    if x.shape[0] != cap:
        pytest.skip("fixture class not full")
    dev = _dev()
    bank = torch.zeros(C, cap, D, device=dev)
    bank[c] = _t(x)
    mu = torch.zeros(C, K, D, device=dev)
    mu[c] = _t(g["em_mu"][0])
    sg = torch.ones(C, K, D, device=dev)
    sg[c] = _t(g["em_sigma"][0])
    wt = torch.zeros(C, C * K, device=dev)
    wt[c, c * K:(c + 1) * K] = _t(g["em_pi"].reshape(K))
    order = torch.full((C,), -1, dtype=torch.int32, device=dev)
    order[c] = 0
    sched = torch.tensor([1, 0], dtype=torch.int32, device=dev)
    for n_split in (1, 3):
        stats = torch.empty(C, n_split, ops.em_stat_stride(K, D), device=dev)
        ops.em_stats(bank, order, mu, sg, wt, float(g["alpha"]), stats, n_split)
        grad = torch.zeros(C, K, D, device=dev)
        w2 = wt.clone()
        ops.em_update(stats, n_split, cap, order, sched, mu, sg, w2, None, None, 0, 3, 1, 0.0, 0.9, 0.999, 1e-8,
                      float(g["tau"]), grad_out=grad)
        ref = g["em_div_grad"]
        np.testing.assert_allclose(grad[c].cpu().numpy(), ref, rtol=1e-3, atol=1e-5 * np.abs(ref).max() + 1e-9)
        pi_new = (w2[c, c * K:(c + 1) * K].cpu().numpy() - float(g["tau"]) * g["em_pi"].reshape(K)) / (1 - float(g["tau"]))
        np.testing.assert_allclose(pi_new, g["em_div_pi"].reshape(K), rtol=2e-3)


def test_bank_ring_wraps_like_reference_fifo():
    """FIFO semantics across many pushes (all four branches of utils/memory.py:56-67) against the oracle."""
    from mgproto_b200 import ops
    from oracle import mgproto_oracle as O
    rng = np.random.default_rng(0)
    C, K, D, cap, HW, T, B = 3, 4, 8, 10, 9, 2, 5
    dev = _dev()
    bank = torch.zeros(C, cap, D, device=dev)
    mem_len = torch.zeros(C, dtype=torch.int64, device=dev)
    head = torch.zeros(C, dtype=torch.int32, device=dev)
    upd = torch.zeros(C, dtype=torch.uint8, device=dev)
    ob = O.MemoryBankOracle(C, D, cap)
    for it in range(12):
        xhat = rng.standard_normal((B * HW, D)).astype(np.float32)
        idx = rng.integers(0, HW, size=(B, C * K, T)).astype(np.int32)
        gt = rng.integers(0, C, size=(B,)).astype(np.int64)
        gtt = _t(gt, torch.int64)
        top1, rows = ops.mined_gather(_t(xhat), _t(idx, torch.int32), gtt, HW, C, K)
        ops.bank_enqueue(bank, mem_len, head, upd, rows, top1, gtt)
        for c, rows in O.enqueue_rows(xhat, idx, gt, C, K, HW):
            ob.push(c, rows)
        lin = ops.bank_linearize(bank, mem_len, head).cpu().numpy()
        np.testing.assert_array_equal(mem_len.cpu().numpy(), ob.mem_len)
        for c in range(C):
            n = int(ob.mem_len[c])
            np.testing.assert_array_equal(lin[c, :n], ob.data[c, :n])


def test_state_dict_roundtrip(golden):
    g = golden
    net = _model_from(g, "fp32")
    with torch.no_grad():
        for it in range(2):
            net.head(_t(g["it%d_x_add" % it]), _t(g["it%d_gt" % it], torch.int64))
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    assert "queue.cls0" in sd and "queue.mem_len" in sd and "prototype_means" in sd and "last_layer.weight" in sd
    net2 = _model_from(g, "fp32")
    net2.load_state_dict(sd)
    sd2 = net2.state_dict()
    for k in sd:
        assert torch.equal(sd[k].cpu(), sd2[k].cpu()), k


# ---------------------------------------------------------------------------------------------
# tensor-core log-likelihood kernel (tcgen05, fp16 hi/lo x3) against the exact fp32 SIMT kernel
# and a float64 restatement, at shapes with ragged tiles and at the BASELINE size
@pytest.mark.parametrize("sigma_mode", ["iso", "diag"])
@pytest.mark.parametrize("shape", [(3, 49, 130, 64), (5, 196, 2000, 128), (2, 200, 257, 128)])
def test_logprob_tc_vs_fp32(shape, sigma_mode):
    from mgproto_b200 import ops, _lib
    if not _lib.load().mgp_has_tensor_core_path():
        pytest.skip("library built without the tcgen05 path")
    B, HW, P, D = shape
    g = torch.Generator().manual_seed(5)
    x = F.normalize(torch.randn(B * HW, D, generator=g), dim=1).to(_dev())
    mu = F.normalize(torch.rand(P, D, generator=g), dim=1).to(_dev())
    if sigma_mode == "iso":
        sg = (0.25 + 0.5 * torch.rand(P, 1, generator=g)).expand(P, D).contiguous().to(_dev())
    else:
        sg = (0.2 + 0.6 * torch.rand(P, D, generator=g)).to(_dev())
    ref64 = (-0.5 * D * np.log(2 * np.pi) - sg.double().log().sum(1)[None, :]
             - 0.5 * (((x.double()[:, None, :] - mu.double()[None]) / sg.double()[None]) ** 2).sum(-1))
    for layout in (0, 1, 2):
        a = ops.logprob(x, mu, sg, layout, B=B, HW=HW, math="tc")
        b = ops.logprob(x, mu, sg, layout, B=B, HW=HW, math="fp32")
        r = ref64 if layout == 0 else ref64.view(B, HW, P).permute(0, 2, 1)
        if layout == 2:
            r = -r.exp()
        torch.testing.assert_close(a.double(), r, rtol=2e-5, atol=2e-5 if layout != 2 else 1e-12)
        torch.testing.assert_close(a, b, rtol=2e-5, atol=2e-5 if layout != 2 else 1e-12)


@pytest.mark.parametrize("shape", [(3, 49, 130, 64), (5, 196, 2000, 128), (2, 200, 257, 128), (1, 7, 5, 128), (9, 196, 1000, 64),
                                   (2, 196, 300, 256), (7, 49, 2000, 256), (1, 7, 5, 256)])
def test_logprob_tmem_resident_kernel_vs_fp64(shape):
    """compute_log_prob's [N,P] kernel with the patch tile resident in tensor memory and the fp16 hi/lo split fused
    (csrc/logprob_tcz.cu; taken by math='auto' when sigma is isotropic, D <= 256 -- D = 256 keeps ONE operand buffer in
    tensor memory and lands / converts the patch tile in two halves): ragged tiles on both sides, against
    float64 and against the kernel that splits x in a pre-pass (csrc/logprob_tc.cu)."""
    from mgproto_b200 import ops, _lib
    lib = _lib.load()
    if not lib.mgp_has_tensor_core_path():
        pytest.skip("library built without the tcgen05 path")
    B, HW, P, D = shape
    g = torch.Generator().manual_seed(11)
    x = F.normalize(torch.randn(B * HW, D, generator=g), dim=1).to(_dev())
    mu = F.normalize(torch.rand(P, D, generator=g), dim=1).to(_dev())
    sg = (0.25 + 0.5 * torch.rand(P, 1, generator=g)).expand(P, D).contiguous().to(_dev())
    ref64 = (-0.5 * D * np.log(2 * np.pi) - sg.double().log().sum(1)[None, :]
             - 0.5 * (((x.double()[:, None, :] - mu.double()[None]) / sg.double()[None]) ** 2).sum(-1))
    a = ops.logprob(x, mu, sg, 0, math="auto")
    prev = lib.mgp_set_option(b"tc_z", 0)
    try:
        b = ops.logprob(x, mu, sg, 0, math="auto")
    finally:
        lib.mgp_set_option(b"tc_z", prev)
    torch.testing.assert_close(a.double(), ref64, rtol=2e-5, atol=2e-5)
    torch.testing.assert_close(a, b, rtol=2e-5, atol=2e-5)


def test_logprob_prototype_operands_are_reused_only_when_passed_explicitly():
    """ops.logprob ([N,P], isotropic sigma) skips the prototype-side pre-pass of the TMEM-resident kernel when the
    caller hands back the workspace of an earlier call (math='tc_iso_reuse'), and rebuilds the operands on every auto
    call -- a write through `.data` bumps no version counter, so cached operands could be stale without anything
    noticing."""
    from mgproto_b200 import ops, _lib
    if not _lib.load().mgp_has_tensor_core_path():
        pytest.skip("library built without the tcgen05 path")
    B, HW, P, D = 4, 49, 300, 128
    g = torch.Generator().manual_seed(5)
    x = F.normalize(torch.randn(B * HW, D, generator=g), dim=1).to(_dev())
    mu = F.normalize(torch.rand(P, D, generator=g), dim=1).to(_dev())
    sg = torch.full((P, D), 0.4, device=_dev())

    def ref(m):
        return (-0.5 * D * np.log(2 * np.pi) - sg.double().log().sum(1)[None, :]
                - 0.5 * (((x.double()[:, None, :] - m.double()[None]) / sg.double()[None]) ** 2).sum(-1))
    n0 = ops.launch_count()
    a, ws = ops.logprob(x, mu, sg, 0, math="tc_iso", return_ws=True)
    n1 = ops.launch_count()
    b = ops.logprob(x, mu, sg, 0, math="tc_iso_reuse", ws=ws)          # the pre-pass is skipped
    n2 = ops.launch_count()
    assert (n2 - n1) < (n1 - n0)
    assert torch.equal(a, b)
    torch.testing.assert_close(a.double(), ref(mu), rtol=2e-5, atol=2e-5)
    for _ in range(2):                                                 # auto: the same kernel, the pre-pass every time
        n3 = ops.launch_count()
        c = ops.logprob(x, mu, sg, 0, math="auto")
        assert ops.launch_count() - n3 == n1 - n0
        assert torch.equal(c, a)
    mu.data.mul_(0.5)                                                  # no version bump
    d = ops.logprob(x, mu, sg, 0, math="auto")
    torch.testing.assert_close(d.double(), ref(mu), rtol=2e-5, atol=2e-5)
    mu.mul_(0.5)                                                       # in place: new version
    e = ops.logprob(x, mu, sg, 0, math="auto")
    torch.testing.assert_close(e.double(), ref(mu), rtol=2e-5, atol=2e-5)
    v = mu._version
    torch.autograd.graph.increment_version(mu)                         # what MGProto.update_GMM does after its kernels
    assert mu._version == v + 1


def test_logprob_tc_baseline_size_properties():
    """cfg2 size (B=256, P=2000, D=128): KA1 identity on a strided sample + exact agreement of the
    three output layouts with each other (size-independent properties; no CPU oracle at this size)."""
    from mgproto_b200 import ops, _lib
    if not _lib.load().mgp_has_tensor_core_path():
        pytest.skip("library built without the tcgen05 path")
    B, HW, P, D = 256, 196, 2000, 128
    g = torch.Generator().manual_seed(1)
    x = F.normalize(torch.randn(B * HW, D, generator=g), dim=1).to(_dev())
    mu = F.normalize(torch.rand(P, D, generator=g), dim=1).to(_dev())
    sg = torch.full((P, D), 1 / np.sqrt(2 * np.pi), device=_dev())
    lp = ops.logprob(x, mu, sg, 0, math="tc")
    rows = torch.arange(0, B * HW, 97, device=_dev())
    ref = -np.pi * ((x[rows].double()[:, None, :] - mu.double()[None]) ** 2).sum(-1)       # KA1
    torch.testing.assert_close(lp[rows].double(), ref, rtol=1e-5, atol=2e-5)
    lpz = ops.logprob(x, mu, sg, 0, math="auto")                                           # TMEM-resident kernel
    torch.testing.assert_close(lpz[rows].double(), ref, rtol=1e-5, atol=2e-5)
    torch.testing.assert_close(lpz, lp, rtol=2e-5, atol=2e-5)
    lp_b = ops.logprob(x, mu, sg, 1, B=B, HW=HW, math="tc")
    assert torch.equal(lp_b, lp.view(B, HW, P).permute(0, 2, 1).contiguous())
    assert torch.isfinite(lp).all()


def test_mine_cross_entropy_matches_torch():
    """Fused loss helper == CE(level 0) + 0.2 * mean CE(levels 1..T-1) of train_and_test.py:37-41,:55."""
    from mgproto_b200 import ops
    g = torch.Generator().manual_seed(0)
    B, C, T = 37, 23, 7
    out = (torch.randn(B, C, T, generator=g) * 3 - 5).to(_dev()).requires_grad_(True)
    gt = torch.randint(0, C, (B,), generator=g).to(_dev())
    ref = _loss(out, gt)
    gref, = torch.autograd.grad(ref, out)
    out2 = out.detach().clone().requires_grad_(True)
    got = ops.mine_cross_entropy(out2, gt, 0.2)
    (got * 1.7).backward()
    torch.testing.assert_close(got, ref.detach(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(out2.grad, 1.7 * gref, rtol=1e-4, atol=1e-7)


# ---------------------------------------------------------------------------------------------
# BASELINE.json configs[3] shapes (prototype sweep K x D) and configs[4] (OoD scoring) as parity cases
@pytest.mark.parametrize("K,D", [(5, 64), (20, 128), (40, 64), (10, 256), (5, 512)])
def test_head_sweep_shapes_vs_fp64(K, D):
    """forward logits / top-T values for the sweep shapes against a float64 torch restatement of
    model.py:208-254 (tensor-core path where the shape qualifies, exact SIMT path otherwise)."""
    from mgproto_b200 import ops
    C, B, H, W, T = 8, 3, 14, 14, 20
    g = torch.Generator().manual_seed(K * 1000 + D)
    x = torch.randn(B, D, H, W, generator=g).to(_dev())
    mu = F.normalize(torch.rand(C, K, D, generator=g), dim=2).to(_dev())
    sg = torch.full((C, K, D), 1 / np.sqrt(2 * np.pi), device=_dev())
    pi = torch.softmax(torch.randn(C, K, generator=g), dim=1)
    wt = torch.zeros(C, C * K)
    for c in range(C):
        wt[c, c * K:(c + 1) * K] = pi[c]
    wt = wt.to(_dev())
    gt = torch.randint(0, C, (B,), generator=g).to(_dev())
    lg, _, idx = ops.head_forward(x, mu, sg, wt, gt, T, "auto")
    xd = F.normalize(x.double(), dim=1).permute(0, 2, 3, 1).reshape(B, H * W, D)
    lp = (-0.5 * D * np.log(2 * np.pi) - sg.double().log().sum(-1).view(1, 1, -1)
          - 0.5 * (((xd[:, :, None, :] - mu.double().view(1, 1, C * K, D)) / sg.double().view(1, 1, C * K, D)) ** 2).sum(-1))
    v, _ = torch.topk(lp.exp().permute(0, 2, 1), T, dim=2)                     # [B,P,T]
    wrong = (torch.arange(C * K, device=_dev()) // K)[None, :] != gt[:, None]
    v = torch.where(wrong[:, :, None], v[:, :, :1].expand(-1, -1, T), v)
    ref = torch.log(torch.einsum("bpt,cp->bct", v, wt.double()))
    torch.testing.assert_close(lg.double(), ref, rtol=RTOL, atol=1e-6)


def test_ood_score_auroc_matches_oracle():
    """configs[4]: OoD score sum_c exp(logit_c0) (ref train_and_test.py:184-199) on synthetic in-dist / OoD
    features: scores within 1e-4 and AUROC equal to the oracle's."""
    from sklearn.metrics import roc_auc_score
    from mgproto_b200 import ops
    from oracle import mgproto_oracle as O
    C, K, D, H, W, n = 6, 4, 64, 7, 7, 24
    g = torch.Generator().manual_seed(9)
    mu = F.normalize(torch.rand(C, K, D, generator=g), dim=2)
    sg = torch.full((C, K, D), 1 / np.sqrt(2 * np.pi))
    wt = torch.zeros(C, C * K)
    for c in range(C):
        wt[c, c * K:(c + 1) * K] = 1.0 / K
    pick = torch.randint(0, C * K, (n, H * W), generator=g)
    x_in = (mu.view(C * K, D)[pick] + 0.1 * torch.randn(n, H * W, D, generator=g)).permute(0, 2, 1).reshape(n, D, H, W)
    x_out = torch.randn(n, D, H, W, generator=g)
    x = torch.cat([x_in, x_out]).contiguous()
    lg, _, _ = ops.head_forward(x.to(_dev()), mu.to(_dev()), sg.to(_dev()), wt.to(_dev()), None, 1, "auto")
    score = lg[:, :, 0].exp().sum(1).cpu().numpy()
    fw = O.head_forward(x.numpy().astype(np.float64), mu.numpy().astype(np.float64), sg.numpy().astype(np.float64),
                        wt.numpy().astype(np.float64), None, 1)
    ref = np.exp(fw["logits"][:, :, 0]).sum(1)
    np.testing.assert_allclose(score, ref, rtol=RTOL)
    y = np.r_[np.ones(n), np.zeros(n)]
    assert abs(roc_auc_score(y, score) - roc_auc_score(y, ref)) < 1e-9
    assert roc_auc_score(y, ref) > 0.9


def test_logprob_tc_bphw_tma_path():
    """[B,P,HW] written by 3-D TMA stores (taken when 32 | HW): against the exact fp32 kernel."""
    from mgproto_b200 import ops, _lib
    if not _lib.load().mgp_has_tensor_core_path():
        pytest.skip("library built without the tcgen05 path")
    B, HW, P, D = 5, 64, 300, 128
    g = torch.Generator().manual_seed(3)
    x = F.normalize(torch.randn(B * HW, D, generator=g), dim=1).to(_dev())
    mu = F.normalize(torch.rand(P, D, generator=g), dim=1).to(_dev())
    sg = torch.full((P, D), 0.4, device=_dev())
    for layout in (1, 2):
        a = ops.logprob(x, mu, sg, layout, B=B, HW=HW, math="tc")
        b = ops.logprob(x, mu, sg, layout, B=B, HW=HW, math="fp32")
        torch.testing.assert_close(a, b, rtol=2e-5, atol=2e-5 if layout == 1 else 1e-12)


def test_push_search_from_the_top1_epilogue_vs_materialised_map():
    """f1 without the [B,P,HW] map: push_search through mgp_push_argmin_top1 (packed max / arg-max of the tensor-core
    epilogue) against mgp_push_argmin on the materialised fp32 map and against float64."""
    import mgproto_b200 as M
    from mgproto_b200 import ops, _lib
    if not _lib.load().mgp_has_tensor_core_path():
        pytest.skip("library built without the tcgen05 path")
    C, K, D, H, W, B = 12, 10, 128, 14, 14, 6
    torch.manual_seed(9)
    net = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 16, 1)), img_size=H, prototype_shape=(C * K, D, 1, 1),
                    proto_layer_rf_info=None, num_classes=C, add_on_layers_type="regular", sz_embedding=8,
                    mem_capacity=8, mine_K=4).to(_dev())
    g = torch.Generator().manual_seed(10)
    x_add = torch.randn(B, D, H, W, generator=g).to(_dev())
    labs = torch.randint(0, C, (B,), generator=g).to(_dev())
    labs[0] = -1                                                   # no valid class: arg -1, val 0 (as mgp_push_argmin)
    n0 = ops.launch_count()
    arg, val, xhat = net.push_search(x_add, labs)
    assert ops.launch_count() - n0 <= 4                            # normalise+stage, prototype pre-pass + GEMM, gather
    lp = ops.logprob(xhat, net.prototype_means.detach().reshape(C * K, D), net.prototype_covs.detach().reshape(C * K, D),
                     1, B=B, HW=H * W, math="fp32")
    arg0, val0 = ops.push_argmin(lp, labs, C, K)
    torch.testing.assert_close(val, val0, rtol=RTOL, atol=1e-30)
    lp64 = lp.double().cpu().numpy()
    a, a0 = arg.cpu().numpy(), arg0.cpu().numpy()
    assert (a[0] == -1).all() and float(val[0].abs().max()) == 0.0
    for b in range(1, B):
        c = int(labs[b])
        for k in range(K):
            row = lp64[b, c * K + k]
            assert a[b, k] == a0[b, k] or row[a[b, k]] >= row.max() - 1e-4 * abs(row.max())


def test_push_prototypes_matches_oracle():
    """Prototype projection (push.py:82-200, numeric half) on a synthetic push set: chosen (image, patch) per
    prototype and the copied feature vectors against the oracle run on the distance maps of push_forward."""
    import mgproto_b200 as M
    from oracle import mgproto_oracle as O
    C, K, D, H, W, n = 5, 3, 64, 6, 6, 23
    torch.manual_seed(4)
    net = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 16, 1)), img_size=H, prototype_shape=(C * K, D, 1, 1),
                    proto_layer_rf_info=None, num_classes=C, add_on_layers_type="regular", sz_embedding=8,
                    mem_capacity=8, mine_K=4).to(_dev())
    g = torch.Generator().manual_seed(5)
    imgs = torch.randn(n, 3, H, W, generator=g)
    labs = torch.randint(0, C, (n,), generator=g)
    labs[:C] = torch.arange(C)
    loader = [(imgs[i:i + 6], labs[i:i + 6]) for i in range(0, n, 6)]
    with torch.no_grad():
        feat, dist = net.push_forward(imgs.to(_dev()))
    dist = dist.cpu().numpy()
    feat = feat.cpu().numpy()
    oi, ov = O.push_argmin(dist, labs.numpy(), K)
    want = O.push_assign(ov, labs.numpy(), C, K)
    mu0 = net.prototype_means.detach().clone()
    res = M.push_prototypes(loader, net, log=lambda *_: None)
    np.testing.assert_array_equal(res["image"], want)
    for j in range(C * K):
        c, k = divmod(j, K)
        i = want[j]
        if i < 0:
            assert torch.equal(net.prototype_means[c, k], mu0[c, k])
            continue
        assert res["patch"][j] == oi[i, k]
        hh, ww = divmod(int(oi[i, k]), W)
        np.testing.assert_allclose(net.prototype_means[c, k].detach().cpu().numpy(), feat[i, :, hh, ww], rtol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W,C,K,D,T,aniso", [(5, 14, 14, 7, 10, 128, 20, False), (3, 7, 7, 5, 4, 64, 6, False),
                                                 (4, 4, 4, 3, 5, 64, 4, False), (3, 14, 14, 4, 10, 128, 20, True),
                                                 (2, 16, 16, 3, 3, 128, 32, False)])
def test_fused_top1_path_vs_materialised(B, H, W, C, K, D, T, aniso):
    """Labelled head: the tensor-core epilogue's packed max/arg-max (MGP_OUT_TOP1_BP) + mgp_head_select_top1 against
    the path that materialises log p [B,P,HW] and mines it (mgp_head_select), and against fp64."""
    from mgproto_b200 import ops
    g = torch.Generator().manual_seed(B * 100 + D + T)
    HW, P = H * W, C * K
    x = torch.randn(B, D, H, W, generator=g).to(_dev())
    mu = F.normalize(torch.rand(C, K, D, generator=g), dim=2).to(_dev())
    sg = torch.full((C, K, D), 1 / np.sqrt(2 * np.pi))
    if aniso:
        sg = sg * (0.8 + 0.4 * torch.rand(C, K, D, generator=g))
    sg = sg.to(_dev())
    pi = torch.softmax(torch.randn(C, K, generator=g), dim=1)
    wt = torch.zeros(C, P)
    for c in range(C):
        wt[c, c * K:(c + 1) * K] = pi[c]
    wt = wt.to(_dev())
    gt = torch.randint(0, C, (B,), generator=g).to(_dev())
    gt[0] = -1 if B > 2 else gt[0]                      # an image without a valid class: every class is "wrong"
    xhat, _, _ = ops.normalize_fwd(x)
    mu2, sg2 = mu.reshape(P, D).contiguous(), sg.reshape(P, D).contiguous()
    best = ops.logprob_top1(xhat, mu2, sg2, B, HW, "tc")
    assert best is not None
    xd = xhat.double().reshape(B, HW, D)
    lp64 = (-0.5 * D * np.log(2 * np.pi) - sg2.double().log().sum(-1).view(1, 1, P)
            - 0.5 * (((xd[:, :, None, :] - mu2.double().view(1, 1, P, D)) / sg2.double().view(1, 1, P, D)) ** 2).sum(-1))
    lp64 = lp64.permute(0, 2, 1)                                               # [B,P,HW]
    bv = best.cpu().numpy().astype(np.uint64)
    key = (bv >> np.uint64(32)).astype(np.uint32)
    u = np.where(key & np.uint32(0x80000000), key & np.uint32(0x7fffffff), ~key).astype(np.uint32)
    val = u.view(np.float32)
    arg = (np.uint32(0xffffffff) - (bv & np.uint64(0xffffffff)).astype(np.uint32)).astype(np.int64)
    m64, a64 = lp64.max(dim=2)
    np.testing.assert_allclose(val, m64.cpu().numpy(), rtol=RTOL, atol=1e-4)
    srt = torch.sort(lp64, dim=2, descending=True).values
    sep = ((srt[:, :, 0] - srt[:, :, 1]) > 1e-3).cpu().numpy()
    assert (arg[sep] == a64.cpu().numpy()[sep]).all()
    # the same through the fused normalise + operand staging pass (what HeadFunction runs when 32 <= HW <= 256)
    stage = ops._stage_for_top1(B, HW, P, D, sg2, "tc")
    if stage is not None:
        assert stage[1] == aniso
        xh2, inv2, _, ws = ops.normalize_fwd(x, stage=stage)
        assert torch.equal(xh2, xhat)
        best2 = ops.logprob_top1(xh2, mu2, sg2, B, HW, "tc", ws=ws, staged=stage)
        b2 = best2.cpu().numpy().astype(np.uint64)
        k2 = (b2 >> np.uint64(32)).astype(np.uint32)
        u2 = np.where(k2 & np.uint32(0x80000000), k2 & np.uint32(0x7fffffff), ~k2).astype(np.uint32)
        np.testing.assert_allclose(u2.view(np.float32), val, rtol=1e-6, atol=1e-6)    # (|xhat|^2 is summed in another order)
        arg2 = (np.uint32(0xffffffff) - (b2 & np.uint64(0xffffffff)).astype(np.uint32)).astype(np.int64)
        assert (arg2[sep] == a64.cpu().numpy()[sep]).all()
    # whole head, both routes
    lg1, v1, i1 = ops.head_select_top1(best, xhat, mu2, sg2, wt, gt, T, C, K, HW)
    lp = ops.logprob(xhat, mu2, sg2, 1, B=B, HW=HW, math="tc")
    lg0, v0, i0 = ops.head_select(lp, wt, gt, T, C, K)
    torch.testing.assert_close(lg1, lg0, rtol=RTOL, atol=1e-6)
    torch.testing.assert_close(v1[:, :, 0], v0[:, :, 0], rtol=RTOL, atol=1e-30)
    for b in range(B):
        c = int(gt[b])
        if c < 0:
            continue
        rows = slice(c * K, (c + 1) * K)
        torch.testing.assert_close(v1[b, rows], v0[b, rows], rtol=RTOL, atol=1e-30)
        s = torch.sort(lp64[b, rows], dim=1, descending=True).values[:, :T + 1]
        okm = ((s[:, :-1] - s[:, 1:]) > 1e-3).cpu().numpy()
        ref_i = torch.topk(lp64[b, rows], T, dim=1).indices.cpu().numpy()
        assert (i1[b, rows].cpu().numpy()[okm] == ref_i[okm]).all()
    # through autograd (the route HeadFunction takes with labels) against the materialised route's gradient
    xa = x.clone().requires_grad_(True)
    out, _, _ = ops.head_forward(xa, mu, sg, wt, gt, T, "tc")
    gl = torch.randn(out.shape, generator=torch.Generator().manual_seed(3)).to(_dev())
    out.backward(gl)
    torch.testing.assert_close(out.detach(), lg0, rtol=RTOL, atol=1e-6)
    assert torch.isfinite(xa.grad).all()


@pytest.mark.gpu
def test_host_pipeline_roundtrip():
    """pipeline.HostFeeder / HostSink: staged copies arrive intact and in order while work is queued behind them."""
    from mgproto_b200.pipeline import HostFeeder, HostSink
    dev = _dev()
    hosts = [torch.full((4, 8), float(i)).pin_memory() for i in range(7)]
    feeder = HostFeeder((4, 8), dev, depth=2)
    sink = HostSink((4, 8), depth=2, device=dev)
    got = []
    feeder.stage(hosts[0])
    for i in range(7):
        if i + 1 < 7:
            feeder.stage(hosts[i + 1])
        x = feeder.acquire()
        y = x * 2 + 1
        h = sink.put(y)
        feeder.release(x)
        sink.wait()
        got.append(h.clone())
    for i, h in enumerate(got):
        assert torch.equal(h, torch.full((4, 8), 2.0 * i + 1))


@pytest.mark.gpu
@pytest.mark.parametrize("math", ["auto", "fp32"])
def test_head_level0_matches_unlabelled_head(golden, math):
    """f2: the test / OoD loop's output[:, :, 0] (ref train_and_test.py:182-199) from the max/arg-max path equals
    level 0 of the full unlabelled head."""
    from mgproto_b200 import ops
    g = golden
    net = _model_from(g, math)
    net.prototype_means.data.copy_(_t(g["it0_mu"]))
    x = _t(g["it0_x_add"])
    with torch.no_grad():
        full, _, _ = ops.head_forward(x, net.prototype_means, net.prototype_covs, net.last_layer.weight, None,
                                      net.mine_T, math)
        l0 = net.head_level0(x)
    np.testing.assert_allclose(l0.cpu().numpy(), full[:, :, 0].cpu().numpy(), rtol=RTOL, atol=1e-6)
    np.testing.assert_allclose(l0.cpu().numpy(), g["it0_logits_nogt"][:, :, 0], rtol=RTOL, atol=1e-6)


@pytest.mark.gpu
def test_reference_training_body_with_real_backbone():
    """construct_MGProto('resnet18') driven by the body of the reference's training loop (train_and_test.py:26-63):
    forward(image, target) through a real backbone, the CE + mining losses, backward into the backbone, the joint
    optimiser step, then update_GMM once the banks are full -- two iterations.  The logits are checked against the
    float64 oracle on the add-on features the backbone produced, the enqueue against the oracle's, and the gradient
    must reach the backbone."""
    import mgproto_b200 as M
    from oracle import mgproto_oracle as O
    torch.manual_seed(0)
    C, K, D, T, cap, B = 6, 4, 64, 4, 8, 12
    net = M.construct_MGProto("resnet18", pretrained=False, img_size=64, prototype_shape=(C * K, D, 1, 1), num_classes=C,
                              add_on_layers_type="regular", sz_embedding=16, mem_capacity=cap, mine_K=T).to(_dev())
    assert net.proto_layer_rf_info is not None and len(net.proto_layer_rf_info) == 4
    net.prototype_optimizer = torch.optim.Adam([{"params": net.prototype_means, "lr": 3e-3}])
    joint = torch.optim.Adam([{"params": net.features.parameters(), "lr": 1e-4},
                              {"params": net.add_on_layers.parameters(), "lr": 3e-3}])
    model = torch.nn.DataParallel(net, device_ids=[0])                      # the reference drives `.module` (train_and_test.py:61)
    net.train()
    g = torch.Generator().manual_seed(1)
    bank = O.MemoryBankOracle(C, D, cap)
    for it in range(2):
        image = torch.randn(B, 3, 64, 64, generator=g).to(_dev())
        target = torch.randint(0, C, (B,), generator=g).to(_dev())
        output, x_aux = model(image, target)
        assert output.shape == (B, C, T) and x_aux.shape == (B, 16)
        mine_loss = sum(F.cross_entropy(output[:, :, k], target) for k in range(1, T)) / (T - 1)
        loss = F.cross_entropy(output[:, :, 0], target) + 0.2 * mine_loss
        joint.zero_grad()
        loss.backward()
        gn = sum(float(p.grad.abs().sum()) for p in net.features.parameters() if p.grad is not None)
        assert np.isfinite(gn) and gn > 0
        # oracle on the features the (unchanged-so-far) backbone produced
        with torch.no_grad():
            x_add, _ = net.conv_features(image)
        fw = O.head_forward(x_add.double().cpu().numpy(), net.prototype_means.detach().double().cpu().numpy(),
                            net.prototype_covs.double().cpu().numpy(), net.last_layer.weight.double().cpu().numpy(),
                            target.cpu().numpy(), T)
        np.testing.assert_allclose(output.detach().cpu().numpy(), fw["logits"], rtol=RTOL, atol=1e-5)
        for c, rows in O.enqueue_rows(fw["xhat"].astype(np.float32), fw["idx"], target.cpu().numpy(), C, K, x_add.shape[2] * x_add.shape[3]):
            bank.push(c, rows)
        np.testing.assert_array_equal(net.queue.mem_len.cpu().numpy(), bank.mem_len)
        joint.step()
        # train_and_test.py:61-63
        if model.module.queue.mem_len.sum() > 0 and model.module.iteration_counter % model.module.update_interval == 0:
            mu0 = net.prototype_means.detach().clone()
            model.module.update_GMM()
            full = (net.queue.mem_len == cap).cpu().numpy()
            moved = (net.prototype_means.detach() - mu0).abs().amax(dim=(1, 2)).cpu().numpy() > 0
            assert (moved[full] | ~full[full]).all() or not full.any()
        assert int(net.memory_updated_cls.sum()) == 0
    net.sync_optimizer_state()
    assert torch.isfinite(net.prototype_means).all() and torch.isfinite(net.last_layer.weight).all()


@pytest.mark.gpu
def test_boundary_methods_m_step_diversified_and_topT(golden):
    """The reference's private methods as a caller would drive them: _e_step -> _m_step_diversified on a bank class
    (gradient = the reference's autograd gradient, then the optimiser step on the whole mean tensor) and
    global_max_pooling_gmm_topT on probabilities (values / indices / gathered features)."""
    g = golden
    if "em_div_grad" not in g or g["em_x"].shape[0] < 2:
        pytest.skip("fixture without a full EM class")
    net = _model_from(g, "fp32")
    C, K, D = (int(g[k]) for k in "C K D".split())
    c = int(g["em_class"])
    net.prototype_means.data[c].copy_(_t(g["em_mu"][0]))
    net.prototype_covs.data[c].copy_(_t(g["em_sigma"][0]))
    x = _t(g["em_x"])
    pi_old = _t(g["em_pi"])
    mu_view = net.prototype_means[c].unsqueeze(0)
    ll, log_resp = net._e_step(x, mu_view.detach(), net.prototype_covs[c].unsqueeze(0), pi_old)
    before = net.prototype_means.detach().clone()
    pi_new, mu_ret, var_ret = net._m_step_diversified(x, log_resp, mu_view, net.prototype_covs[c].unsqueeze(0), pi_old)
    np.testing.assert_allclose(pi_new.cpu().numpy().reshape(-1), g["em_div_pi"].reshape(-1), rtol=1e-5)
    assert mu_ret is mu_view
    # the optimiser took one Adam step with the reference's gradient on class c and zero elsewhere
    grad = np.zeros((C, K, D), np.float64)
    grad[c] = g["em_div_grad"]
    from oracle import mgproto_oracle as O
    adam = O.AdamOracle((C, K, D), lr=float(g["lr"]))
    want = adam.step(before.double().cpu().numpy(), grad)
    np.testing.assert_allclose(net.prototype_means.detach().cpu().numpy(), want, rtol=1e-4, atol=1e-6)
    # global_max_pooling_gmm_topT
    B, _, H, W = g["it0_x_add"].shape
    T = int(g["T"])
    from mgproto_b200 import ops
    xhat, _, nchw = ops.normalize_fwd(_t(g["it0_x_add"]), want_nchw=True)
    prob = _t(g["it0_logp"]).exp().view(B, H, W, C, K).permute(0, 3, 4, 1, 2).contiguous()
    vals, feats, idx = net.global_max_pooling_gmm_topT(prob, nchw, mine_T=T)
    np.testing.assert_allclose(vals.cpu().numpy(), g["it0_topk_vals"], rtol=1e-6)
    assert idx.dtype == torch.int64 and tuple(feats.shape) == (B, C, K, D, T)
    sep = _separated(g["it0_topk_vals"])
    assert (idx.view(B, C * K, T).cpu().numpy()[sep] == g["it0_topk_idx"][sep]).all()
    f = feats.view(B, C * K, D, T).cpu().numpy()
    xn = nchw.view(B, D, H * W).cpu().numpy()
    ii = idx.view(B, C * K, T).cpu().numpy()
    for b in range(B):
        for p in range(0, C * K, 3):
            for t in range(0, T, 2):
                np.testing.assert_array_equal(f[b, p, :, t], xn[b, :, ii[b, p, t]])


@pytest.mark.gpu
def test_ood_scorer_device_side_vs_oracle_and_sklearn():
    """configs[4] path: mgproto_b200.ood.OoDScorer (head_level0 + mgp_ood_score per batch, threshold / FPR95 / AUROC on
    the device) against the numpy oracle's scores, numpy.percentile and sklearn's AUROC on 384 + 384 synthetic images."""
    from sklearn.metrics import roc_auc_score
    import mgproto_b200 as M
    from mgproto_b200.ood import OoDScorer
    from oracle import mgproto_oracle as O
    C, K, D, H, W, n, bs = 12, 5, 64, 7, 7, 384, 128
    torch.manual_seed(3)
    net = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 16, 1)), img_size=14, prototype_shape=(C * K, D, 1, 1),
                    proto_layer_rf_info=None, num_classes=C, add_on_layers_type="regular", sz_embedding=8,
                    mem_capacity=8, mine_K=4).to(_dev())
    g = torch.Generator().manual_seed(9)
    mu = net.prototype_means.detach().cpu()
    pick = torch.randint(0, C * K, (n, H * W), generator=g)
    x_in = (mu.view(C * K, D)[pick] + 0.1 * torch.randn(n, H * W, D, generator=g)).permute(0, 2, 1).reshape(n, D, H, W)
    lab = (pick[:, 0] // K)
    x_out = torch.randn(n, D, H, W, generator=g)
    sc = OoDScorer(net)
    for i in range(0, n, bs):
        sc.add_in_distribution(x_in[i:i + bs].contiguous().to(_dev()), lab[i:i + bs])
        sc.add_out_of_distribution(x_out[i:i + bs].contiguous().to(_dev()))
    res = sc.results()
    f64 = lambda t: t.numpy().astype(np.float64)                                  # noqa: E731
    wt = net.last_layer.weight.detach().cpu()
    sg = net.prototype_covs.detach().cpu()
    ref_in = np.exp(O.head_forward(f64(x_in), f64(mu), f64(sg), f64(wt), None, 1)["logits"][:, :, 0])
    ref_out = np.exp(O.head_forward(f64(x_out), f64(mu), f64(sg), f64(wt), None, 1)["logits"][:, :, 0])
    np.testing.assert_allclose(torch.cat(sc.id_sum).cpu().numpy(), ref_in.sum(1), rtol=RTOL)
    np.testing.assert_allclose(torch.cat(sc.ood_mean).cpu().numpy(), ref_out.mean(1), rtol=RTOL)
    thr = np.percentile(ref_in.sum(1), 5)                                          # train_and_test.py:199
    np.testing.assert_allclose(res["threshold"], thr, rtol=RTOL)
    assert abs(res["FPR95"] - float((ref_out.mean(1) > thr).mean())) < 1e-9         # :213, :216
    y = np.r_[np.ones(n), np.zeros(n)]
    assert abs(res["AUROC"] - roc_auc_score(y, np.r_[ref_in.sum(1), ref_out.sum(1)])) < 1e-6
    assert abs(res["accuracy"] - float((ref_in.argmax(1) == lab.numpy()).mean())) < 1e-9


@pytest.mark.gpu
def test_graphed_step_replays_the_eager_step_bit_for_bit():
    """mgproto_b200.pipeline.GraphedStep (head forward + loss + backward + enqueue + update_GMM in one CUDA graph)
    against the same sequence of eager steps on a twin model: logits, feature gradient, means, mixture weights, bank and
    the Adam step count must be identical -- every piece of step-dependent state lives on the device."""
    import copy
    import mgproto_b200 as M
    from mgproto_b200 import ops
    from mgproto_b200.pipeline import GraphedStep
    torch.manual_seed(3)
    C, K, D, T, cap, B, H = 6, 4, 128, 4, 8, 16, 6
    net_a = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 8, 1)), img_size=H, prototype_shape=(C * K, D, 1, 1),
                      proto_layer_rf_info=None, num_classes=C, add_on_layers_type="regular", sz_embedding=8,
                      mem_capacity=cap, mine_K=T).to(_dev())
    net_b = copy.deepcopy(net_a)
    for n in (net_a, net_b):
        n.prototype_optimizer = torch.optim.Adam([{"params": n.prototype_means, "lr": 3e-3}])
        n.train()
    g = torch.Generator().manual_seed(4)
    xs = [torch.randn(B, D, H, H, generator=g).to(_dev()) for _ in range(4)]
    gts = [torch.randint(0, C, (B,), generator=g).to(_dev()) for _ in range(4)]

    def loss_fn(out, gt):
        return ops.mine_cross_entropy(out, gt, 0.2)

    seq = [0, 0, 0, 1, 2, 3, 1]                      # warm-up (2) + 5 replays
    for i in seq:
        x = xs[i].clone().requires_grad_(True)
        out_a = net_a.head(x, gts[i])
        loss_a = loss_fn(out_a, gts[i])
        loss_a.backward()
        net_a.update_GMM()
        grad_a = x.grad
    step = GraphedStep(net_b, loss_fn, xs[0], gts[0], warmup=2)
    assert step.launches >= 10
    for i in seq[2:]:
        v0 = net_b.prototype_means._version
        out_b, loss_b = step(xs[i], gts[i])
        assert net_b.prototype_means._version > v0
    torch.cuda.synchronize()
    assert torch.equal(out_b, out_a) and torch.equal(loss_b, loss_a) and torch.equal(step.x_grad, grad_a)
    assert torch.equal(net_b.prototype_means, net_a.prototype_means)
    assert torch.equal(net_b.last_layer.weight, net_a.last_layer.weight)
    assert torch.equal(net_b.queue.bank, net_a.queue.bank) and torch.equal(net_b.queue.mem_len, net_a.queue.mem_len)
    net_a.sync_optimizer_state()
    net_b.sync_optimizer_state()
    sa = net_a.prototype_optimizer.state[net_a.prototype_means]
    sb = net_b.prototype_optimizer.state[net_b.prototype_means]
    assert int(sa["step"]) == int(sb["step"]) and int(sa["step"]) > 0
    assert torch.equal(sa["exp_avg"], sb["exp_avg"]) and torch.equal(sa["exp_avg_sq"], sb["exp_avg_sq"])
