"""State the library keeps between calls must follow every write to the model (-m gpu).

The kernels read mu, sigma, the mixture weights, the bank and the Adam state through raw pointers, and some derived
state is kept across calls: the isotropy answer for sigma (which selects the tensor-core kernels), the fp16 shadow of
the bank, the Adam step count held on the device between update_GMM calls, and the whole training step as a CUDA graph
(pipeline.GraphedStep).  Each test below writes the model through one route the reference's own loop uses -- in-place
ops, `.data` writes (push.py:198), push_prototypes, optimiser reloads and replacement, a StepLR schedule, model
load_state_dict, MemoryBank.push, the last-layer utilities -- with the consumers warmed up before the write, and then
compares every consumer with a float64 restatement of the CURRENT parameters (or, for the graphed step, with an eager
twin model bit for bit).  A stale result is O(1) away from the reference; the tolerances are the suite's usual ones.

No test here launches an isotropic-sigma kernel on anisotropic sigma: the recycled-sigma case checks the host-side
decision only."""
import contextlib
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import headline_case as HC

pytestmark = pytest.mark.gpu

C, K, T, B, H = 20, 10, 4, 4, 14
CAP = 24
LR = 3e-3
FLAGS = (3, 11)                  # classes update_GMM works on: 6 Adam steps per call, so bias correction matters


def _dev():
    return torch.device("cuda:0")


def _t(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device=_dev())


def _f64(t):
    return t.detach().double().cpu().numpy()


def normwise(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / np.abs(b).max())


def _net(D, seed=0, cap=CAP):
    """C = 20 classes x K = 10 prototypes, sigma = the model's isotropic initial value, random pi rows."""
    import mgproto_b200 as M
    torch.manual_seed(seed)
    net = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 16, 1)), img_size=H, prototype_shape=(C * K, D, 1, 1),
                    proto_layer_rf_info=None, num_classes=C, add_on_layers_type="regular", sz_embedding=8,
                    mem_capacity=cap, mine_K=T).to(_dev())
    mu, sg, wt = HC.mixture(C, K, D, seed=30 + seed)
    net.prototype_means.data.copy_(_t(mu))
    net.prototype_covs.data.copy_(_t(sg))
    net.last_layer.weight.data.copy_(_t(wt))
    net.prototype_optimizer = torch.optim.Adam([{"params": net.prototype_means, "lr": LR}])
    net.train()
    return net


def _fill_bank(net, seed):
    """Every class's ring full of rows near its prototypes."""
    q = net.queue
    rows = HC.bank_rows(C, K, q.dim_feature, q.cap_cls, net.prototype_means.detach().cpu().numpy(), seed=seed)
    q.bank.copy_(_t(rows))
    q.mem_len.fill_(q.cap_cls)
    q.head.zero_()


def _batch(D, seed):
    mu = HC.mixture(C, K, D, seed=30)[0]
    x, gt = HC.head_batch(B, C, K, D, H, H, mu, seed=seed)
    return _t(x), _t(gt, torch.int64)


def _far_rows(x, n, seed):
    """n normalised patches of x: each is far from every current mean, so a result computed from the old means
    cannot pass within tolerance."""
    xhat = F.normalize(x.permute(0, 2, 3, 1).reshape(-1, x.shape[1]), dim=1)
    pick = torch.randperm(xhat.shape[0], generator=torch.Generator().manual_seed(seed))[:n]
    return xhat[pick.to(x.device)].clone()


@contextlib.contextmanager
def em_serial():
    """update_GMM's tensor-core kernel one bank tile at a time instead of pipelined (csrc/em_tc.cu)."""
    from mgproto_b200 import _lib
    lib = _lib.load()
    prev = lib.mgp_set_option(b"em_pipe", 0)
    try:
        yield
    finally:
        lib.mgp_set_option(b"em_pipe", prev)


# ------------------------------------------------------------------------------------------------ consumers
def check_consumers(net, x, gt):
    """compute_log_prob, the labelled and unlabelled head, head_level0 and push_search against float64 on the
    model's current mu / sigma / pi."""
    from mgproto_b200 import ops
    from oracle import mgproto_oracle as O
    D = net.prototype_means.shape[2]
    P = C * K
    mu, sg, wt = _f64(net.prototype_means), _f64(net.prototype_covs), _f64(net.last_layer.weight)
    xhat = ops.normalize_fwd(x)[0]
    # compute_log_prob in auto mode: isotropic sigma, D in {128, 256} -> the TMEM-resident [N,P] kernel
    lp = net.compute_log_prob(xhat).view(-1, P)
    x64, mu64, sg64 = xhat.double(), _t(mu, torch.float64).view(P, D), _t(sg, torch.float64).view(P, D)
    ref = (-0.5 * D * np.log(2 * np.pi) - sg64.log().sum(1)[None, :]
           - 0.5 * (((x64[:, None, :] - mu64[None]) / sg64[None]) ** 2).sum(-1))
    torch.testing.assert_close(lp.double(), ref, rtol=2e-5, atol=2e-5)
    # heads
    xn = _f64(x)
    g = gt.cpu().numpy()
    fw = O.head_forward(xn, mu, sg, wt, g, T)
    fw0 = O.head_forward(xn, mu, sg, wt, None, T)
    with torch.no_grad():
        lg = ops.head_forward(x, net.prototype_means, net.prototype_covs, net.last_layer.weight, gt, T, net.math_mode)[0]
        lg0 = ops.head_forward(x, net.prototype_means, net.prototype_covs, net.last_layer.weight, None, T,
                               net.math_mode)[0]
    np.testing.assert_allclose(lg.cpu().numpy(), fw["logits"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(lg0.cpu().numpy(), fw0["logits"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(net.head_level0(x).cpu().numpy(), fw0["logits"][:, :, 0], rtol=1e-4, atol=1e-5)
    # push_search: per image, the best patch of each own-class prototype
    arg, val, _ = net.push_search(x, gt)
    lp64 = fw["logp"].reshape(B, H * H, P)
    a = arg.cpu().numpy()
    for b in range(B):
        own = lp64[b, :, g[b] * K:(g[b] + 1) * K]                            # [HW, K]
        np.testing.assert_allclose(val[b].cpu().numpy(), -np.exp(own.max(0)), rtol=1e-4)
        picked = own[a[b], np.arange(K)]
        assert (picked >= own.max(0) - 1e-4 * np.abs(own.max(0))).all(), b


def check_update_gmm(net, adam, flags=FLAGS):
    """Flag `flags`, run the float64 oracle from the model's current bank / mu / pi and `adam` (the optimiser state
    the model should be at), then update_GMM: mu, pi, the Adam moments and step must match."""
    from oracle import mgproto_oracle as O
    q = net.queue
    D = net.prototype_means.shape[2]
    q.updated.zero_()
    q.updated[list(flags)] = 1
    mu0, sg, wt0 = _f64(net.prototype_means), _f64(net.prototype_covs), _f64(net.last_layer.weight)
    bank = O.MemoryBankOracle(C, D, q.cap_cls, dtype=np.float64)
    bank.data[:] = _f64(q.linear())
    bank.mem_len[:] = q.mem_len.cpu().numpy()
    upd = np.zeros(C, bool)
    upd[list(flags)] = True
    mu_ref, wt_ref, _ = O.update_gmm(bank, upd, mu0, sg, wt0, adam, num_em_loop=net.num_em_loop, alpha=net.alpha,
                                     tau=net.tau)
    net.update_GMM()
    net.sync_optimizer_state()
    got = _f64(net.prototype_means)
    e_mu, e_mv = normwise(got, mu_ref), normwise(got - mu0, mu_ref - mu0)
    assert e_mu < 1e-4 and e_mv < 1e-3, (e_mu, e_mv)
    np.testing.assert_allclose(_f64(net.last_layer.weight), wt_ref, rtol=1e-4, atol=1e-9)
    st = net.prototype_optimizer.state[net.prototype_means]
    assert int(st["step"]) == adam.t
    assert normwise(_f64(st["exp_avg"]), adam.m) < 1e-4
    assert normwise(_f64(st["exp_avg_sq"]), adam.v) < 1e-4


def _adam_from(state):
    from oracle import mgproto_oracle as O
    adam = O.AdamOracle((C, K, state["exp_avg"].shape[-1]), lr=LR)
    adam.t, adam.m, adam.v = int(state["step"]), _f64(state["exp_avg"]), _f64(state["exp_avg_sq"])
    return adam


# ------------------------------------------------------------------------------------------------ W0 / W1 / W2
@pytest.mark.parametrize("route", ["inplace", "data_rows", "data_whole", "push_prototypes"])
@pytest.mark.parametrize("D", [128, 256])
def test_mean_writes_reach_every_consumer(D, route):
    """W0: an in-place op under no_grad (bumps the version counter).  W1: the reference push's
    `prototype_means[c, k].data.copy_(v)` and a whole-tensor `.data.copy_` (no version bump).  W2:
    mgproto_b200.push_prototypes.  Every consumer runs once before the write (warm caches), then must agree with
    float64 on the new means; update_GMM then starts from them."""
    import mgproto_b200 as M
    from oracle import mgproto_oracle as O
    net = _net(D)
    x, gt = _batch(D, seed=40)
    check_consumers(net, x, gt)
    mu_before = net.prototype_means.detach().clone()
    if route == "inplace":
        with torch.no_grad():
            net.prototype_means.copy_(F.normalize(torch.rand(C, K, D, device=_dev()), dim=2))
    elif route == "data_rows":
        v = _far_rows(x, 6, seed=1)
        for i, (c, k) in enumerate([(0, 0), (int(gt[0]), 3), (int(gt[1]), K - 1), (7, 5), (C - 1, 2), (12, 9)]):
            net.prototype_means[c, k].data.copy_(v[i])
    elif route == "data_whole":
        net.prototype_means.data.copy_(_far_rows(x, C * K, seed=2).view(C, K, D))
    else:
        g = torch.Generator().manual_seed(5)
        n = 2 * C
        imgs = torch.randn(n, 3, H, H, generator=g)
        labs = torch.arange(n) % C
        loader = [(imgs[i:i + 8], labs[i:i + 8]) for i in range(0, n, 8)]
        res = M.push_prototypes(loader, net, log=lambda *_: None)
        assert (res["image"] >= 0).sum() >= C
    moved = (net.prototype_means.detach() - mu_before).norm(dim=2) > 0.1
    assert int(moved.sum()) >= 6
    check_consumers(net, x, gt)
    _fill_bank(net, seed=6)
    check_update_gmm(net, O.AdamOracle((C, K, D), lr=LR))


# ------------------------------------------------------------------------------------------------ W3
def test_recycled_sigma_block_gets_a_fresh_isotropy_answer():
    """W3: the isotropy answer is cached per sigma.  An isotropic sigma is checked and freed; the caching allocator
    hands its block to the next allocation of that size, and a fresh tensor starts again at version 0.  The
    anisotropic sigma allocated there must be judged anisotropic, so that the tensor-core kernels that assume
    isotropy are not chosen for it.  Host-side decision only: nothing is launched on it."""
    from mgproto_b200 import ops, _lib
    if not _lib.load().mgp_has_tensor_core_path():
        pytest.skip("library built without the tcgen05 path")
    D, P, HW = 128, C * K, H * H
    torch.cuda.synchronize()
    iso = torch.full((P, D), 0.4, device=_dev())
    assert ops.sigma_is_isotropic(iso)
    ptr = iso.data_ptr()
    del iso
    aniso = torch.rand((P, D), device=_dev())                 # one allocation of the same size, version 0
    recycled = aniso.data_ptr() == ptr
    assert aniso._version == 0
    assert not ops.sigma_is_isotropic(aniso), "stale isotropy answer (block recycled: %s)" % recycled
    assert ops._stage_for_top1(B, HW, P, D, aniso, "auto")[1]
    assert not ops.sigma_is_isotropic(aniso.view(C, K, D))


# ------------------------------------------------------------------------------------------------ W4
@pytest.mark.parametrize("case", ["reload_at_last_seen_step", "reload_earlier_step", "fresh_adam"])
def test_optimizer_reload_or_replacement_reseeds_the_adam_step(case):
    """W4: update_GMM keeps Adam's step count on the device between calls.  After
    `prototype_optimizer.load_state_dict(sd)` (sd taken at the step last folded back, or at an earlier one) or after
    assigning a fresh Adam, with no sync_optimizer_state in between, the next update_GMM must continue from the
    LOADED / fresh state, exactly as torch.optim.Adam would."""
    from oracle import mgproto_oracle as O
    D = 128
    net = _net(D)
    _fill_bank(net, seed=6)
    check_update_gmm(net, O.AdamOracle((C, K, D), lr=LR))       # step 6, folded back
    opt = net.prototype_optimizer

    def em():
        net.queue.updated[list(FLAGS)] = 1
        net.update_GMM()

    if case == "reload_at_last_seen_step":
        sd = copy.deepcopy(opt.state_dict())
        em()
        em()
        opt.load_state_dict(sd)
        adam = _adam_from(sd["state"][0])
    elif case == "reload_earlier_step":
        sd = copy.deepcopy(opt.state_dict())
        em()
        opt.state_dict()                                          # a checkpoint: folds step 12 back
        em()
        opt.load_state_dict(sd)
        adam = _adam_from(sd["state"][0])
    else:
        em()
        em()
        net.prototype_optimizer = torch.optim.Adam([{"params": net.prototype_means, "lr": LR}])
        adam = O.AdamOracle((C, K, D), lr=LR)
    assert adam.t <= 6
    check_update_gmm(net, adam)


# ------------------------------------------------------------------------------------------------ W5
@pytest.mark.parametrize("D,path", [(64, "cluster"), (128, "tc"), (256, "tc"), (256, "tc_serial")])
def test_loaded_or_pushed_bank_reaches_update_gmm(D, path):
    """W5: after update_GMM has built the fp16 shadow of the bank (tensor-core path: D in {128, 256}, isotropic
    sigma), `load_state_dict` of another model's bank and means, then one MemoryBank.push: each following update_GMM
    must match the oracle started from the bank the model now holds.  D = 64 runs the fp32 cluster kernel (control)."""
    from oracle import mgproto_oracle as O
    net = _net(D)
    _fill_bank(net, seed=6)
    adam = O.AdamOracle((C, K, D), lr=LR)
    with em_serial() if path == "tc_serial" else contextlib.nullcontext():
        check_update_gmm(net, adam)
        other = _net(D, seed=1)
        _fill_bank(other, seed=9)
        sd = other.state_dict()
        net.load_state_dict(sd)
        for c in range(C):
            assert torch.equal(net.queue.linear()[c], sd["queue.cls%d" % c])
        assert torch.equal(net.prototype_means, other.prototype_means)
        check_update_gmm(net, adam)
        c = FLAGS[0]
        rows = F.normalize(net.prototype_means.detach()[c, :5] + 0.3 * torch.randn(5, D, device=_dev()), dim=1)
        net.queue.push(rows, torch.full((5,), c, dtype=torch.int64, device=_dev()))
        assert torch.equal(net.queue.linear()[c, -5:], rows)
        check_update_gmm(net, adam, flags=(c,))


# ------------------------------------------------------------------------------------------------ W6
def test_last_layer_utilities_reach_head_and_update_gmm():
    """W6: set_last_layer_incorrect_connection and prune_prototypes_topM write last_layer.weight through `.data`:
    the heads and update_GMM's pi must use the new weights."""
    from oracle import mgproto_oracle as O
    D = 128
    net = _net(D)
    _fill_bank(net, seed=6)
    adam = O.AdamOracle((C, K, D), lr=LR)
    x, gt = _batch(D, seed=41)
    check_consumers(net, x, gt)
    net.set_last_layer_incorrect_connection(0.0)
    assert torch.equal(net.last_layer.weight[0, :K], torch.full((K,), 1.0 / K, device=_dev()))
    check_consumers(net, x, gt)
    check_update_gmm(net, adam)
    net.last_layer.weight.data.copy_(_t(HC.mixture(C, K, D, seed=50)[2]))
    net.prune_prototypes_topM(top_M=4)
    pruned = (net.last_layer.weight == 0).sum().item() - C * (C - 1) * K
    assert pruned == C * (K - 4)
    check_consumers(net, x, gt)
    check_update_gmm(net, adam)


# ------------------------------------------------------------------------------------------------ W7
@pytest.mark.parametrize("change", ["step_lr", "optimizer_load_state_dict", "mean_data_write"])
def test_graphed_step_follows_changes_between_replays(change):
    """W7: pipeline.GraphedStep replayed around a change the reference's loop makes between steps -- a StepLR step on
    prototype_optimizer (main.py steps one every epoch), a prototype_optimizer.load_state_dict, a `.data` write to
    the means -- plus an optimiser checkpoint (state_dict) mid-way.  The replayed steps must equal an eager twin bit for
    bit: logits, loss, feature gradient, mu, pi, bank and the Adam state."""
    import mgproto_b200 as M
    from mgproto_b200 import ops
    from mgproto_b200.pipeline import GraphedStep
    torch.manual_seed(3)
    Cg, Kg, D, Tg, cap, Bg, Hg = 6, 4, 128, 4, 8, 16, 6
    net_a = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 8, 1)), img_size=Hg, prototype_shape=(Cg * Kg, D, 1, 1),
                      proto_layer_rf_info=None, num_classes=Cg, add_on_layers_type="regular", sz_embedding=8,
                      mem_capacity=cap, mine_K=Tg).to(_dev())
    net_b = copy.deepcopy(net_a)
    nets = (net_a, net_b)
    for n in nets:
        n.prototype_optimizer = torch.optim.Adam([{"params": n.prototype_means, "lr": LR}])
        n.train()
    g = torch.Generator().manual_seed(4)
    xs = [torch.randn(Bg, D, Hg, Hg, generator=g).to(_dev()) for _ in range(5)]
    gts = [torch.randint(0, Cg, (Bg,), generator=g).to(_dev()) for _ in range(5)]

    def loss_fn(out, gt):
        return ops.mine_cross_entropy(out, gt, 0.2)

    def eager(i):
        x = xs[i].clone().requires_grad_(True)
        out = net_a.head(x, gts[i])
        loss = loss_fn(out, gts[i])
        loss.backward()
        net_a.update_GMM()
        return out, loss, x.grad

    for i in (0, 0):                                               # GraphedStep's warm-up steps
        eager(i)
    step = GraphedStep(net_b, loss_fn, xs[0], gts[0], warmup=2)
    sd = None
    for i in (1, 2):
        eager(i)
        step(xs[i], gts[i])
        if i == 1:
            sd = [copy.deepcopy(n.prototype_optimizer.state_dict()) for n in nets]    # checkpoint (folds the step)
    ckpt_step = int(sd[0]["state"][0]["step"])
    assert int(sd[1]["state"][0]["step"]) == ckpt_step > 0
    keep = []
    if change == "step_lr":
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")                        # (scheduler stepped without optimizer.step())
            for n in nets:
                torch.optim.lr_scheduler.StepLR(n.prototype_optimizer, step_size=1, gamma=0.4).step()
        assert net_b.prototype_optimizer.param_groups[0]["lr"] == pytest.approx(0.4 * LR)
    elif change == "optimizer_load_state_dict":
        for n, s in zip(nets, sd):
            keep.append(dict(n.prototype_optimizer.state[n.prototype_means]))    # the replaced moments stay allocated
            n.prototype_optimizer.load_state_dict(s)
    else:
        v = _far_rows(xs[3], 3, seed=7)
        for n in nets:
            for i, (c, k) in enumerate([(0, 1), (2, 3), (Cg - 1, 0)]):
                n.prototype_means[c, k].data.copy_(v[i])
    for i in (3, 1, 4):
        out_a, loss_a, grad_a = eager(i)
        out_b, loss_b = step(xs[i], gts[i])
        torch.cuda.synchronize()
        assert torch.equal(out_b, out_a) and torch.equal(loss_b, loss_a) and torch.equal(step.x_grad, grad_a), i
    assert torch.equal(net_b.prototype_means, net_a.prototype_means)
    assert torch.equal(net_b.last_layer.weight, net_a.last_layer.weight)
    assert torch.equal(net_b.queue.bank, net_a.queue.bank) and torch.equal(net_b.queue.mem_len, net_a.queue.mem_len)
    for n in nets:
        n.sync_optimizer_state()
    sa = net_a.prototype_optimizer.state[net_a.prototype_means]
    sb = net_b.prototype_optimizer.state[net_b.prototype_means]
    assert int(sa["step"]) == int(sb["step"]) > ckpt_step
    assert torch.equal(sa["exp_avg"], sb["exp_avg"]) and torch.equal(sa["exp_avg_sq"], sb["exp_avg_sq"])
    step.close()
