"""Pins oracle/mgproto_oracle.py against fixtures produced by the unmodified reference
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

from oracle import mgproto_oracle as O


def _i(g, k):
    return int(g[k])


def test_compute_log_prob(golden):
    g = golden
    xhat = O.features_to_rows(O.l2_normalize(g["it0_x_add"], axis=1))
    lp = O.compute_log_prob(xhat, g["it0_mu"], g["sigma"])
    np.testing.assert_allclose(lp, g["it0_logp"], rtol=2e-5, atol=2e-5)


def test_ka1_isotropic_identity(golden):
    """SURVEY KA1: with sigma = 1/sqrt(2 pi), log p = -pi |x - mu|^2."""
    g = golden
    if not np.allclose(g["sigma"], 1 / np.sqrt(2 * np.pi)):
        pytest.skip("general sigma case")
    xhat = O.features_to_rows(O.l2_normalize(g["it0_x_add"].astype(np.float64), axis=1))
    mu = g["it0_mu"].astype(np.float64).reshape(-1, _i(g, "D"))
    ref = -np.pi * ((xhat[:, None] - mu[None]) ** 2).sum(-1)
    np.testing.assert_allclose(g["it0_logp"].reshape(ref.shape), ref, atol=2e-5)


def test_topk_and_logits(golden):
    g = golden
    T = _i(g, "T")
    for use_gt in (True, False):
        fw = O.head_forward(g["it0_x_add"], g["it0_mu"], g["sigma"], g["it0_weight"],
                            g["it0_gt"] if use_gt else None, T)
        ref = g["it0_logits"] if use_gt else g["it0_logits_nogt"]
        np.testing.assert_allclose(fw["logits"], ref, rtol=1e-4, atol=1e-5)
    # raw top-k (before the wrong-class rule): values always, indices where separated
    fw = O.head_forward(g["it0_x_add"], g["it0_mu"], g["sigma"], g["it0_weight"], None, T)
    np.testing.assert_allclose(fw["vals"], g["it0_topk_vals"], rtol=1e-4, atol=1e-12)
    v = g["it0_topk_vals"].astype(np.float64)
    gap_prev = np.ones_like(v, dtype=bool)
    gap_next = np.ones_like(v, dtype=bool)
    rel = np.abs(np.diff(v, axis=-1)) > 1e-5 * np.abs(v[..., :-1])
    gap_prev[..., 1:] = rel
    gap_next[..., :-1] = rel
    sep = gap_prev & gap_next
    assert sep.mean() > 0.5
    assert (fw["idx"][sep] == g["it0_topk_idx"][sep]).all()


def test_push_forward(golden):
    g = golden
    xhat, dist = O.push_forward(g["it0_x_add"], g["it0_mu"], g["sigma"])
    np.testing.assert_allclose(xhat[g["sample"]], g["it0_push_feat"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(dist, g["it0_push_dist"], rtol=1e-4, atol=1e-12)


def test_head_backward(golden):
    g = golden
    if g["name"] != "tiny":
        pytest.skip("python-loop backward oracle: tiny case only")
    B, C, T = _i(g, "B"), _i(g, "C"), _i(g, "T")
    x = g["it0_x_add"].astype(np.float64)
    fw = O.head_forward(x, g["it0_mu"].astype(np.float64), g["sigma"].astype(np.float64),
                        g["it0_weight"].astype(np.float64), g["it0_gt"], T)
    # d loss / d logits for loss = CE(level0) + 0.2 * mean_t>=1 CE(level t)
    lg = fw["logits"]
    sm = np.exp(lg - O.logsumexp(lg, axis=1, keepdims=True))
    oh = np.zeros((B, C))
    oh[np.arange(B), g["it0_gt"]] = 1
    wts = np.full(T, 0.2 / (T - 1))
    wts[0] = 1.0
    gl = (sm - oh[:, :, None]) / B * wts[None, None, :]
    gx = O.head_backward(x, g["it0_mu"].astype(np.float64), g["sigma"].astype(np.float64),
                         g["it0_weight"].astype(np.float64), g["it0_gt"], T, gl)
    np.testing.assert_allclose(gx[g["sample"]], g["it0_grad_x"], rtol=2e-3, atol=2e-6)


def test_enqueue_and_bank_sequence(golden):
    g = golden
    C, K, D, T, cap = (_i(g, k) for k in "C K D T cap".split())
    hw = _i(g, "H") * _i(g, "W")
    bank = O.MemoryBankOracle(C, D, cap)
    for it in range(_i(g, "iters")):
        pre = "it%d_" % it
        fw = O.head_forward(g[pre + "x_add"], g[pre + "mu"], g["sigma"], g[pre + "weight"], g[pre + "gt"], T)
        # use the reference-consistent top-1 indices (ties are vanishingly rare in these fixtures)
        for c, rows in O.enqueue_rows(fw["xhat"], fw["idx"], g[pre + "gt"], C, K, hw):
            assert rows.shape[0] <= cap
            bank.push(c, rows)
        np.testing.assert_array_equal(bank.mem_len, g[pre + "mem_len"])
        for c in range(C):
            n = bank.mem_len[c]
            np.testing.assert_allclose(bank.data[c, :n], g[pre + "bank"][c, :n], rtol=1e-5, atol=1e-6)


def test_update_gmm_sequence(golden):
    """Whole-sequence parity of update_GMM incl. the Adam cross-class coupling (KA7):
    bank states are taken from the fixture, mu / pi / Adam state are carried by the oracle."""
    g = golden
    C, K, D, cap = (_i(g, k) for k in "C K D cap".split())
    f64 = np.float64
    adam = O.AdamOracle((C, K, D), lr=float(g["lr"]))
    mu = g["mu0"].astype(f64)
    wt = g["weight0"].astype(f64)
    for it in range(_i(g, "iters")):
        pre = "it%d_" % it
        np.testing.assert_allclose(mu, g[pre + "mu"], rtol=1e-4, atol=2e-6)
        bank = O.MemoryBankOracle(C, D, cap, dtype=f64)
        bank.data[:] = g[pre + "bank"]
        bank.mem_len[:] = g[pre + "mem_len"]
        mu, wt, upd = O.update_gmm(bank, g[pre + "updated"], mu, g["sigma"].astype(f64), wt, adam,
                                   num_em_loop=_i(g, "num_em_loop"), alpha=float(g["alpha"]), tau=float(g["tau"]))
        assert not upd.any()
        np.testing.assert_allclose(mu, g[pre + "mu_after"], rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(wt, g[pre + "weight_after"], rtol=1e-4, atol=1e-7)
    assert adam.t == int(g["adam_step"])
    np.testing.assert_allclose(adam.m, g["adam_m"], rtol=1e-3, atol=1e-7)
    np.testing.assert_allclose(adam.v, g["adam_v"], rtol=1e-3, atol=1e-10)


def test_em_building_blocks(golden):
    g = golden
    K = _i(g, "K")
    x = g["em_x"]
    mu, sg, pi = g["em_mu"][0], g["em_sigma"][0], g["em_pi"].reshape(K)
    ll, log_resp = O.e_step(x, mu, sg, pi)
    np.testing.assert_allclose(ll, g["em_loglik"], rtol=1e-5)
    np.testing.assert_allclose(log_resp, g["em_log_resp"][:, :, 0], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(np.exp(log_resp).sum(1), 1.0, rtol=1e-5)          # KA2
    p, m, v = O.m_step(x, g["em_log_resp"][:, :, 0], float(g["alpha"]))
    np.testing.assert_allclose(p, g["em_mstep_pi"].reshape(K), rtol=1e-5)
    np.testing.assert_allclose(p.sum(), 1.0, rtol=1e-5)                           # KA2
    np.testing.assert_allclose(m, g["em_mstep_mu"][0], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(v, g["em_mstep_var"][0], rtol=2e-3, atol=2e-5)
    np.testing.assert_allclose(O.score(x, mu, sg, pi, as_average=False), g["em_score"], rtol=1e-5)
    np.testing.assert_allclose(O.estimate_log_prob(x, mu, sg), g["em_est_log_prob"][:, :, 0], rtol=1e-5)
    pn, grad, loss = O.m_step_diversified_grad(x.astype(np.float64), g["em_log_resp"][:, :, 0].astype(np.float64),
                                               mu.astype(np.float64), sg.astype(np.float64),
                                               pi.astype(np.float64), float(g["alpha"]))
    np.testing.assert_allclose(grad, g["em_div_grad"], rtol=1e-4, atol=1e-7)      # KA6
    np.testing.assert_allclose(loss, g["em_div_loss"], rtol=1e-5)
    np.testing.assert_allclose(pn, g["em_div_pi"].reshape(K), rtol=1e-5)
