"""CPU: the numpy oracle against the reference-generated golden outputs at the HEADLINE shapes
(tests/golden/headline.npz, made by tests/golden/make_golden_headline.py from the unmodified reference):
200 classes x 10 prototypes x 128-d, T = 20, 800-row banks, ~150 active classes per update_GMM, Adam state
pre-seeded at step 1000.  This pins the oracle where bench.py measures, and records how far the reference's own
fp32 arithmetic sits from the fp64 oracle (the yardstick for the GPU tolerances)."""
import os

import numpy as np
import pytest

import headline_case as HC
from oracle import mgproto_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "headline.npz")


@pytest.fixture(scope="module")
def hl():
    z = np.load(GOLD)
    g = {k: z[k] for k in z.files}
    C, K, D, cap = (int(g[k]) for k in "C K D cap".split())
    g["mu"], g["sg"], g["wt"] = HC.mixture(C, K, D)
    g["x"], gt = HC.head_batch(int(g["B"]), C, K, D, int(g["H"]), int(g["W"]), g["mu"], gt_fixed=(12, 25, 199, 0, 38, 12))
    assert (gt == g["gt"]).all()
    return g


def normwise(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_head_oracle_vs_reference_headline(hl):
    g = hl
    T = int(g["T"])
    f64 = lambda a: a.astype(np.float64)                                        # noqa: E731
    fw = O.head_forward(f64(g["x"]), f64(g["mu"]), f64(g["sg"]), f64(g["wt"]), g["gt"], T)
    np.testing.assert_allclose(fw["logits"], g["logits"], rtol=1e-4, atol=1e-5)
    fw0 = O.head_forward(f64(g["x"]), f64(g["mu"]), f64(g["sg"]), f64(g["wt"]), None, T)
    np.testing.assert_allclose(fw0["logits"], g["logits_nogt"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(fw0["logp"].reshape(-1, g["mu"].shape[0] * g["mu"].shape[1])[HC.LOGP_ROWS], g["logp_rows"],
                               rtol=1e-4, atol=1e-5)
    sep = (g["top1_val"] - g["top2_val"]) > 1e-5 * g["top1_val"]
    assert sep.mean() > 0.95
    assert (fw0["idx"][:, :, 0][sep] == g["top1_idx"][sep]).all()
    # gradient of the training loss w.r.t. the add-on features (autograd in the reference)
    B, C = g["logits"].shape[:2]
    lg = fw["logits"]
    gl = np.zeros_like(lg)
    for t in range(T):
        z = lg[:, :, t] - lg[:, :, t].max(1, keepdims=True)
        p = np.exp(z) / np.exp(z).sum(1, keepdims=True)
        p[np.arange(B), g["gt"]] -= 1.0
        gl[:, :, t] = p / B * (1.0 if t == 0 else 0.2 / (T - 1))
    gx = O.head_backward(f64(g["x"]), f64(g["mu"]), f64(g["sg"]), f64(g["wt"]), g["gt"], T, gl)
    err = normwise(g["grad_x"], gx[HC.GRAD_X])
    print("reference fp32 grad_x vs fp64 oracle: normwise %.2e" % err)
    assert err < 1e-4


def _oracle_em(g, dtype):
    C, K, D, cap = (int(g[k]) for k in "C K D cap".split())
    rows = HC.bank_rows(C, K, D, cap, g["mu"])
    am, av, flags, short, step0 = HC.em_state(C, K, D)
    bank = O.MemoryBankOracle(C, D, cap)
    bank.data[:] = rows
    bank.mem_len[:] = cap
    for s in short:
        bank.mem_len[s] = int(g["short_len"])
        bank.data[s, int(g["short_len"]):] = 0
    # the enqueue of the labelled step (oracle indices from the fp64 forward)
    fw = O.head_forward(g["x"].astype(np.float64), g["mu"].astype(np.float64), g["sg"].astype(np.float64),
                        g["wt"].astype(np.float64), g["gt"], int(g["T"]))
    upd = np.zeros(C, bool)
    for c, r in O.enqueue_rows(fw["xhat"].astype(np.float32), fw["idx"], g["gt"], C, K, int(g["H"]) * int(g["W"])):
        bank.push(c, r)
        upd[c] = True
    adam = O.AdamOracle((C, K, D), lr=float(g["lr"]), dtype=dtype)
    adam.m, adam.v, adam.t = am.astype(dtype), av.astype(dtype), step0
    mu, wt = g["mu"].astype(dtype), g["wt"].astype(dtype)
    outs = []
    for it in range(2):
        upd = upd | flags[it]
        assert (upd == g["flags%d" % it]).all()
        mu, wt, upd = O.update_gmm(bank, upd, mu, g["sg"].astype(dtype), wt, adam)
        outs.append((mu.copy(), np.stack([wt[i, i * K:(i + 1) * K] for i in range(C)])))
    return bank, outs, adam


def test_enqueue_and_update_gmm_oracle_vs_reference_headline(hl):
    g = hl
    bank, outs, adam = _oracle_em(g, np.float64)
    np.testing.assert_array_equal(bank.mem_len, g["mem_len_after_enqueue"])
    for i, c in enumerate(g["touched"]):                     # the newest slots of every class the step pushed to
        np.testing.assert_allclose(bank.data[c, -HC.BANK_TAIL:], g["bank_tail"][i], rtol=1e-5, atol=1e-6)
    (mu0, pi0), (mu1, pi1) = outs
    e0, e1 = normwise(g["mu_after0"], mu0[HC.MU_AFTER0]), normwise(g["mu_after1"], mu1[HC.MU_AFTER1])
    print("reference fp32 mu after update_GMM vs fp64 oracle: normwise %.2e / %.2e" % (e0, e1))
    assert e0 < 1e-4 and e1 < 1e-4
    np.testing.assert_allclose(pi0, g["pi_after0"], rtol=1e-4)
    np.testing.assert_allclose(pi1, g["pi_after1"], rtol=1e-4)
    assert adam.t == int(g["adam_step"])
    em, ev = normwise(g["adam_m"], adam.m[HC.ADAM]), normwise(g["adam_v"], adam.v[HC.ADAM])
    print("reference fp32 Adam moments vs fp64 oracle: normwise %.2e / %.2e" % (em, ev))
    assert em < 1e-4 and ev < 1e-4
