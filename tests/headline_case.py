"""Seeded inputs of the headline-shape parity cases (BASELINE.json configs[1] mixture: 200 classes x 10 prototypes,
800-row banks; D = 128, and the D = 256 / K = 20 / K = 40 variants) and the feature maps of the small golden cases.
Pure numpy (PCG64 streams are stable across machines), shared by tests/golden/make_golden*.py -- which feed them to
the UNMODIFIED reference and store its outputs -- and by the tests, which regenerate them and feed them to the CUDA
path and to the numpy oracle.  Test infrastructure only."""
import numpy as np

# headline.npz stores fixed samples of the reference's larger outputs (a fixture file stays under 1 MB); the tests take
# the same samples of what they compute
MU_AFTER0 = np.s_[::3, :, ::4]         # mu after the first update_GMM: every 3rd class, every 4th dimension
MU_AFTER1 = np.s_[:, :, ::8]           # mu after the second: every class, every 8th dimension
ADAM = np.s_[::7, :, ::4]              # Adam moments after both calls
GRAD_X = np.s_[:, :, ::2, ::2]         # feature gradient: every other patch row and column
LOGP_ROWS = np.s_[::194]               # rows of the unlabelled log p [B*H*W, P]
BANK_TAIL = 16                         # newest bank rows of every class the labelled step pushed to


def l2n(x, axis):
    return x / np.maximum(np.sqrt((x * x).sum(axis=axis, keepdims=True)), 1e-12)


def mixture(C, K, D, seed=2, sigma_mode="init", pi_mode="rand"):
    """mu as model.py:148-149 (l2-normalised uniform), sigma 1/sqrt(2 pi) (model.py:151) or per-prototype /
    per-dimension random, pi rows on the simplex."""
    r = np.random.default_rng(seed)
    mu = l2n(r.random((C, K, D), dtype=np.float64), 2).astype(np.float32)
    if sigma_mode == "init":
        sg = np.full((C, K, D), 1.0 / np.sqrt(2 * np.pi), np.float32)
    elif sigma_mode == "iso":                                   # constant over d inside each prototype
        sg = np.repeat((0.3 + 0.3 * r.random((C, K, 1))).astype(np.float32), D, axis=2)
    else:                                                       # general diagonal
        sg = (0.3 + 0.3 * r.random((C, K, D))).astype(np.float32)
    if pi_mode == "rand":
        e = np.exp(r.standard_normal((C, K)))
        pi = (e / e.sum(1, keepdims=True)).astype(np.float32)
    else:
        pi = np.full((C, K), 1.0 / K, np.float32)
    wt = np.zeros((C, C * K), np.float32)
    for c in range(C):
        wt[c, c * K:(c + 1) * K] = pi[c]
    return mu, sg, wt


def head_batch(B, C, K, D, H, W, mu, seed=1, gt_fixed=()):
    """Add-on feature maps [B,D,H,W]: noise plus, on a third of the patches, a pull towards a random prototype
    (so top-k gaps vary); labels hit the classes in gt_fixed first (classes whose prototypes straddle the
    128-row tensor-core tiles)."""
    r = np.random.default_rng(seed)
    x = r.standard_normal((B, D, H, W)).astype(np.float32)
    P = C * K
    pick = r.integers(0, P, size=(B, H, W))
    pull = (r.random((B, H, W)) < 0.33).astype(np.float32) * (2.0 + 4.0 * r.random((B, H, W))).astype(np.float32)
    x = x + np.transpose(mu.reshape(P, D)[pick], (0, 3, 1, 2)) * pull[:, None] * np.sqrt(D).astype(np.float32)
    x = x * (0.5 + r.random((B, 1, H, W))).astype(np.float32)
    gt = r.integers(0, C, size=(B,)).astype(np.int64)
    for i, c in enumerate(gt_fixed):
        if i < B:
            gt[i] = c
    return x, gt


def fixture_features(B, D, H, W, seed, it):
    """Add-on feature maps [B,D,H,W] of iteration `it` of the small golden cases (tests/golden/make_golden.py): what
    the reference's 'regular' add-on layers (two 1x1 convolutions) make of a random 3-channel image -- an affine map of
    rank 3, fixed per case -- with every patch scaled by 1 .. 1.5.  Element-wise float64 arithmetic only, so every
    machine regenerates the same values."""
    r = np.random.default_rng(seed)
    a = r.standard_normal((3, D, 1, 1)) / np.sqrt(3)
    c = 0.2 * r.standard_normal((D, 1, 1))
    r = np.random.default_rng([seed, it])
    img = r.standard_normal((B, 3, 1, H, W))
    x = c + a[0] * img[:, 0] + a[1] * img[:, 1] + a[2] * img[:, 2]
    return (x * (1.0 + 0.5 * r.random((B, 1, H, W)))).astype(np.float32)


def bank_rows(C, K, D, cap, mu, seed=6):
    """SURVEY 8(d): rows = l2_normalize(mu_c,k + 0.3 randn), every class full."""
    r = np.random.default_rng(seed)
    kk = r.integers(0, K, size=(C, cap))
    rows = mu[np.arange(C)[:, None], kk] + 0.3 * r.standard_normal((C, cap, D)).astype(np.float32)
    return l2n(rows.astype(np.float32), 2)


def em_state(C, K, D, seed=7, n_active=(160, 140), n_short=5, step0=1000):
    """Pre-seeded Adam state (as after `step0` steps), the update flags of two successive update_GMM calls, and a few
    flagged classes whose bank is not full (their flag is cleared without an update, model.py:287-289)."""
    r = np.random.default_rng(seed)
    m = (1e-3 * r.standard_normal((C, K, D))).astype(np.float32)
    v = ((1e-3) ** 2 * (0.1 + r.random((C, K, D)))).astype(np.float32)
    flags = []
    for n in n_active:
        f = np.zeros(C, bool)
        f[r.choice(C, size=min(n, C), replace=False)] = True
        flags.append(f)
    short = r.choice(C, size=min(n_short, C), replace=False)
    for f in flags:
        f[short] = True
    return m, v, flags, short, step0
