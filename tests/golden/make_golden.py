#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/*.npz by running the UNMODIFIED
reference (cwangrun/MGProto, a checkout named by $MGPROTO_REFERENCE) on CPU.

    MGPROTO_REFERENCE=<reference checkout> python tests/golden/make_golden.py

The feature maps are regenerated from seeds by tests/headline_case.py (numpy) on both
sides, so only the reference's outputs are stored; of the feature gradients and the
normalised features, every hw_stride-th patch row and column (a fixture file stays
under 1 MB).  Nothing in tests/, bench.py or smoke() reads the reference.

Only this script imports the reference.  It touches no reference file; the two
shims below exist because the reference hard-codes ``.cuda()`` (model.py:391, :472)
and requires a backbone whose repr starts with VGG/RES/DENSE (model.py:107-115).
"""
import os
import sys

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.environ["MGPROTO_REFERENCE"])
torch.Tensor.cuda = lambda self, *a, **k: self          # CPU shim for hard-coded .cuda()
import model as ref_model                               # noqa: E402  (the reference's model.py)
import headline_case as HC                              # noqa: E402

OUT = HERE


class ResTiny(nn.Module):
    """1x1-conv stand-in backbone; repr starts with 'RES' as model.py:108 requires."""

    def __init__(self, cin):
        super().__init__()
        self.conv = nn.Conv2d(3, cin, kernel_size=1)

    def forward(self, x):
        return self.conv(x)


def build(C, K, D, cap, T, cin=16, seed=0):
    torch.manual_seed(seed)
    m = ref_model.MGProto(features=ResTiny(cin), img_size=14, prototype_shape=(C * K, D, 1, 1),
                          proto_layer_rf_info=None, num_classes=C, init_weights=True,
                          prototype_activation_function='log', add_on_layers_type='regular',
                          sz_embedding=8, mem_capacity=cap, mine_K=T)
    m.prototype_optimizer = torch.optim.Adam([{'params': m.prototype_means, 'lr': 3e-3}])
    return m


def bank_arrays(m, C):
    return (np.stack([getattr(m.queue, 'cls%d' % i).numpy().copy() for i in range(C)]),
            m.queue.mem_len.numpy().copy())


def loss_fn(out, gt):
    ce0 = F.cross_entropy(out[:, :, 0], gt)
    mine = sum(F.cross_entropy(out[:, :, k], gt) for k in range(1, out.shape[2])) / (out.shape[2] - 1)
    return ce0 + 0.2 * mine                                              # train_and_test.py:37-41,55


def make_case(name, C, K, D, B, H, W, T, cap, iters, sigma_mode, pi_mode, seed, hw_stride):
    sample = np.s_[:, :, ::hw_stride, ::hw_stride]
    g = torch.Generator().manual_seed(seed)
    m = build(C, K, D, cap, T, seed=seed)
    m.train()
    if sigma_mode == 'rand':                                             # general diagonal path
        m.prototype_covs.data.copy_(0.2 + 0.6 * torch.rand(C, K, D, generator=g))
    if pi_mode == 'rand':
        pi = torch.softmax(torch.randn(C, K, generator=g), dim=1)
        wt = torch.zeros(C, C * K)
        for c in range(C):
            wt[c, c * K:(c + 1) * K] = pi[c]
        m.last_layer.weight.data.copy_(wt)
    rec = dict(C=C, K=K, D=D, B=B, H=H, W=W, T=T, cap=cap, iters=iters, alpha=m.alpha, tau=m.tau,
               num_em_loop=m.num_em_loop, lr=3e-3, seed=seed, hw_stride=hw_stride)
    rec['mu0'] = m.prototype_means.detach().numpy().copy()
    rec['sigma'] = m.prototype_covs.detach().numpy().copy()
    rec['weight0'] = m.last_layer.weight.detach().numpy().copy()

    for it in range(iters):
        img = None                                                       # conv_features is pointed at x_leaf
        gt = torch.randint(0, C, (B,), generator=g)
        # keep every push within capacity: the reference's over-capacity branch draws an
        # unseeded randperm (utils/memory.py:51-53) and would make the fixture RNG-dependent
        while int(torch.bincount(gt, minlength=C).max()) * K > cap:
            gt = torch.randint(0, C, (B,), generator=g)
        x_leaf = torch.from_numpy(HC.fixture_features(B, D, H, W, seed, it)).requires_grad_(True)
        emb = torch.zeros(B, 8)
        orig = m.conv_features
        m.conv_features = lambda _x, _l=x_leaf, _e=emb: (_l, _e)
        mu_before = m.prototype_means.detach().numpy().copy()
        w_before = m.last_layer.weight.detach().numpy().copy()
        out, _ = m(img, gt)
        loss = loss_fn(out, gt)
        loss.backward()
        m.conv_features = orig
        pre = 'it%d_' % it
        rec[pre + 'gt'] = gt.numpy().copy()
        rec[pre + 'mu'] = mu_before
        rec[pre + 'weight'] = w_before
        rec[pre + 'logits'] = out.detach().numpy().copy()
        rec[pre + 'grad_x'] = x_leaf.grad.numpy()[sample].copy()
        rec[pre + 'loss'] = np.float32(loss.item())
        if it == 0:
            with torch.no_grad():
                bf = F.normalize(x_leaf.detach(), p=2, dim=1)
                feat = bf.permute(0, 2, 3, 1).reshape(-1, D)
                lp = m.compute_log_prob(feat)
                prob = lp.exp().reshape(B, H * W, C * K).permute(0, 2, 1)
                v, ix = torch.topk(prob, T, dim=2)
                rec['it0_logp'] = lp.numpy().copy()
                rec['it0_topk_vals'] = v.numpy().copy()
                rec['it0_topk_idx'] = ix.numpy().copy()
                m.conv_features = lambda _x, _l=x_leaf.detach(), _e=emb: (_l, _e)
                o2, _ = m(img, None)                                     # eval-style call, gt=None
                pf_feat, pf_dist = m.push_forward(img)
                m.conv_features = orig
                rec['it0_logits_nogt'] = o2.numpy().copy()
                rec['it0_push_feat'] = pf_feat.numpy()[sample].copy()
                rec['it0_push_dist'] = pf_dist.numpy().copy()
        bank, mem_len = bank_arrays(m, C)
        rec[pre + 'bank'] = bank
        rec[pre + 'mem_len'] = mem_len
        rec[pre + 'updated'] = m.memory_updated_cls.numpy().copy()
        # train_and_test.py:61-63
        if m.queue.mem_len.sum() > 0:
            m.update_GMM()
        rec[pre + 'mu_after'] = m.prototype_means.detach().numpy().copy()
        rec[pre + 'weight_after'] = m.last_layer.weight.detach().numpy().copy()
    st = m.prototype_optimizer.state[m.prototype_means]
    rec['adam_step'] = np.float32(float(st['step'])) if 'step' in st else np.float32(0)
    rec['adam_m'] = st['exp_avg'].numpy().copy() if 'exp_avg' in st else np.zeros((C, K, D), np.float32)
    rec['adam_v'] = st['exp_avg_sq'].numpy().copy() if 'exp_avg_sq' in st else np.zeros((C, K, D), np.float32)

    # EM building blocks on the fullest class (model.py:303-365, :403-421)
    cfull = int(torch.argmax(m.queue.mem_len))
    n = int(m.queue.mem_len[cfull])
    if n > 0:
        x = getattr(m.queue, 'cls%d' % cfull)[:n].clone()
        mu = m.prototype_means[cfull].detach().unsqueeze(0)
        sg = m.prototype_covs[cfull].detach().unsqueeze(0)
        pi = m.last_layer.weight[cfull, cfull * K:(cfull + 1) * K].detach().view(1, K, 1)
        with torch.no_grad():
            ll, log_resp = m._e_step(x, mu, sg, pi)
            pi_n, mu_n, var_n = m._m_step(x, log_resp)
            sc = m._score(x.unsqueeze(1), mu, sg, pi, as_average=False)
            elp = m._estimate_log_prob(x, mu, sg)
        rec['em_class'] = np.int64(cfull)
        rec['em_x'] = x.numpy().copy()
        rec['em_mu'] = mu.numpy().copy()
        rec['em_sigma'] = sg.numpy().copy()
        rec['em_pi'] = pi.numpy().copy()
        rec['em_loglik'] = np.float32(ll.item())
        rec['em_log_resp'] = log_resp.numpy().copy()
        rec['em_mstep_pi'] = pi_n.numpy().copy()
        rec['em_mstep_mu'] = mu_n.numpy().copy()
        rec['em_mstep_var'] = var_n.numpy().copy()
        rec['em_score'] = sc.numpy().copy()
        rec['em_est_log_prob'] = elp.numpy().copy()
        # diversified M-step gradient via the reference's own autograd graph (model.py:385-396)
        mu_p = m.prototype_means
        m.prototype_optimizer.zero_grad()
        resp = torch.exp(log_resp)
        resp = (resp + m.alpha) / (resp + m.alpha).sum(1, keepdim=True)
        llk = m._estimate_log_prob(x, mu_p[cfull].unsqueeze(0), sg) + torch.log(pi + 1e-10)
        wll = -(resp * llk).sum(1).mean(0).squeeze()
        from utils.helpers import list_of_distances
        pdist = list_of_distances(mu_p[cfull], mu_p[cfull])
        I = 1 - torch.eye(K, K)
        loss = wll + (torch.exp(-pdist) * I).sum() / I.sum()
        loss.backward()
        rec['em_div_grad'] = mu_p.grad[cfull].numpy().copy()
        rec['em_div_loss'] = np.float32(loss.item())
        rec['em_div_pi'] = ((resp.sum(0, keepdim=True) + 1e-10) / x.shape[0]).detach().numpy().copy()
    np.savez_compressed(os.path.join(OUT, name + '.npz'), **rec)
    print(name, 'written;', 'final mem_len', m.queue.mem_len.tolist(), 'adam step', float(rec['adam_step']))


if __name__ == '__main__':
    torch.set_num_threads(4)
    make_case('tiny', C=4, K=3, D=8, B=8, H=4, W=4, T=5, cap=9, iters=8,
              sigma_mode='init', pi_mode='init', seed=11, hw_stride=1)
    make_case('small_diag', C=6, K=5, D=32, B=8, H=14, W=14, T=20, cap=20, iters=5,
              sigma_mode='rand', pi_mode='rand', seed=12, hw_stride=2)
    make_case('k10d128', C=5, K=10, D=128, B=4, H=14, W=14, T=20, cap=20, iters=4,
              sigma_mode='init', pi_mode='init', seed=13, hw_stride=2)
