#!/usr/bin/env python
"""Golden outputs of the UNMODIFIED reference at the HEADLINE shapes (BASELINE.json configs[1]: 200 classes x 10
prototypes x 128-d, T = 20, 800-row banks) -> tests/golden/headline.npz.

    MGPROTO_REFERENCE=<reference checkout> python tests/golden/make_golden_headline.py          (CPU, ~2 min)

The inputs are regenerated from seeds by tests/headline_case.py (numpy) on both sides, so only the reference's
OUTPUTS are stored: logits / loss / feature gradient / top-k indices of a labelled 8-image step whose labels include
classes straddling the 128-prototype tensor-core tiles, the unlabelled logits, the newest bank rows after the enqueue,
and mu / pi / Adam moments after two update_GMM calls with >= 140 active classes each on a pre-seeded Adam state
(step 1000) -- the regime bench.py times.  The larger outputs are stored as the fixed samples headline_case.py
names, so that the file stays under 1 MB.  The tests read only the stored file, never the reference.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import headline_case as HC                                       # noqa: E402
from make_golden import ResTiny, loss_fn, ref_model              # noqa: E402  (imports the reference, CPU shim)

CFG = dict(C=200, K=10, D=128, T=20, cap=800, B=8, H=14, W=14, lr=3e-3, short_len=763)
GT_FIXED = (12, 25, 199, 0, 38, 12)          # prototypes 120..129 / 250..259 / 380..389 straddle 128-row tiles; 12 twice


def main():
    c = CFG
    C, K, D, T, cap, B, H, W = (c[k] for k in "C K D T cap B H W".split())
    torch.manual_seed(0)
    torch.set_num_threads(8)
    m = ref_model.MGProto(features=ResTiny(16), img_size=224, prototype_shape=(C * K, D, 1, 1),
                          proto_layer_rf_info=None, num_classes=C, init_weights=True,
                          prototype_activation_function='log', add_on_layers_type='regular',
                          sz_embedding=8, mem_capacity=cap, mine_K=T)
    m.train()
    mu, sg, wt = HC.mixture(C, K, D)
    m.prototype_means.data.copy_(torch.from_numpy(mu))
    m.prototype_covs.data.copy_(torch.from_numpy(sg))
    m.last_layer.weight.data.copy_(torch.from_numpy(wt))
    rows = HC.bank_rows(C, K, D, cap, mu)
    am, av, flags, short, step0 = HC.em_state(C, K, D)
    for i in range(C):
        getattr(m.queue, 'cls%d' % i).copy_(torch.from_numpy(rows[i]))
    m.queue.mem_len.fill_(cap)
    for s in short:                                               # flagged but not full: no update (model.py:289)
        m.queue.mem_len[int(s)] = c["short_len"]
        getattr(m.queue, 'cls%d' % int(s))[c["short_len"]:] = 0
    opt = torch.optim.Adam([{'params': m.prototype_means, 'lr': c["lr"]}])
    opt.state[m.prototype_means] = {'step': torch.tensor(float(step0)), 'exp_avg': torch.from_numpy(am.copy()),
                                    'exp_avg_sq': torch.from_numpy(av.copy())}
    m.prototype_optimizer = opt

    x, gt = HC.head_batch(B, C, K, D, H, W, mu, gt_fixed=GT_FIXED)
    rec = {k: np.asarray(v) for k, v in c.items()}
    rec['gt'] = gt
    img = torch.zeros(B, 3, H, W)
    emb = torch.zeros(B, 8)
    gtt = torch.from_numpy(gt)

    # unlabelled (eval / OoD) forward
    with torch.no_grad():
        m.conv_features = lambda _x: (torch.from_numpy(x), emb)
        o2, _ = m(img, None)
        rec['logits_nogt'] = o2.numpy().copy()
        feat = F.normalize(torch.from_numpy(x), p=2, dim=1).permute(0, 2, 3, 1).reshape(-1, D)
        lp = m.compute_log_prob(feat)                                       # [N,C,K]
        prob = lp.exp().reshape(B, H * W, C * K).permute(0, 2, 1)
        v, ix = torch.topk(prob, T, dim=2)
        rec['top1_idx'] = ix[:, :, 0].numpy().astype(np.int32)              # [B,P]
        rec['top1_val'] = v[:, :, 0].numpy().copy()
        rec['top2_val'] = v[:, :, 1].numpy().copy()
        own = np.stack([np.arange(int(g) * K, int(g) * K + K) for g in gt])
        rec['own_idx'] = np.stack([ix[b, own[b]].numpy() for b in range(B)]).astype(np.int32)   # [B,K,T]
        rec['own_val'] = np.stack([v[b, own[b]].numpy() for b in range(B)])
        rec['logp_rows'] = lp.reshape(-1, C * K)[HC.LOGP_ROWS].numpy().copy()

    # labelled training step: forward (+ enqueue) + backward
    x_leaf = torch.from_numpy(x.copy()).requires_grad_(True)
    m.conv_features = lambda _x: (x_leaf, emb)
    out, _ = m(img, gtt)
    loss = loss_fn(out, gtt)
    loss.backward()
    rec['logits'] = out.detach().numpy().copy()
    rec['loss'] = np.float32(loss.item())
    rec['grad_x'] = x_leaf.grad.numpy()[HC.GRAD_X].copy()
    rec['mem_len_after_enqueue'] = m.queue.mem_len.numpy().copy()
    touched = np.unique(gt)
    rec['touched'] = touched
    rec['bank_tail'] = np.stack([getattr(m.queue, 'cls%d' % int(t))[-HC.BANK_TAIL:].numpy().copy() for t in touched])
    rec['updated_after_enqueue'] = m.memory_updated_cls.numpy().copy()

    # two update_GMM calls
    for it in range(2):
        m.memory_updated_cls |= torch.from_numpy(flags[it])
        rec['flags%d' % it] = m.memory_updated_cls.numpy().copy()
        m.update_GMM()
        rec['mu_after%d' % it] = m.prototype_means.detach().numpy()[(HC.MU_AFTER0, HC.MU_AFTER1)[it]].copy()
        w = m.last_layer.weight.detach().numpy()
        rec['pi_after%d' % it] = np.stack([w[i, i * K:(i + 1) * K] for i in range(C)])
        assert int(m.memory_updated_cls.sum()) == 0
    st = opt.state[m.prototype_means]
    rec['adam_step'] = np.float32(float(st['step']))
    rec['adam_m'] = st['exp_avg'].numpy()[HC.ADAM].copy()
    rec['adam_v'] = st['exp_avg_sq'].numpy()[HC.ADAM].copy()
    np.savez_compressed(os.path.join(HERE, 'headline.npz'), **rec)
    print('headline.npz written; adam step', float(rec['adam_step']), 'loss', float(rec['loss']),
          'active', int(rec['flags0'].sum()), int(rec['flags1'].sum()))


if __name__ == '__main__':
    main()
