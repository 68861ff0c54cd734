"""Prototype projection ("push"), numeric half of the reference's push.py:82-200 (SURVEY.md section 8f-1).

For every prototype, find over the push set the image of the prototype's class whose best patch is closest
(highest p), greedily keeping images unique across prototypes (push.py:165-200), and copy that patch's normalised
feature vector into ``prototype_means``.  The reference copies the whole [B,P,H,W] distance map (401 MB at
B=256) to the host per batch and searches it with Python loops; here the per-(image, own-class prototype) argmin
runs on the device (``mgp_push_argmin``) and only [B,K] indices / values / feature rows are kept.  The image
dumping half of push.py (heat maps, bounding boxes, JPEGs) is out of scope.
"""
from __future__ import annotations

import time

import numpy as np
import torch


def _unpack(item):
    """Reference loader items are ((images, labels), (paths, labels)) (utils/helpers.py MyImageFolder);
    plain (images, labels) batches are accepted too."""
    if isinstance(item[0], (tuple, list)):
        names = item[1][0] if len(item) > 1 else None
        return item[0][0], item[0][1], names
    return item[0], item[1], None


@torch.no_grad()
def push_prototypes(dataloader, prototype_network_parallel, class_specific=True, preprocess_input_function=None,
                    prototype_layer_stride=1, root_dir_for_saving_prototypes=None, epoch_number=None,
                    prototype_img_filename_prefix=None, prototype_self_act_filename_prefix=None,
                    proto_bound_boxes_filename_prefix=None, save_prototype_class_identity=True, log=print,
                    prototype_activation_function_in_numpy=None):
    """Same signature as the reference's push_prototypes (push.py:14-26); returns a dict with, per prototype,
    the chosen global image index (-1: unchanged), the flat patch index and the distance -p."""
    net = getattr(prototype_network_parallel, "module", prototype_network_parallel)
    net.eval()
    log("\tpush")
    start = time.time()
    C, K = net.num_classes, net.num_prototypes_per_class
    dev = net.prototype_means.device
    vals, args, feats, labels = [], [], [], []
    for item in dataloader:
        x, y, _ = _unpack(item)
        if preprocess_input_function is not None:
            x = preprocess_input_function(x)
        x = x.to(dev)
        y = torch.as_tensor(y).to(dev).long()
        x_add, _ = net.conv_features(x)                                        # push.py:107 (push_forward)
        arg, val, xhat = net.push_search(x_add, y)                             # push.py:125-158 on the device
        hw = x_add.shape[2] * x_add.shape[3]
        rows = (torch.arange(x.shape[0], device=dev)[:, None] * hw + arg.long())          # [B,K] rows of xhat
        vals.append(val.cpu())
        args.append(arg.cpu())
        feats.append(xhat[rows.reshape(-1)].view(x.shape[0], K, -1).cpu())
        labels.append(y.cpu())
    val = torch.cat(vals).numpy()
    arg = torch.cat(args).numpy()
    feat = torch.cat(feats)
    lab = torch.cat(labels).numpy()

    log("\tExecuting push ...")
    chosen_img = np.full(C * K, -1, np.int64)
    chosen_patch = np.full(C * K, -1, np.int64)
    chosen_dist = np.full(C * K, np.inf, np.float32)
    used = set()                                                               # has_pushed_img, push.py:165
    by_class = {c: np.nonzero(lab == c)[0] for c in range(C)}
    for j in range(C * K):                                                     # push.py:166-200
        c, k = divmod(j, K)
        cand = by_class[c]
        if cand.size == 0:
            continue
        for i in cand[np.argsort(val[cand, k])]:                               # most negative -p first
            if int(i) in used:
                continue
            net.prototype_means.data[c, k].copy_(feat[i, k].to(dev))           # push.py:197-198
            used.add(int(i))
            chosen_img[j], chosen_patch[j], chosen_dist[j] = i, arg[i, k], val[i, k]
            break
    if (chosen_img >= 0).any():
        torch.autograd.graph.increment_version(net.prototype_means)          # the `.data` writes above bump nothing
    log("\tpush time: \t{0}".format(time.time() - start))
    return {"image": chosen_img, "patch": chosen_patch, "distance": chosen_dist}
