#!/usr/bin/env python
"""bench.py -- throughput of the MGProto Gaussian-prototype hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1)
    python bench.py --impl reference ...                     (CPU arm: the reference algorithm on host cores)
    python bench.py ... --dump-outputs DIR                   (also write the last timed step's outputs as DIR/*.npy)

Workload (BASELINE.json configs[1], named in config.workload): per GPU a batch of 256 images'
add-on feature maps [256,128,14,14] against a 200-class x 10-prototype x 128-d diagonal-Gaussian
mixture, T=20 mining levels, a full 800-row/class memory bank.  One *step* is one pass of the
training hot path over one batch: normalise -> log-likelihood -> top-T mining -> pi-mix logits
-> loss -> backward to the features -> bank enqueue -> update_GMM (3 EM loops, sequential Adam).
The backbone is outside the path (SURVEY.md section 8) and is not timed.

  value   images/s, whole job, inputs resident in HBM
  e2e     images/s through MGProto.head()/update_GMM() with HOST (pinned) feature batches: every step's H2D of
          its features and D2H of its logits are inside the timed region, double-buffered on copy streams
          (mgproto_b200.pipeline) so that they overlap the neighbouring steps' compute
  roofline  the log-likelihood kernel (mgp_logprob_fwd, [N,P] output: the north-star kernel), timed
          alone with CUDA events: algorithmic bytes 4*(N*D + 2*P*D + N*P) per launch / duration,
          against MEASURED_PEAKS.json's HBM copy bandwidth (burst figure: kernel timed alone);
          roofline_step_logprob: the variant the labelled step runs (max/arg-max epilogue, log p stays on
          chip) against the measured dense bf16 tensor peak
  cpu_baseline  the UNMODIFIED reference (baseline/_ref, tools/install_reference.py) on the host cores, bounded
          sample; the numpy oracle port only if baseline/_ref is absent
  reference_gpu_eager  the same-box GPU bar: the unmodified reference model.py run eagerly on cuda:0 at the same
          shapes (no_grad forward, train forward+backward, update_GMM), timed beside our stages

Timing: exactly --steps timed steps after the warm-up, between two CUDA events (none between the steps, which would
add their own gaps); `value` is the images of those steps over that window.  The end-to-end leg is timed the same way.

--dump-outputs DIR writes what the last timed step returned to its caller -- logits [B,C,T], loss, the feature gradient
[B,D,H,W] -- and the mixture it left behind (means [C,K,D], weights [C,C*K]) as float32 DIR/<name>.npy (32 MB; rank 0).
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: bench.py writes nothing into it

CFG = dict(B=256, C=200, K=10, D=128, H=14, W=14, T=20, cap=800)
N_ROT = 8   # distinct input batches rotated through (8 x 25.7 MB of features > the 126 MB L2)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


# ------------------------------------------------------------------------------------------ CPU arm
def _cpu_threads():
    return max(1, min(os.cpu_count() or 1, 32))


def cpu_reference_step(n_img, seed=0, with_em=True, threads=1):
    """One bounded-sample step of the reference algorithm (numpy oracle port) -> seconds.  The per-image head
    (log-likelihood, top-T, logits) is spread over `threads` host threads (numpy releases the GIL); enqueue
    and update_GMM are the reference's sequential per-class loops."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from oracle import mgproto_oracle as O
    c = CFG
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n_img, c["D"], c["H"], c["W"])).astype(np.float32)
    mu = O.l2_normalize(rng.random((c["C"], c["K"], c["D"])).astype(np.float32), axis=2)
    sg = np.full_like(mu, 1 / np.sqrt(2 * np.pi))
    wt = np.zeros((c["C"], c["C"] * c["K"]), np.float32)
    for i in range(c["C"]):
        wt[i, i * c["K"]:(i + 1) * c["K"]] = 1.0 / c["K"]
    gt = rng.integers(0, c["C"], size=(n_img,))
    bank = O.MemoryBankOracle(c["C"], c["D"], c["cap"])
    for cc in np.unique(gt):
        bank.data[cc] = O.l2_normalize(mu[cc][rng.integers(0, c["K"], c["cap"])] +
                                       0.3 * rng.standard_normal((c["cap"], c["D"])).astype(np.float32), axis=1)
        bank.mem_len[cc] = c["cap"]
    t0 = time.perf_counter()
    chunks = [list(range(i, n_img, threads)) for i in range(min(threads, n_img))]

    def work(ids):
        return ids, O.head_forward(x[ids], mu, sg, wt, gt[ids], c["T"])
    if threads > 1:
        with ThreadPoolExecutor(threads) as ex:
            parts = list(ex.map(work, chunks))
    else:
        parts = [work(ch) for ch in chunks]
    hw = c["H"] * c["W"]
    xhat = np.empty((n_img * hw, c["D"]), np.float32)
    idx = np.empty((n_img, c["C"] * c["K"], c["T"]), np.int64)
    for ids, fw in parts:
        for j, i in enumerate(ids):
            xhat[i * hw:(i + 1) * hw] = fw["xhat"][j * hw:(j + 1) * hw]
            idx[i] = fw["idx"][j]
    rows = O.enqueue_rows(xhat, idx, gt, c["C"], c["K"], hw)
    if with_em:
        upd = np.zeros(c["C"], bool)
        for cc, r in rows:
            bank.push(cc, r)
            upd[cc] = True
        adam = O.AdamOracle(mu.shape, lr=3e-3, dtype=np.float32)
        O.update_gmm(bank, upd, mu, sg, wt, adam)
    return time.perf_counter() - t0



# ------------------------------------------------------------------------------------------ the real reference
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def reference_available():
    return os.path.exists(os.path.join(REF_DIR, "model.py"))


def _import_reference(cpu):
    """Import the unmodified reference model.py from baseline/_ref.  On the CPU arm `Tensor.cuda` becomes a no-op
    (model.py:391 hard-codes .cuda()); no reference file is touched."""
    import importlib
    import torch
    if cpu:
        torch.Tensor.cuda = lambda self, *a, **k: self
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    return importlib.import_module("model")


def synthetic_state(seed_mu=2, seed_bank=6):
    """mu [C,K,D] and full bank rows [C,cap,D] (SURVEY 8d), shared by our model and the reference legs."""
    import torch
    import torch.nn.functional as F
    c = CFG
    mu = F.normalize(torch.rand(c["C"], c["K"], c["D"], generator=torch.Generator().manual_seed(seed_mu)), p=2, dim=2)
    g6 = torch.Generator().manual_seed(seed_bank)
    kk = torch.randint(0, c["K"], (c["C"], c["cap"]), generator=g6)
    rows = mu[torch.arange(c["C"])[:, None], kk] + 0.3 * torch.randn(c["C"], c["cap"], c["D"], generator=g6)
    return mu, F.normalize(rows, p=2, dim=2)


def build_reference_model(ref, dev):
    """The reference's MGProto (its own constructor) with the same synthetic mixture / full bank as build_model."""
    import torch
    import torch.nn as nn
    c = CFG

    class RESStub(nn.Module):                      # model.py:107-115 wants a backbone whose repr starts with "RES"
        def __init__(self):
            super().__init__()
            self.conv = nn.Conv2d(3, 16, kernel_size=1)

        def forward(self, x):
            return self.conv(x)

    m = ref.MGProto(features=RESStub(), img_size=224, prototype_shape=(c["C"] * c["K"], c["D"], 1, 1),
                    proto_layer_rf_info=None, num_classes=c["C"], init_weights=True,
                    prototype_activation_function="log", add_on_layers_type="regular", sz_embedding=32,
                    mem_capacity=c["cap"], mine_K=c["T"])
    mu, rows = synthetic_state()
    m.prototype_means.data.copy_(mu)
    for i in range(c["C"]):
        getattr(m.queue, "cls%d" % i).copy_(rows[i])
    m.queue.mem_len.fill_(c["cap"])
    m = m.to(dev)
    m.prototype_optimizer = torch.optim.Adam([{"params": m.prototype_means, "lr": 3e-3}])
    m.train()
    return m


def reference_step(m, x_add, gt, with_em=True):
    """One hot-path step through the reference's own methods: forward (from the add-on features on: the backbone is
    outside the path, so conv_features is pointed at the precomputed feature batch), the training loss of
    train_and_test.py:37-45, backward to the features, update_GMM (train_and_test.py:61-63)."""
    import torch
    import torch.nn.functional as F
    x_leaf = x_add.detach().clone().requires_grad_(True)
    emb = torch.zeros(x_add.shape[0], 32, device=x_add.device)
    m.conv_features = lambda _x: (x_leaf, emb)
    out, _ = m(None, gt)
    mine = sum(F.cross_entropy(out[:, :, k], gt) for k in range(1, out.shape[2])) / (out.shape[2] - 1)
    loss = F.cross_entropy(out[:, :, 0], gt) + 0.2 * mine
    loss.backward()
    if with_em and m.queue.mem_len.sum() > 0:
        m.update_GMM()
    return out


def cpu_reference_real(n_img, steps, warmup, threads):
    """The unmodified reference on the host cores: `steps` timed steps of `n_img` images each -> mean seconds/step."""
    import torch
    torch.set_num_threads(threads)
    ref = _import_reference(cpu=True)
    m = build_reference_model(ref, torch.device("cpu"))
    c = CFG
    gen = torch.Generator().manual_seed(1)
    ts = []
    for i in range(warmup + steps):
        x = torch.randn(n_img, c["D"], c["H"], c["W"], generator=gen)
        gt = torch.randint(0, c["C"], (n_img,), generator=gen)
        t0 = time.perf_counter()
        reference_step(m, x, gt)
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
        elif dt > 40.0:                       # a slow host: the warm-up step is the sample (keeps the run bounded)
            return dt
    return statistics.mean(ts)


def reference_gpu_eager(dev, feats, gts, ours):
    """SURVEY 2b / 8(d): the same-box GPU bar -- the unmodified reference run eagerly on the B200 at the bench
    shapes, stage by stage, beside our own stages (`ours`: dict of callables).  CUDA events, 1 warm-up + 3 timed."""
    import torch
    ref = _import_reference(cpu=False)
    m = build_reference_model(ref, dev)
    c = CFG
    res = {"what": "unmodified reference model.py (baseline/_ref) on cuda:0, eager ATen/cuBLAS kernels, same synthetic "
                   "mixture, bank and feature batches; conv_features points at the precomputed add-on features"}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, n=3, warm=1):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(n):
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    emb = torch.zeros(c["B"], 32, device=dev)
    x, gt = feats[0], gts[0]

    def ref_fwd_nograd():
        with torch.no_grad():
            m.conv_features = lambda _x: (x, emb)
            m(None, None)

    def ref_train():
        reference_step(m, x, gt, with_em=False)

    def ref_em():
        m.memory_updated_cls[:] = False
        m.memory_updated_cls[torch.unique(gt).cpu()] = True
        m.update_GMM()

    stages = (("forward_nograd", ref_fwd_nograd), ("train_fwd_bwd_enqueue", ref_train), ("update_GMM", ref_em))
    for name, fn in stages:
        try:
            t_ref = timed(fn)
            t_ours = timed(ours[name], n=10, warm=2)
            res[name] = {"reference_ms": t_ref, "ours_ms": t_ours, "speedup": t_ref / t_ours}
        except Exception as ex:  # noqa: BLE001 -- e.g. out of memory in the reference's [N/4,P,D] temporaries
            res[name] = {"error": str(ex)[:160]}
            torch.cuda.empty_cache()
    res["active_classes_update_GMM"] = int(torch.unique(gt).numel())
    del m
    torch.cuda.empty_cache()
    return res

def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    th = _cpu_threads()
    c = CFG
    if reference_available():
        # the unmodified reference (torch CPU, all host threads): 8 images per step keeps a step at ~10-20 s
        # (torch's CPU kernels stop scaling -- and at 128 threads get 10x slower -- on these small ATen ops: 16 threads)
        th = min(os.cpu_count() or 1, 16)
        n_img, steps = 8, max(1, min(args.steps, 2))
        t = cpu_reference_real(n_img, steps, warmup=1, threads=th)
        kind = "reference"
        sample = ("%d images of the 256-image batch per step x %d steps, full 200x10x128 mixture and 800-row banks: "
                  "unmodified reference model.py (baseline/_ref) forward from the add-on features + loss + backward + "
                  "enqueue + update_GMM of the touched classes, torch CPU on %d threads" % (n_img, steps, th))
    else:
        n_img = max(2, th)
        for _ in range(max(1, min(args.warmup, 1))):
            cpu_reference_step(n_img, threads=th)
        ts = [cpu_reference_step(n_img, seed=s, threads=th) for s in range(max(1, min(args.steps, 5)))]
        t, steps, kind = statistics.mean(ts), len(ts), "port"
        sample = ("%d images of the 256-image batch per step, full 200x10x128 mixture, forward + enqueue + update_GMM of "
                  "the touched classes; numpy oracle port, head on %d threads (baseline/_ref absent)" % (n_img, th))
    val = n_img / t
    line = {
        "impl": "reference", "metric": "images/sec", "value": val, "unit": "images/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": 1, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args.gpus),
        "pairs_per_sec": val * c["H"] * c["W"] * c["C"] * c["K"],
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": th, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def _config(n_gpus):
    c = CFG
    par = "single GPU" if n_gpus == 1 else ("dp%d: images sharded, prototypes/bank replicated; one all-gather of the mined "
                                            "rows per step, update_GMM replicated on every rank (no EM collective)" % n_gpus)
    return {"workload": "head-only, pre-computed add-on features (backbone outside the path): BASELINE.json configs[1] "
                        "shapes, batch %d/GPU feature maps [%d,%d,%d,%d], %dx%dx%d diag-Gaussian mixture, T=%d, bank %d "
                        "rows/class; step = head fwd+bwd + enqueue + update_GMM"
                        % (c["B"], c["B"], c["D"], c["H"], c["W"], c["C"], c["K"], c["D"], c["T"], c["cap"]),
            "global_batch": c["B"] * n_gpus, "parallelism": par,
            "l2": "inputs rotate through %d distinct batches (%.0f MB) > 126 MB L2; the labelled step keeps log p on chip (no [B,P,HW] intermediate)"
                  % (N_ROT, N_ROT * c["B"] * c["D"] * c["H"] * c["W"] * 4 / 1e6)}


# ------------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [f.strip() for f in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """Samples inside the timed window [t0, t1]; a window shorter than a few sampling periods falls back to
        every sample taken under load (warm-up + timed + end-to-end loops run the same step back to back)."""
        if self.proc is not None:
            self.proc.terminate()
        ok = [(t, r) for t, r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        inside = [r for t, r in ok if t0 is not None and t0 <= t <= t1]
        window = "timed"
        if len(inside) < 3:
            inside, window = [r for _, r in ok], "warmup+timed+e2e (timed region shorter than 3 samples)"
        sm = [float(r[0]) for r in inside]
        mx = [float(r[1]) for r in inside if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in inside)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "window": window}


def build_model(dev, seed=0):
    import torch
    import torch.nn as nn
    import mgproto_b200 as M
    c = CFG
    g = torch.Generator().manual_seed(seed)
    net = M.MGProto(features=nn.Sequential(nn.Conv2d(3, 8, 1)), img_size=224, prototype_shape=(c["C"] * c["K"], c["D"], 1, 1),
                    proto_layer_rf_info=None, num_classes=c["C"], add_on_layers_type="regular", sz_embedding=32,
                    mem_capacity=c["cap"], mine_K=c["T"])
    mu, rows = synthetic_state()
    net.prototype_means.data.copy_(mu)
    net = net.to(dev)
    net.queue.bank.copy_(rows.to(dev))                    # every class's bank full (SURVEY 8d)
    net.queue.mem_len.fill_(c["cap"])
    net.prototype_optimizer = torch.optim.Adam([{"params": net.prototype_means, "lr": 3e-3}])
    net.train()
    return net


def dump_outputs(path, arrays):
    """Write each tensor as float32 path/<name>.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def loss_fn(out, gt):
    """CE on level 0 + 0.2 * mean CE over the mining levels (ref train_and_test.py:37-41, :55) -- the library's
    fused value+gradient helper (one launch instead of the ~25 ATen launches of T separate cross_entropy calls)."""
    from mgproto_b200 import ops
    return ops.mine_cross_entropy(out, gt, 0.2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--math", default="auto", choices=["auto", "fp32", "tc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference_gpu_eager leg")
    ap.add_argument("--no-ood", action="store_true", help="skip the configs[4] OoD-scoring throughput leg")
    ap.add_argument("--no-graph", action="store_true", help="run the device-resident leg eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/nccl_bench_%h_%p.log")   # (NCCL prints its version banner on stdout)
        dist.init_process_group("nccl", device_id=dev)
    from mgproto_b200 import ops, parallel
    c = CFG
    W = max(3, args.warmup)
    net = build_model(dev)
    net.math_mode = args.math
    if world > 1:
        parallel.attach(net)
    B, D, H, Wd, HW = c["B"], c["D"], c["H"], c["W"], c["H"] * c["W"]
    gen = torch.Generator().manual_seed(1 + rank)
    feats_host = [torch.randn(B, D, H, Wd, generator=gen).pin_memory() for _ in range(N_ROT)]
    gts = [torch.randint(0, c["C"], (B,), generator=gen).to(dev) for _ in range(N_ROT)]
    feats = [f.to(dev) for f in feats_host]

    def step(x, gt):
        x.grad = None
        x.requires_grad_(True)
        out = net.head(x, gt)
        loss = loss_fn(out, gt)
        loss.backward()
        net.update_GMM()
        return out, loss, x.grad

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The device-resident leg replays the step from a CUDA graph (mgproto_b200.pipeline.GraphedStep): same kernels, same
    # work, one cudaGraphLaunch + two small input copies per step on the host.  --no-graph (or a failed capture) runs
    # the eager step; the e2e leg below always runs eager (its inputs arrive in rotating device buffers).
    launch_mode = "eager"
    graphed = None
    if not args.no_graph:
        try:
            from mgproto_b200.pipeline import GraphedStep
            graphed = GraphedStep(net, loss_fn, feats[0], gts[0], warmup=3)
            launch_mode = "cuda_graph"
        except Exception as exc:                                  # noqa: BLE001 -- report and fall back
            if rank == 0:
                print("bench: CUDA-graph capture failed (%s: %s); eager step" % (type(exc).__name__, exc), file=sys.stderr)
            graphed = None
            torch.cuda.synchronize()
    eager_step = step
    if graphed is not None:
        def step(x, gt):                                          # noqa: F811
            return graphed(x, gt) + (graphed.x_grad,)

    # ---- device-resident throughput -------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(W):
        step(feats[i % N_ROT], gts[i % N_ROT])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_w0 = time.time()
    l0 = ops.launch_count()
    e0.record()
    t_h0 = time.perf_counter()
    for i in range(args.steps):
        last = step(feats[i % N_ROT], gts[i % N_ROT])
    e1.record()
    host_enq = (time.perf_counter() - t_h0) * 1e3                 # host time to ENQUEUE the steps (no sync inside)
    barrier()
    t_w1 = time.time()
    launches = ops.launch_count() - l0
    if graphed is not None:                          # replays do not pass through the Python launch counter
        launches = graphed.launches * args.steps
    tm = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    window_ms = float(tm)
    ms = window_ms / args.steps
    value = B * world * args.steps / (window_ms / 1e3)
    timing = {"steps": args.steps, "window_ms": window_ms,
              "value_from": "one window of %d timed steps between two CUDA events, max over ranks" % args.steps,
              "launch": launch_mode,
              "host_enqueue_ms": host_enq,
              "host_note": "wall time the Python / ctypes side needs to enqueue the timed steps (no synchronisation inside): "
                           "the step is GPU-bound while this stays below window_ms"}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"logits": last[0], "loss": last[1], "x_grad": last[2],
                                         "prototype_means": net.prototype_means, "mixture_weights": net.last_layer.weight})

    # ---- end to end: host buffers in, logits out ---------------------------------------------
    # every step copies its own pinned-host feature batch to the device and reads its logits back to pinned host
    # memory; mgproto_b200.pipeline double-buffers both so the copies of neighbouring steps overlap the compute
    from mgproto_b200.pipeline import HostFeeder, HostSink
    feeder = HostFeeder((B, D, H, Wd), dev, depth=2)
    sink = HostSink((B, c["C"], c["T"]), depth=2, device=dev)

    def e2e_run(n):
        feeder.stage(feats_host[0])
        for i in range(n):
            if i + 1 < n:
                feeder.stage(feats_host[(i + 1) % N_ROT])
            x_dev = feeder.acquire()
            out = eager_step(x_dev, gts[i % N_ROT])[0]
            sink.put(out.detach())
            feeder.release(x_dev)
        sink.wait()

    e2e_run(W)
    barrier()
    e0.record()
    e2e_run(args.steps)
    e1.record()
    barrier()
    tm = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    e2e_val = B * world * args.steps / (float(tm) / 1e3)
    timing["e2e_window_ms"] = float(tm)
    clocks = sampler.stop(t_w0, t_w1) if rank == 0 else None

    # ---- roofline of the log-likelihood kernel (timed alone, rank 0) --------------------------
    roof = None
    extra = {}
    if rank == 0:
        peak, how = peaks()
        P, N = c["C"] * c["K"], B * HW
        mu = net.prototype_means.detach().reshape(P, D).contiguous()
        sg = net.prototype_covs.detach().reshape(P, D).contiguous()
        xs = [ops.normalize_fwd(f)[0] for f in feats[:6]]                     # 6 x 25.7 MB inputs rotate
        outs = [torch.empty(N, P, device=dev) for _ in range(2)]               # 2 x 401 MB outputs alternate
        for i in range(3):
            ops.logprob(xs[i % 6], mu, sg, 0, math=args.math, out=outs[i % 2])
        torch.cuda.synchronize()
        reps = 20
        e0.record()
        for i in range(reps):
            ops.logprob(xs[i % 6], mu, sg, 0, math=args.math, out=outs[i % 2])
        e1.record()
        torch.cuda.synchronize()
        t_op = e0.elapsed_time(e1) / reps / 1e3
        abytes = 4.0 * (N * D + 2 * P * D + N * P)
        # `roofline` describes mgp_logprob_fwd AS CALLED by compute_log_prob (prototype operand pre-pass + the GEMM
        # kernel; with isotropic sigma the x operand split is fused into the kernel: csrc/logprob_tcz.cu); the kernel
        # alone (prototype operands pre-staged) is an extra key
        from mgproto_b200 import _lib
        iso = ops.sigma_is_isotropic(sg)
        kname = "mgp_logprob_fwd [N,P] as called (math=%s): %s" % (
            args.math, "tc_proto_prep + logprob_z_kernel (TMEM-resident patch tile, fused fp16 hi/lo split, TMA-store epilogue)"
            if (iso and args.math == "auto") else "operand pre-passes + logprob kernel")
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("logprob_dram_bytes_per_launch")
        roof = {"kernel": kname, "bound": "hbm", "achieved": abytes / t_op / 1e9,
                "peak": peak, "unit": "GB/s", "frac": abytes / t_op / 1e9 / peak, "traffic": traffic,
                "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs, burst: op timed alone)",
                "us_per_launch": t_op * 1e6, "algorithmic_bytes": abytes,
                "pairs_per_sec": N * P / t_op, "tensor_tflops_equiv": 4.0 * N * P * D / t_op / 1e12,
                "note": "north-star kernel K-A (compute_log_prob / eval / push: log p materialised), the whole op as the "
                        "API calls it, 6 x 25.7 MB inputs and 2 x 401 MB outputs rotating; the [N,P] TMA-store stream "
                        "alone tops out at 5.1-5.5 TB/s on this part (profiles/r2_tma_store_bw.txt); the labelled training "
                        "step runs the max/arg-max variant instead (roofline_step_logprob)"}
        if args.math != "fp32" and _lib.load().mgp_has_tensor_core_path():
            mode_full, mode_reuse = ("tc_iso", "tc_iso_reuse") if iso and D in (64, 128, 256) else ("tc", "tc_reuse")
            wss = [ops.logprob(xs[i], mu, sg, 0, math=mode_full, out=outs[0], return_ws=True)[1] for i in range(6)]
            torch.cuda.synchronize()
            e0.record()
            for i in range(reps):
                ops.logprob(xs[i % 6], mu, sg, 0, math=mode_reuse, ws=wss[i % 6], out=outs[i % 2])
            e1.record()
            torch.cuda.synchronize()
            t_ka = e0.elapsed_time(e1) / reps / 1e3
            extra["roofline_logprob_kernel"] = {
                "kernel": "the GEMM kernel alone (prototype operands pre-staged)", "bound": "hbm",
                "achieved": abytes / t_ka / 1e9, "peak": peak, "unit": "GB/s", "frac": abytes / t_ka / 1e9 / peak,
                "us_per_launch": t_ka * 1e6}
        del outs
        # the variant the labelled step runs: same GEMM, max/arg-max epilogue, no log p output -> tensor-bound
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops") if \
            os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else None
        tpk, tsrc = (pk, "MEASURED_PEAKS.json bf16_tflops (burst)") if pk else (2250.0, "nominal dense bf16 (B200_PROFILING.md fallback)")
        if args.math != "fp32" and _lib.load().mgp_has_tensor_core_path():
            w1 = [ops.logprob_top1(xs[i], mu, sg, B, HW, "tc", return_ws=True)[1] for i in range(6)]
            torch.cuda.synchronize()
            e0.record()
            for i in range(reps):
                ops.logprob_top1(xs[i % 6], mu, sg, B, HW, "tc_reuse", ws=w1[i % 6])
            e1.record()
            torch.cuda.synchronize()
            t_t1 = e0.elapsed_time(e1) / reps / 1e3
            fl = 3 * 2.0 * N * P * D                                  # three fp16 passes of the K = D GEMM (isotropic sigma)
            extra["roofline_step_logprob"] = {
                "kernel": "logprob_tc_kernel<top1> (in-step variant: 4 MB memset + GEMM with max/arg-max epilogue, no [N,P] store)",
                "bound": "tensor", "achieved": fl / t_t1 / 1e12, "peak": tpk, "unit": "TFLOP/s",
                "frac": fl / t_t1 / 1e12 / tpk, "peak_source": tsrc, "us_per_launch": t_t1 * 1e6,
                "pairs_per_sec": N * P / t_t1, "algorithmic_GBps_equiv": abytes / t_t1 / 1e9,
                # SURVEY 8(d) K-B (fused head, no [N,P] in HBM): its algorithmic bytes and the sustained tensor figure
                "kb_algorithmic_bytes": 4.0 * N * D + 8.0 * P * D + 8.0 * B * P * c["T"] + 4.0 * B * c["C"] * c["T"]
                                        + 4.0 * B * c["K"] * D,
                "kb_GBps": (4.0 * N * D + 8.0 * P * D + 8.0 * B * P * c["T"] + 4.0 * B * c["C"] * c["T"]
                            + 4.0 * B * c["K"] * D) / t_t1 / 1e9,
                "frac_of_sustained_bf16": fl / t_t1 / 1e12 / 1431.0}
            del w1
        # EM statistics kernel, same treatment (second kernel the north star names)
        order = torch.arange(c["C"], dtype=torch.int32, device=dev)
        stats = torch.empty(c["C"], net.em_n_split, ops.em_stat_stride(c["K"], D), device=dev)
        wt = net.last_layer.weight.data
        for _ in range(3):
            ops.em_stats(net.queue.bank, order, net.prototype_means.data, net.prototype_covs.data, wt, 0.1, stats,
                         net.em_n_split)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            ops.em_stats(net.queue.bank, order, net.prototype_means.data, net.prototype_covs.data, wt, 0.1, stats,
                         net.em_n_split)
        e1.record()
        torch.cuda.synchronize()
        t_em = e0.elapsed_time(e1) / reps / 1e3
        eb = 4.0 * c["C"] * c["cap"] * D
        extra["roofline_em_stats"] = {"kernel": "mgp_em_stats (200 classes x 800 rows)", "bound": "hbm",
                                      "achieved": eb / t_em / 1e9, "peak": peak, "unit": "GB/s",
                                      "frac": eb / t_em / 1e9 / peak, "us_per_launch": t_em * 1e6,
                                      "note": "bank (82 MB) fits in L2 across repeats: upper-bound figure"}
        # the largest kernel of the step: the whole update_GMM (em_plan + one cluster launch), all classes active
        try:
            Lp = int(getattr(net, "num_em_loop", 3))
            for _ in range(3):
                net.queue.updated.fill_(1)
                net.update_GMM()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                net.queue.updated.fill_(1)
                net.update_GMM()
            e1.record()
            torch.cuda.synchronize()
            t_ug = e0.elapsed_time(e1) / reps / 1e3
            ub = Lp * eb
            # ... and with the classes one 256-image batch touches (what the timed step runs: <= #SMs active classes
            # take the software-pipelined kernel, more take the serial one)
            flags = torch.zeros_like(net.queue.updated)
            flags[torch.unique(gts[0])] = 1
            n_batch_active = int(flags.sum())
            for _ in range(3):
                net.queue.updated.copy_(flags)
                net.update_GMM()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                net.queue.updated.copy_(flags)
                net.update_GMM()
            e1.record()
            torch.cuda.synchronize()
            t_ub = e0.elapsed_time(e1) / reps / 1e3
            extra["roofline_step_update_gmm"] = {
                "kernel": "update_GMM = em_plan + em_tc_kernel (tcgen05; 200 active classes, %d EM loops; + one fill)" % Lp,
                "bound": "hbm", "achieved": ub / t_ug / 1e9, "peak": peak, "unit": "GB/s", "frac": ub / t_ug / 1e9 / peak,
                "us_per_call": t_ug * 1e6, "algorithmic_bytes": ub,
                "batch_active_classes": n_batch_active, "us_per_call_batch_active": t_ub * 1e6,
                "frac_batch_active": ub * n_batch_active / float(flags.numel()) / t_ub / 1e9 / peak,
                "note": "latency-bound chain per class (DESIGN.md 5.3): one CTA per class, 7 row tiles x 3 loops; the bank's "
                        "fp16 hi/lo shadow (same bytes as the fp32 bank) is re-read per EM loop, L2-resident after the first"}
        except Exception as ex:  # noqa: BLE001 -- an auxiliary figure must never cost the bench line
            extra["roofline_step_update_gmm"] = {"error": str(ex)[:200]}

    # ---- BASELINE.json configs[4]: OoD log-likelihood scoring, 50k in-distribution + 50k OoD synthetic images ----
    if rank == 0 and not args.no_ood:
        try:
            from mgproto_b200.ood import OoDScorer
            n_each, bs = 50000, 500
            g5 = torch.Generator(device=dev).manual_seed(5)
            protos = net.prototype_means.detach().reshape(-1, D)

            def batch_in():
                pick = torch.randint(0, protos.shape[0], (bs, HW), device=dev, generator=g5)
                v = protos[pick] + 0.1 * torch.randn(bs, HW, D, device=dev, generator=g5)
                return v.permute(0, 2, 1).reshape(bs, D, H, Wd).contiguous()

            def batch_out():
                return torch.randn(bs, D, H, Wd, device=dev, generator=g5)

            pool_in = [batch_in() for _ in range(4)]               # 4 x 49 MB of each kind rotate (> L2 together)
            pool_out = [batch_out() for _ in range(4)]
            sc = OoDScorer(net)
            sc.add_in_distribution(pool_in[0])
            sc.add_out_of_distribution(pool_out[0])
            sc = OoDScorer(net)
            torch.cuda.synchronize()
            e0.record()
            for i in range(n_each // bs):
                sc.add_in_distribution(pool_in[i % 4])
                sc.add_out_of_distribution(pool_out[i % 4])
            res = sc.results()
            e1.record()
            torch.cuda.synchronize()
            t_ood = e0.elapsed_time(e1) / 1e3
            extra["ood_scoring"] = {
                "workload": "BASELINE.json configs[4]: 50k in-distribution (random prototype + 0.1 randn per patch) + 50k OoD "
                            "(random) synthetic feature maps, batches of %d: head_level0 + mgp_ood_score per batch, 5th-percentile "
                            "threshold / FPR95 / AUROC on the device (mgproto_b200.ood.OoDScorer)" % bs,
                "images_per_s": 2 * n_each / t_ood, "seconds": t_ood, "AUROC": res["AUROC"], "FPR95": res["FPR95"],
                "threshold": res["threshold"],
                "parity": "scores / threshold / FPR95 / AUROC against the oracle, numpy.percentile and sklearn at n = 384 + 384: "
                          "tests/test_gpu_parity.py::test_ood_scorer_device_side_vs_oracle_and_sklearn"}
        except Exception as ex:  # noqa: BLE001
            extra["ood_scoring"] = {"error": str(ex)[:200]}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        if reference_available():
            # the unmodified reference on the host cores, in a child process without GPUs (its `.cuda()` shim and
            # its thread pool stay out of this one)
            env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
            for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS"):
                env.pop(k, None)
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                    "--warmup", "1"], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                   timeout=600)
                cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception as ex:  # noqa: BLE001
                cpu = {"error": str(ex)[:200]}
        if cpu is None or "error" in cpu:
            th = _cpu_threads()
            n_img = max(2, th)
            cpu_reference_step(n_img, threads=th)
            ts = [cpu_reference_step(n_img, seed=s, threads=th) for s in range(3)]
            cpu = {"value": n_img / statistics.mean(ts), "unit": "images/s", "cores": th, "kind": "port",
                   "sample": "%d images/step x 3 steps of the same workload (forward + enqueue + update_GMM of the touched "
                             "classes), numpy oracle port of the reference algorithm, head on %d threads" % (n_img, th)}

    # ---- the same-box GPU bar: the unmodified reference, eager, on this GPU (rank 0, N = 1) -----------------
    if rank == 0 and world == 1 and not args.no_ref_gpu and reference_available():
        try:
            def ours_fwd():
                with torch.no_grad():
                    net.head(feats[0], None)

            def ours_train():
                x = feats[0]
                x.grad = None
                x.requires_grad_(True)
                out = net.head(x, gts[0])
                loss_fn(out, gts[0]).backward()
                x.requires_grad_(False)

            def ours_em():
                net.queue.updated.zero_()
                net.queue.updated[torch.unique(gts[0])] = 1
                net.update_GMM()

            extra["reference_gpu_eager"] = reference_gpu_eager(
                dev, feats, gts, {"forward_nograd": ours_fwd, "train_fwd_bwd_enqueue": ours_train, "update_GMM": ours_em})
        except Exception as ex:  # noqa: BLE001
            extra["reference_gpu_eager"] = {"error": str(ex)[:200]}

    if rank == 0:
        line = {
            "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": _config(world),
            "pairs_per_sec": value * HW * c["C"] * c["K"],
            "e2e": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": B * D * HW * 4,
                    "d2h_bytes_per_step": B * c["C"] * c["T"] * 4},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "math": args.math, "timing": timing,
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        # NCCL communicators must outlive every CUDA graph that captured their kernels: drop the graph first; and a rank
        # that is done (ranks > 0 skip the single-GPU legs) must never be able to hang the launcher -- the teardown runs
        # in a thread and the process leaves with os._exit whatever it does
        import threading
        sys.stdout.flush()
        sys.stderr.flush()
        if graphed is not None:
            try:
                graphed.close()
            except Exception:                                     # noqa: BLE001
                pass
        graphed = None
        torch.cuda.synchronize()

        def _teardown():
            try:
                dist.destroy_process_group()
            except Exception:                                     # noqa: BLE001
                pass

        th = threading.Thread(target=_teardown, daemon=True)
        th.start()
        th.join(20.0)
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
