"""Host <-> device staging around the hot path (the reference's DataLoader + ``.cuda()`` + ``.cpu()`` glue,
train_and_test.py:24-34): double-buffered so that the host->device copy of batch i+1 and the device->host read of
batch i's logits overlap the compute of batch i.  Plain CUDA streams and events; nothing here touches the kernels."""
from __future__ import annotations

import torch


class HostFeeder:
    """``depth`` device buffers fed from pinned host tensors on a copy stream.

        feeder.stage(x_host)            # enqueue the H2D copy of a batch (call one batch ahead)
        x = feeder.acquire()            # device tensor of the oldest staged batch; the current stream waits for its copy
        ... launch work reading x on the current stream ...
        feeder.release(x)               # the buffer may be overwritten once that work has finished
    """

    def __init__(self, shape, device, dtype=torch.float32, depth: int = 2):
        self.bufs = [torch.empty(shape, device=device, dtype=dtype) for _ in range(depth)]
        self.copy_stream = torch.cuda.Stream(device=device)
        self.ready = [torch.cuda.Event() for _ in range(depth)]
        self.free = [None] * depth
        self.staged = []            # indices in FIFO order
        self.next = 0

    def stage(self, x_host: torch.Tensor):
        i = self.next
        self.next = (self.next + 1) % len(self.bufs)
        if i in self.staged:
            raise RuntimeError("mgproto_b200: HostFeeder overrun (stage() called more than `depth` batches ahead)")
        buf = self.bufs[i]
        buf.requires_grad_(False)
        with torch.cuda.stream(self.copy_stream):
            if self.free[i] is not None:
                self.copy_stream.wait_event(self.free[i])
            buf.copy_(x_host, non_blocking=True)
            self.ready[i].record(self.copy_stream)
        self.staged.append(i)

    def acquire(self) -> torch.Tensor:
        i = self.staged.pop(0)
        torch.cuda.current_stream().wait_event(self.ready[i])
        return self.bufs[i]

    def release(self, buf: torch.Tensor):
        i = next(k for k, b in enumerate(self.bufs) if b is buf)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self.free[i] = ev


class HostSink:
    """Device -> pinned host copies on their own stream (``depth`` host buffers, reused round-robin)."""

    def __init__(self, shape, dtype=torch.float32, depth: int = 2, device=None):
        self.bufs = [torch.empty(shape, dtype=dtype, pin_memory=True) for _ in range(depth)]
        self.stream = torch.cuda.Stream(device=device)
        self.done = [None] * depth
        self.next = 0

    def put(self, t_dev: torch.Tensor) -> torch.Tensor:
        """Enqueue the read-back of ``t_dev`` (produced on the current stream); returns the host buffer it lands in
        (valid after ``wait()`` or once its event has completed)."""
        i = self.next
        self.next = (self.next + 1) % len(self.bufs)
        produced = torch.cuda.Event()
        produced.record(torch.cuda.current_stream())
        if self.done[i] is not None:
            self.done[i].synchronize()                 # the host buffer is about to be overwritten
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(produced)
            self.bufs[i].copy_(t_dev, non_blocking=True)
            t_dev.record_stream(self.stream)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self.done[i] = ev
        return self.bufs[i]

    def wait(self):
        self.stream.synchronize()


class GraphedStep:
    """The whole training step -- head forward, loss, backward, bank enqueue, update_GMM -- captured ONCE in a CUDA
    graph and replayed per batch: the ~20 kernel launches of a step cost the host one ``cudaGraphLaunch`` instead of
    ~400 us of Python / ctypes / dispatcher work, and the kernels run back to back.

        step = GraphedStep(net, loss_fn, x0, gt0)     # runs `warmup` REAL steps on (x0, gt0), then captures one more
        for x, gt in batches:
            out, loss = step(x, gt)                   # x [B,D,H,W] features, gt [B] int64 (same shapes as x0, gt0)
            # step.x_grad holds d loss / d x for the backbone (static buffer, overwritten by the next call)

    Everything the step does on the host (version bumps, the optimiser-state bookkeeping of update_GMM) happens at
    capture time only, so ``__call__`` re-announces the raw-pointer writes to torch after every replay.  The library's
    kernels keep all step-dependent state (Adam step counter, bank cursors, update flags) on the device, which is what
    makes the step replayable.  Shapes are fixed; with ``torch.distributed`` initialised the all-gather of the
    multi-GPU exchange is captured with the rest (every rank must construct and call the step in lock-step).

    A capture bakes in host values: prototype_optimizer's lr / betas / eps and its moment tensors, the model's tau,
    alpha, num_em_loop, mine_T and math_mode, and the addresses of the means, sigmas and mixture weights.  Every call
    compares them with the captured ones; after a change (an lr scheduler step, optimizer.load_state_dict, a new
    optimiser, ...) the step is captured again before it is replayed.  A capture runs no kernels, so the step stays
    equal to the eager one.  With torch.distributed every rank must make the same change before the same call.
    Writes into the tensors themselves (in place, or through ``.data``) need nothing: the graph reads them.
    """

    def __init__(self, net, loss_fn, x_example: torch.Tensor, gt_example: torch.Tensor, warmup: int = 3):
        self.net, self.loss_fn = net, loss_fn
        dev = x_example.device
        self.x = torch.empty_like(x_example).requires_grad_(True)
        self.gt = torch.empty_like(gt_example)
        with torch.no_grad():
            self.x.copy_(x_example)
            self.gt.copy_(gt_example)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):       # lazy initialisations (workspaces, shadows, device counters) happen here
                self._body()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = None
        self._capture()

    def _baked(self):
        """What a capture bakes in: (objects compared by identity, values compared by equality)."""
        net = self.net
        opt = net.prototype_optimizer
        g = opt.param_groups[0] if opt is not None else {}
        st = opt.state.get(net.prototype_means, {}) if opt is not None else {}
        objs = (opt, st.get("exp_avg"), st.get("exp_avg_sq"))
        vals = (float(g.get("lr", 0.0)), tuple(g.get("betas", ())), g.get("eps"), net.tau, net.alpha, net.num_em_loop,
                net.mine_T, net.math_mode, net.prototype_means.data_ptr(), net.prototype_covs.data_ptr(),
                net.last_layer.weight.data_ptr())
        return objs, vals

    def _capture(self):
        from . import ops
        prepare = getattr(self.net, "_prepare_adam", None)
        if prepare is not None and self.net.prototype_optimizer is not None:
            prepare()                               # Adam state and step counter: eager, never inside the capture
        if self.graph is not None:
            self.graph.reset()
        self.graph = torch.cuda.CUDAGraph()
        n0 = ops.launch_count()
        with torch.cuda.graph(self.graph):
            self.out, self.loss = self._body()
        self.launches = ops.launch_count() - n0      # library kernels per replay (torch's own few are not counted)
        self.x_grad = self.x.grad
        self._captured = self._baked()
        self._em_dirty = getattr(self.net, "_em_dirty", False)   # a replay advances the device Adam step count

    def close(self):
        """Release the captured graph (and its private memory pool).  With torch.distributed: call it before
        destroy_process_group -- NCCL communicators must outlive the graphs that captured their kernels."""
        self.graph.reset()
        self.out = self.loss = self.x_grad = None

    def _body(self):
        self.x.grad = None
        out = self.net.head(self.x, self.gt)
        loss = self.loss_fn(out, self.gt)
        loss.backward()
        self.net.update_GMM()
        return out, loss

    def __call__(self, x: torch.Tensor, gt: torch.Tensor):
        objs, vals = self._baked()
        if vals != self._captured[1] or any(a is not b for a, b in zip(objs, self._captured[0])):
            self._capture()
        with torch.no_grad():
            self.x.copy_(x, non_blocking=True)
            self.gt.copy_(gt, non_blocking=True)
        self.graph.replay()
        bump = getattr(self.net, "_bump_versions", None)
        if bump is not None:
            bump()
        if self._em_dirty:
            self.net._em_dirty = True               # sync_optimizer_state folds the replayed steps back
        return self.out, self.loss
