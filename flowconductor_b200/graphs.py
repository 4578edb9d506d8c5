"""CUDA-graph capture of a fixed-shape call through a flow (SURVEY.md §8(f) n2 / n4).

`CompositeTransform._cascade` (flowcon/transforms/base.py:44-52) issues a handful of launches per layer and
`AutoregressiveTransform.inverse` (flowcon/transforms/autoregressive/autoregressive.py:44-53) repeats the
whole conditioner D times: at small batches (cfg 1, the per-GPU shards of cfg 3, sampling from a MAF) the step is
bound by launch latency, not by the kernels.  The B200-first answer is a CUDA graph, not a tracing compiler: the
launch sequence of one call is recorded once, on static buffers, and replayed with a single `cudaGraphLaunch`.

    g = graphs.capture(flow.log_prob, x_example)            # records flow.log_prob(x) for x.shape rows
    lp = g(x)                                               # copy-in, replay; returns the static output
    s = graphs.capture_sampler(flow, 4096)                  # records flow.sample(4096)
    z = s()                                                 # fresh noise every replay (philox state is graph-safe)

Everything the library launches goes to torch's current stream, so the kernels behind the C ABI are captured like
any other work; the path has no host synchronisation as long as the splines use linear tails (the domain check of
`tails=None` reads a device status word on the host, `transforms/splines.py`).  Inference only: the captured call
runs under `torch.no_grad()`.  There is no CPU fallback: capturing needs CUDA tensors.
"""
import torch

__all__ = ["GraphedCall", "GraphedTrainStep", "capture", "capture_sampler"]


def _flatten(out):
    if isinstance(out, torch.Tensor):
        return [out]
    if isinstance(out, (tuple, list)):
        flat = []
        for o in out:
            flat.extend(_flatten(o))
        return flat
    raise TypeError("graph-captured callables must return tensors or tuples of tensors")


class GraphedCall:
    """One recorded call `fn(*inputs)` at fixed input shapes.

    The example inputs define shapes, dtypes and the device; they are copied into static buffers owned by this
    object.  `__call__` copies new inputs into those buffers, replays the graph and returns the static outputs
    (valid until the next replay — `clone()` what must live longer, or pass `clone=True`)."""

    def __init__(self, fn, *example_inputs, warmup=3, pool=None, module=None):
        """module: the nn.Module whose conditioners `fn` runs (default: `fn.__self__` when `fn` is a bound method of a
        module).  The recorded graph contains no weight-packing kernels — the packed tensor-core weights were built during
        the warm-up — so every replay first compares the module's parameter keys (pointer, in-place version) and the
        packed-weight cache generation with those at capture, and records the graph again when the weights have moved on
        (optimizer step, load_state_dict, `tensorcore.invalidate`)."""
        if not example_inputs and not torch.cuda.is_available():
            raise RuntimeError("flowconductor_b200.graphs needs a CUDA device (no CPU fallback)")
        for t in example_inputs:
            if not isinstance(t, torch.Tensor) or not t.is_cuda:
                raise RuntimeError("graph capture needs CUDA tensors as inputs: flowconductor_b200 runs only on the "
                                   "GPU (no CPU fallback)")
        self._fn = fn
        self._static_in = [t.detach().clone() for t in example_inputs]
        self.device = self._static_in[0].device if self._static_in else torch.device("cuda", torch.cuda.current_device())
        if module is None and isinstance(getattr(fn, "__self__", None), torch.nn.Module):
            module = fn.__self__
        self._module = module
        self._warmup, self._pool = warmup, pool
        self.records = 0
        self.replays = 0
        self._record()

    def _weights_state(self):
        from .nn import tensorcore

        if self._module is None:
            return None
        return (tensorcore.cache_generation(), tensorcore.module_param_key(self._module))

    def _record(self):
        fn, warmup, pool = self._fn, self._warmup, self._pool
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.device(self.device), torch.no_grad():
            # warm-up on a side stream: builds the packed-weight plans, sets kernel attributes, fills the allocator
            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                for _ in range(max(1, warmup)):
                    fn(*self._static_in)
            torch.cuda.current_stream(self.device).wait_stream(side)
            torch.cuda.synchronize(self.device)
            with torch.cuda.graph(self.graph, pool=pool):
                self._static_out = fn(*self._static_in)
        self._flat_out = _flatten(self._static_out)
        self._state = self._weights_state()  # after the warm-up built the plans
        self.records += 1

    def __call__(self, *inputs, clone=False):
        if len(inputs) != len(self._static_in):
            raise ValueError("expected {} inputs, got {}".format(len(self._static_in), len(inputs)))
        for dst, src in zip(self._static_in, inputs):
            if src.shape != dst.shape or src.dtype != dst.dtype:
                raise ValueError("graph was captured for inputs of shape {} / {}, got {} / {}".format(
                    tuple(dst.shape), dst.dtype, tuple(src.shape), src.dtype))
            if src.data_ptr() != dst.data_ptr():
                dst.copy_(src, non_blocking=True)
        if self._module is not None and self._weights_state() != self._state:
            self._record()  # the weights changed since capture: the graph holds stale packed copies
        self.graph.replay()
        self.replays += 1
        if not clone:
            return self._static_out
        if isinstance(self._static_out, torch.Tensor):
            return self._static_out.clone()
        return type(self._static_out)(o.clone() if isinstance(o, torch.Tensor) else o for o in self._static_out)

    @property
    def static_inputs(self):
        """The graph's own input buffers: fill them in place to skip the copy-in."""
        return self._static_in


def capture(fn, *example_inputs, warmup=3, pool=None):
    """Record `fn(*example_inputs)` (e.g. `flow.log_prob`, `transform.inverse`) into a CUDA graph."""
    return GraphedCall(fn, *example_inputs, warmup=warmup, pool=pool)


def capture_sampler(flow, num_samples, context=None, with_log_prob=False, warmup=3):
    """Record `flow.sample(num_samples, context)` (or `sample_and_log_prob`).  The base-density noise is drawn
    inside the graph; torch registers the philox offset with the capture, so every replay draws fresh noise."""
    method = flow.sample_and_log_prob if with_log_prob else flow.sample
    if context is None:
        if not next(flow.parameters()).is_cuda:
            raise RuntimeError("graph capture needs the flow on a CUDA device (no CPU fallback)")
        with torch.cuda.device(next(flow.parameters()).device):
            return GraphedCall(lambda: method(num_samples), warmup=warmup, module=flow)
    return GraphedCall(lambda c: method(num_samples, context=c), context, warmup=warmup, module=flow)


class GraphedTrainStep:
    """One whole training step — `zero_grad; loss = loss_fn(*inputs); loss.backward(); [sync_gradients(module)];
    optimizer.step()` (the loop of examples/toy_2d.py:57-67) — recorded into a CUDA graph.  At small per-GPU shards the
    step is bound by its ~450 launches, not by the kernels (cfg 3 at 32 768 rows per rank); a replay is one launch.

    * the optimizer must be capturable (`torch.optim.Adam(..., capturable=True)`): its step counter lives on the device;
    * `sync_gradients` (e.g. `distributed.allreduce_gradients`) is captured with the rest — NCCL collectives are
      graph-capturable;
    * the warm-up steps needed before capture run on the example batch and are UNDONE afterwards (parameters, running
      statistics and optimizer state are restored in place), so constructing the object does not train.
    `step(*inputs)` copies the batch into the static buffers, replays, and returns the (static) loss tensor."""

    def __init__(self, module, optimizer, loss_fn, *example_inputs, sync_gradients=None, warmup=3):
        for t in example_inputs:
            if not isinstance(t, torch.Tensor) or not t.is_cuda:
                raise RuntimeError("graph capture needs CUDA tensors as inputs: flowconductor_b200 runs only on the "
                                   "GPU (no CPU fallback)")
        if not all(g.get("capturable", False) for g in optimizer.param_groups):
            raise ValueError("the optimizer must be constructed with capturable=True to be recorded in a CUDA graph")
        self._static_in = [t.detach().clone() for t in example_inputs]
        self.device = self._static_in[0].device
        params = [p for p in module.parameters()]
        saved_params = [p.detach().clone() for p in params]
        # running statistics (BatchNorm) move during the warm-up too
        buffers = [b for b in module.buffers() if b.is_floating_point()]
        saved_buffers = [b.clone() for b in buffers]
        # optimizer state that already exists (training resumed) is restored; state created by the warm-up is zeroed
        prior = {id(t): t.detach().clone() for st in optimizer.state.values() for t in st.values()
                 if isinstance(t, torch.Tensor)}

        def one_step():
            optimizer.zero_grad(set_to_none=True)
            loss = loss_fn(*self._static_in)
            loss.backward()
            if sync_gradients is not None:
                sync_gradients(module)
            optimizer.step()
            return loss

        with torch.cuda.device(self.device):
            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                for _ in range(max(1, warmup)):
                    one_step()
            torch.cuda.current_stream(self.device).wait_stream(side)
            torch.cuda.synchronize(self.device)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._loss = one_step()
            # undo the warm-up (and the capture itself does not execute): parameters back to their values, optimizer
            # state back to "zero steps taken"
            with torch.no_grad():
                for p, s0 in zip(params + buffers, saved_params + saved_buffers):
                    p.copy_(s0)
                for st in optimizer.state.values():
                    for t in st.values():
                        if isinstance(t, torch.Tensor):
                            if id(t) in prior:
                                t.copy_(prior[id(t)])
                            else:
                                t.zero_()
            torch.cuda.synchronize(self.device)
        self.replays = 0

    def step(self, *inputs):
        if len(inputs) != len(self._static_in):
            raise ValueError("expected {} inputs, got {}".format(len(self._static_in), len(inputs)))
        for dst, src in zip(self._static_in, inputs):
            if src.shape != dst.shape or src.dtype != dst.dtype:
                raise ValueError("graph was captured for inputs of shape {}, got {}".format(tuple(dst.shape),
                                                                                          tuple(src.shape)))
            if src.data_ptr() != dst.data_ptr():
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        self.replays += 1
        return self._loss

    __call__ = step
