"""CUDA-graph capture of fixed-shape stage functions.

Each network stage is ~100-130 small launches; issued one by one from Python they cost more host
time than device time at batch 1 (the stages are serial per frame, so the launch latency is on
the critical path).  A stage whose input shapes repeat is captured once into a CUDA graph with
static input/output buffers and replayed with a single launch; all kernels are stream-ordered
C-ABI launches that never synchronise or allocate outside torch's graph pool, so they capture as is.
Disable with G6D_GRAPHS=0 (the eager path is what the parity tests of the internals exercise).
"""
import os

import torch

from . import _lib

REPLAYED_KERNELS = [0]   # kernels launched through graph replays (the C-ABI launch counter only sees eager calls)


def graphs_enabled():
    return os.environ.get('G6D_GRAPHS', '1') != '0'


class CapturedStage:
    """fn(*tensors) -> tensor or tuple of tensors, captured for one input-shape signature.  `state`: tensors that fn
    updates in place and that carry over from call to call (a tracker's poses and history); the warm-up runs must not
    advance them, so they are restored after the capture."""

    def __init__(self, fn, example_inputs, warmup=2, state=()):
        self.static_in = [t.clone() for t in example_inputs]
        saved = [t.clone() for t in state]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):
                fn(*self.static_in)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        before = _lib.launch_count()
        # thread_local: other host threads (predict_many workers) may keep issuing CUDA calls meanwhile
        with torch.cuda.graph(self.graph, capture_error_mode='thread_local'), torch.no_grad():
            self.static_out = fn(*self.static_in)
        self.kernels = _lib.launch_count() - before     # kernel nodes captured (our C-ABI launches)
        for t, s in zip(state, saved):
            t.copy_(s)

    def __call__(self, *inputs):
        for s, t in zip(self.static_in, inputs):
            s.copy_(t, non_blocking=True)
        self.graph.replay()
        REPLAYED_KERNELS[0] += self.kernels
        return self.static_out


class StageCache:
    """Per-module cache of captured stages keyed by (name, input shapes/dtypes)."""

    def __init__(self):
        self.stages = {}

    def clear(self):
        self.stages.clear()

    def run(self, name, fn, inputs, state=()):
        if not graphs_enabled():
            return fn(*inputs)
        key = (name,) + tuple((tuple(t.shape), t.dtype) for t in inputs)
        st = self.stages.get(key)
        if st is None:
            st = self.stages[key] = CapturedStage(fn, inputs, state=state)
        return st(*inputs)
