"""CUDA-graphed forwards with a static buffer plan (SURVEY.md section 8f-1; reference loop diffusion_ddim.py:244-254,
:157-158 calls the model 2 x 50 times with identical shapes).

A UNet forward is ~1 300 kernel launches and as many output allocations issued from Python.  At config 2 the GPU is
the bottleneck and hides that; at the small configs (VideoLCM 448x256, HiGen stage 1 at one frame) the host is.
So the first call with a given (model, input signature) runs eagerly (it also packs the weights and sets the
per-device function attributes), the second call is captured into a `cudaGraph`:

  * every intermediate of the forward lives in ONE private memory pool owned by the model (the caching allocator's
    capture mode): addresses are fixed, so the TMA tensor maps encoded at capture time stay valid -- this is the
    static buffer plan; nothing is allocated, encoded or launched from Python afterwards;
  * inputs are copied (device-to-device memcpy nodes outside the graph) into static input buffers, the graph is
    replayed with one `cudaGraphLaunch`, and the (small) output is copied out of the pool.

Host-side scalars that vary between calls (DDIM coefficients, guidance scale) never enter a graph: the sampler's
own update kernel stays outside.  Everything a forward needs from its tensor arguments is read on the device.

Graphs are dropped whenever the packed weights are (load_state_dict / .to()): they live inside the packed-weight dict.
VGEN_CUDA_GRAPH=0 disables capture; instrumentation (ops.PROF) and an enclosing user capture also force eager mode.
"""
from __future__ import annotations

import functools
import os
import warnings

import torch

from . import ops

MAX_GRAPHS_PER_MODEL = 8


def enabled() -> bool:
    return os.environ.get("VGEN_CUDA_GRAPH", "1") != "0"


class _Entry:
    __slots__ = ("graph", "static", "out", "uses")

    def __init__(self):
        self.graph, self.static, self.out, self.uses = None, None, None, 0


class GraphCache:
    """Per-model cache: signature -> captured graph.  All graphs of a model share one memory pool."""

    def __init__(self):
        self.entries = {}
        self.seen = {}      # signature -> eager calls so far (capture on the second sighting)
        self.pool = None
        self.replays = 0
        self.captures = 0

    @staticmethod
    def _flatten(args, kwargs):
        """-> (list of CUDA tensors, hashable signature, rebuild(tensors) -> (args, kwargs)) or None if not graphable."""
        tensors, sig = [], []
        slots = [("a", i, v) for i, v in enumerate(args)] + [("k", k, kwargs[k]) for k in sorted(kwargs)]
        for kind, name, v in slots:
            if torch.is_tensor(v):
                if not v.is_cuda:
                    return None
                sig.append((kind, name, "T", tuple(v.shape), v.dtype))
                tensors.append(v)
            elif v is None or isinstance(v, (bool, int, float, str)):
                sig.append((kind, name, "V", v))
            else:
                return None

        def rebuild(ts):
            it = iter(ts)
            a = [next(it) if torch.is_tensor(v) else v for v in args]
            k = {key: (next(it) if torch.is_tensor(kwargs[key]) else kwargs[key]) for key in sorted(kwargs)}
            return a, k
        return tensors, tuple(sig), rebuild

    def run(self, fn, owner, args, kwargs):
        flat = self._flatten(args, kwargs)
        if flat is None:
            return fn(owner, *args, **kwargs)
        tensors, sig, rebuild = flat
        ent = self.entries.get(sig)
        if ent is None:
            n = self.seen.get(sig, 0)
            self.seen[sig] = n + 1
            if n <= 0 or len(self.entries) >= MAX_GRAPHS_PER_MODEL:
                return fn(owner, *args, **kwargs)       # first sighting: eager (doubles as the warm-up)
            try:
                ent = self._capture(fn, owner, tensors, rebuild)
            except Exception as e:  # noqa: BLE001 - capture is an optimisation: say so loudly, then keep working eagerly
                warnings.warn(f"vgen_b200: CUDA graph capture of {type(owner).__name__}.{fn.__name__} failed ({e!r}); "
                              "this input signature stays on the eager launch path")
                self.seen[sig] = -(1 << 30)
                torch.cuda.synchronize()
                return fn(owner, *args, **kwargs)
            self.entries[sig] = ent
        for s, src in zip(ent.static, tensors):
            if s.data_ptr() != src.data_ptr():
                s.copy_(src, non_blocking=True)           # contiguous same-dtype: a D2D memcpy on the current stream
        ent.graph.replay()
        ent.uses += 1
        self.replays += 1
        return ent.out.clone()

    def _capture(self, fn, owner, tensors, rebuild):
        ent = _Entry()
        ent.static = [t.detach().clone(memory_format=torch.contiguous_format) for t in tensors]
        a, k = rebuild(ent.static)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        if self.pool is None:
            self.pool = torch.cuda.graph_pool_handle()
        with torch.cuda.graph(g, pool=self.pool):
            ent.out = fn(owner, *a, **k)
        ent.graph = g
        self.captures += 1
        return ent


def graphed(fn=None, *, key=None):
    """Decorator for a SpecModule method whose tensor arguments fully determine its device work.  `key` names the
    method's graph cache (default: the method's own name)."""
    if fn is None:
        return lambda f: graphed(f, key=key)
    name = key or fn.__name__

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        W = self._packed
        if W is None:                                    # not packed yet (or just invalidated): eager call packs (or raises on CPU)
            out = fn(self, *args, **kwargs)
            if self._packed is not None and enabled():   # it still counts as the first sighting of this signature
                flat = GraphCache._flatten(args, kwargs)
                if flat is not None:
                    c = self._packed.setdefault("__graphs__", {}).setdefault(name, GraphCache())
                    c.seen[flat[1]] = max(c.seen.get(flat[1], 0), 1)
            return out
        if (not enabled() or ops.PROF is not None or not getattr(self, "use_cuda_graph", True)
                or torch.cuda.is_current_stream_capturing()):
            return fn(self, *args, **kwargs)
        cache = W.get("__graphs__")
        if cache is None:
            cache = W["__graphs__"] = {}
        c = cache.get(name)
        if c is None:
            c = cache[name] = GraphCache()
        return c.run(fn, self, args, kwargs)
    wrapper.__wrapped_eager__ = fn
    return wrapper


def stats(module):
    """{method: (captures, replays)} of a module's graph caches (tests / bench)."""
    W = getattr(module, "_packed", None) or {}
    return {k: (c.captures, c.replays) for k, c in (W.get("__graphs__") or {}).items()}
