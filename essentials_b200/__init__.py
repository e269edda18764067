"""essentials_b200 — host-side mirror of the Gunrock/Essentials frontier-operator API over the C ABI.

The product is the sm_100a CUDA code under ``include/gunrock/`` (header-template operator API, the drop-in
for the reference's ``<gunrock/...>`` headers) and its C ABI ``include/essentials_b200.h`` built into
``essentials_b200/libessentials_b200.so``.  This package is the thin ctypes binding a Python host uses:
torch supplies device memory, streams and ``torch.distributed``; every graph kernel runs in the library.

There is NO CPU fallback: importing works anywhere (so the C-ABI symbol test can run without a GPU), but
every compute call goes through the CUDA library and raises if it is missing or fails.

Names follow the reference: ``bfs.run`` -> :func:`bfs`, ``operators::load_balance_t`` -> :data:`LOAD_BALANCE`,
``advance_direction_t`` -> :data:`DIRECTION`, ``filter_algorithm_t`` -> :data:`FILTER`.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, byref, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p
from dataclasses import dataclass

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libessentials_b200.so")

# operators::load_balance_t / advance_direction_t / filter_algorithm_t — same values as
# include/gunrock/framework/operators/configs.hxx (reference :31-59).
LOAD_BALANCE = {"thread_mapped": 0, "warp_mapped": 1, "block_mapped": 2, "bucketing": 3, "merge_path": 4,
                "merge_path_v2": 5, "work_stealing": 6}
DIRECTION = {"forward": 0, "backward": 1, "optimized": 2}
FILTER = {"remove": 0, "predicated": 1, "compact": 2, "bypass": 3}
IMPLEMENTED_LOAD_BALANCERS = ("thread_mapped", "block_mapped", "bucketing", "merge_path")


class EssentialsError(RuntimeError):
    """Raised when a C-ABI call returns non-zero (mirrors gunrock::error::exception_t)."""


class OutputOverflow(EssentialsError):
    """An operator produced more elements than the caller's output buffer holds. `produced` is the full count,
    `prefix` the `capacity` elements the buffer kept (which ones is unspecified, like the slot order), `calls` the
    per-edge call counts of the run."""

    def __init__(self, what: str, produced: int, capacity: int, prefix, calls):
        super().__init__(f"{what}: produced {produced} elements, the output holds {capacity}")
        self.produced, self.capacity, self.prefix, self.calls = produced, capacity, prefix, calls


class RunInfo(Structure):
    _fields_ = [("enact_ms", c_float), ("iterations", c_int32), ("pull_steps", c_int32), ("push_steps", c_int32),
                ("reserved", c_int64 * 8)]

    def as_dict(self):
        return {"enact_ms": float(self.enact_ms), "iterations": int(self.iterations),
                "pull_steps": int(self.pull_steps), "push_steps": int(self.push_steps),
                "pull_vertices": int(self.reserved[0]), "pull_edges": int(self.reserved[1]),
                "push_vertices": int(self.reserved[2]), "push_edges": int(self.reserved[3]),
                "pull_misses": int(self.reserved[4]), "pull_found": int(self.reserved[5]),
                "push_found": int(self.reserved[6])}


_SIGNATURES = {
    "ess_last_error": (c_char_p, []),
    "ess_version": (c_int, []),
    "ess_context_create": (c_int, [c_int, c_void_p, c_int, POINTER(c_void_p)]),
    "ess_context_destroy": (c_int, [c_void_p]),
    "ess_context_synchronize": (c_int, [c_void_p]),
    "ess_tune": (c_int, [c_char_p, c_int]),
    "ess_profile_enable": (c_int, [c_void_p, c_int]),
    "ess_profile_read": (c_int, [c_void_p, c_void_p, c_void_p, c_int]),
    "ess_graph_create_from_host": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                           POINTER(c_void_p)]),
    "ess_graph_create": (c_int, [c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                 c_void_p, POINTER(c_void_p)]),
    "ess_graph_destroy": (c_int, [c_void_p]),
    "ess_graph_build_pull_hints": (c_int, [c_void_p, c_void_p]),
    "ess_bfs_partition_pull": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "ess_transpose_csr": (c_int, [c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ess_bfs": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int, c_int, c_float, c_float, POINTER(RunInfo)]),
    "ess_bfs_tree": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int, c_int, c_float, c_float,
                             POINTER(RunInfo)]),
    "ess_sssp": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int, POINTER(RunInfo)]),
    "ess_sssp_near_far": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_float, POINTER(RunInfo)]),
    "ess_sssp_delta": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_float, POINTER(RunInfo)]),
    "ess_pagerank": (c_int, [c_void_p, c_void_p, c_float, c_float, c_int, c_void_p, c_int, c_int, POINTER(RunInfo)]),
    "ess_ppr": (c_int, [c_void_p, c_void_p, c_int32, c_float, c_float, c_void_p, c_int, POINTER(RunInfo)]),
    "ess_kcore": (c_int, [c_void_p, c_void_p, c_void_p, c_int, POINTER(RunInfo)]),
    "ess_color": (c_int, [c_void_p, c_void_p, c_void_p, POINTER(RunInfo)]),
    "ess_randoms": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_float]),
    "ess_advance_probe": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_int64,
                                  POINTER(c_int64), c_void_p, c_int32]),
    "ess_advance_unique_probe": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p, c_int64,
                                  POINTER(c_int64), c_void_p, c_int32]),
    "ess_filter_probe": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p, POINTER(c_int64), c_void_p,
                                 c_int32]),
    "ess_uniquify_probe": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_int64)]),
    "ess_atomic_probe": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_int]),
    "ess_frontier_to_bitmap": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, POINTER(c_int64)]),
    "ess_bitmap_to_frontier": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_int64)]),
    "ess_bits_to_list_async": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "ess_bfs_partition_step": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_int64]),
    "ess_bfs_merge_gathered": (c_int, [c_void_p, c_void_p, c_int32, c_int64, c_void_p, c_void_p, c_void_p]),
    "ess_bfs_absorb": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int32, c_int64, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p]),
    "ess_nccl_unique_id": (c_int, [c_void_p]),
    "ess_dist_create": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p, POINTER(c_void_p)]),
    "ess_dist_destroy": (c_int, [c_void_p]),
    "ess_dist_bfs": (c_int, [c_void_p, c_int64, c_float, c_float, POINTER(RunInfo)]),
    "ess_dist_copy_depth": (c_int, [c_void_p, c_void_p]),
    "ess_dist_exchange_kind": (c_int, [c_void_p, POINTER(c_int)]),
    "ess_dist_sssp": (c_int, [c_void_p, c_int64, POINTER(RunInfo)]),
    "ess_dist_bfs_enactor": (c_int, [c_void_p, c_int64, c_int, c_void_p, POINTER(RunInfo)]),
    "ess_dist_sssp_enactor": (c_int, [c_void_p, c_int64, c_int, c_void_p, POINTER(RunInfo)]),
    "ess_dist_copy_dist": (c_int, [c_void_p, c_void_p]),
    "ess_sssp_partition_relax": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "ess_sssp_partition_collect": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ess_dist_depth_local": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_int64)]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """The CUDA library. Fails loudly when it has not been built (``python __graft_entry__.py build``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EssentialsError(
                f"{LIB_PATH} is missing: build it with `make -C essentials_b200/csrc -j` "
                "(there is no CPU fallback for the frontier operators)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _check(code: int, what: str):
    if code != 0:
        msg = lib().ess_last_error()
        raise EssentialsError(f"{what} failed ({code}): {msg.decode() if msg else ''}")


def tune(knob: str, value: int):
    """Development knobs of the library (ess_tune)."""
    _check(lib().ess_tune(knob.encode(), int(value)), "ess_tune")


def _p(t):
    return None if t is None else c_void_p(t.data_ptr())


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise EssentialsError("device tensors required: the frontier operators only run on the GPU")


class Context:
    """gcuda::multi_context_t with one device (reference include/gunrock/cuda/context.hxx:136-206)."""

    def __init__(self, device: int = 0, stream=None, own_stream: bool = False):
        """stream: a torch.cuda.Stream (default: torch's current stream on `device`), so library kernels are
        ordered with the torch ops that produce/consume the tensors; own_stream=True gives the context a
        private non-blocking stream like the reference's default context."""
        import torch
        self.device = device
        torch.cuda.init()
        with torch.cuda.device(device):
            if stream is None and not own_stream:
                stream = torch.cuda.current_stream()
            self._stream_obj = stream  # keep the torch stream alive
            raw = None if stream is None else c_void_p(stream.cuda_stream)
            h = c_void_p()
            _check(lib().ess_context_create(device, raw, int(own_stream), byref(h)), "ess_context_create")
        self.handle = h

    def synchronize(self):
        _check(lib().ess_context_synchronize(self.handle), "ess_context_synchronize")

    PROFILE_CLASSES = ("pull_step", "push_expand", "work_prepare", "dense_state", "filter")

    def profile(self, enable: bool):
        """Start (and reset) or stop per-kernel-class CUDA-event timing on this context's stream."""
        _check(lib().ess_profile_enable(self.handle, int(enable)), "ess_profile_enable")

    def profile_read(self):
        """{class: (milliseconds, launches)} accumulated since profile(True)."""
        ms = (ctypes.c_double * 8)()
        cnt = (c_int64 * 8)()
        _check(lib().ess_profile_read(self.handle, ms, cnt, 8), "ess_profile_read")
        out = {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.PROFILE_CLASSES)}
        self.kernel_launches = int(cnt[7])  # all operator kernels launched on this context so far
        return out

    def launches(self) -> int:
        """Kernels the library has launched on this context since it was created."""
        self.profile_read()
        return self.kernel_launches

    def close(self):
        if getattr(self, "handle", None):
            lib().ess_context_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Graph:
    """graph_t view over caller-owned CSR (+ optional CSC) device arrays
    (graph::build::from_csr, reference include/gunrock/graph/build.hxx:21-36)."""

    def __init__(self, csr, csc=None, symmetric: bool | None = None, partition: bool = False):
        """partition=True: `csr` is a row range of a partitioned symmetric graph (global column ids)."""
        _need_cuda(csr.offsets, csr.indices, csr.values)
        self.csr, self.csc = csr, csc
        self.n, self.m = int(csr.offsets.numel() - 1), int(csr.indices.numel())
        self.offset_bits = 64 if csr.offsets.element_size() == 8 else 32
        sym = bool(csr.symmetric) if symmetric is None else symmetric
        if csc is not None:
            _need_cuda(csc.offsets, csc.indices, csc.values)
            assert csc.offsets.dtype == csr.offsets.dtype
        h = c_void_p()
        _check(lib().ess_graph_create(self.n, self.m, self.offset_bits, _p(csr.offsets), _p(csr.indices),
                                      _p(csr.values), (2 if partition else 1) if (sym and csc is None) else 0,
                                      _p(csc.offsets) if csc is not None else None,
                                      _p(csc.indices) if csc is not None else None,
                                      _p(csc.values) if csc is not None else None, byref(h)), "ess_graph_create")
        self.handle = h
        self.has_csc = sym or csc is not None
        self.device = csr.indices.device

    @classmethod
    def from_host(cls, ctx: "Context", csr, symmetric: bool | None = None):
        """ess_graph_create_from_host: `csr` holds HOST tensors (pinned memory lets the copy overlap); the handle owns
        the device copies, and the bottom-up hints are built chunk by chunk while the column indices are still crossing
        PCIe. Mirrors the reference drivers' host csr_t -> device vectors -> from_csr sequence
        (examples/algorithms/bfs/bfs.cu:25-66)."""
        import torch
        for t in (csr.offsets, csr.indices, csr.values):
            if t is not None and t.is_cuda:
                raise EssentialsError("Graph.from_host takes host tensors; use Graph(csr) for device arrays")
            if t is not None and not t.is_contiguous():
                raise EssentialsError("Graph.from_host needs contiguous arrays")
        if csr.indices.dtype != torch.int32 or (csr.values is not None and csr.values.dtype != torch.float32):
            raise EssentialsError("Graph.from_host: column indices are int32 and values float32")
        self = cls.__new__(cls)
        self.csr, self.csc = csr, None
        self.n, self.m = int(csr.offsets.numel() - 1), int(csr.indices.numel())
        self.offset_bits = 64 if csr.offsets.element_size() == 8 else 32
        sym = bool(csr.symmetric) if symmetric is None else bool(symmetric)
        self.handle = None
        h = c_void_p()
        with torch.cuda.device(ctx.device):
            _check(lib().ess_graph_create_from_host(ctx.handle, self.n, self.m, self.offset_bits, _p(csr.offsets),
                                                    _p(csr.indices), _p(csr.values), int(sym), byref(h)),
                   "ess_graph_create_from_host")
        self.handle = h
        self.has_csc = sym
        self.device = torch.device("cuda", ctx.device)
        return self

    def build_pull_hints(self, degree_of_id=None):
        """graph::build::pull_hints; degree_of_id (int32 per global id) is required for partitions."""
        _check(lib().ess_graph_build_pull_hints(self.handle, _p(degree_of_id)), "ess_graph_build_pull_hints")

    def close(self):
        if getattr(self, "handle", None):
            lib().ess_graph_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _out(n, dtype, g):
    import torch
    return torch.empty(n, dtype=dtype, device=g.device)


def bfs(ctx: Context, g: Graph, source: int, lb: str = "block_mapped", direction: str = "forward", out=None,
        alpha: float = 0.0, beta: float = 0.0):
    """gunrock::bfs::run (reference include/gunrock/algorithms/bfs.hxx:151-176). Returns (depth[int32], info)."""
    import torch
    depth = _out(g.n, torch.int32, g) if out is None else out
    info = RunInfo()
    _check(lib().ess_bfs(ctx.handle, g.handle, int(source), _p(depth), LOAD_BALANCE[lb], DIRECTION[direction],
                         alpha, beta, byref(info)), "ess_bfs")
    return depth, info.as_dict()


def _label_buffer(t, g: Graph, what: str):
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.int32 and t.is_contiguous()
            and t.numel() >= g.n and t.device == g.device):
        raise EssentialsError(f"{what} must be a contiguous int32 CUDA tensor of at least {g.n} elements on {g.device}")
    return t


def bfs_tree(ctx: Context, g: Graph, source: int, lb: str = "block_mapped", direction: str = "forward", out=None,
             pred_out=None, alpha: float = 0.0, beta: float = 0.0):
    """gunrock::bfs::run_tree: :func:`bfs` plus the BFS tree. Returns (depth[int32], pred[int32], info).

    `depth` and `info` are what :func:`bfs` returns. pred[source] == source; pred[v] == -1 exactly where v is unreached
    (depth INT32_MAX); every other pred[v] is an in-neighbour u of v (an edge u -> v) with depth[u] == depth[v] - 1.
    Which valid parent is chosen is not deterministic. `out` and `pred_out`, when given, must be contiguous int32 CUDA
    tensors of at least g.n elements on the graph's device, and must not overlap."""
    import torch
    depth = _out(g.n, torch.int32, g) if out is None else _label_buffer(out, g, "out")
    pred = _out(g.n, torch.int32, g) if pred_out is None else _label_buffer(pred_out, g, "pred_out")
    span = 4 * g.n
    if depth.data_ptr() < pred.data_ptr() + span and pred.data_ptr() < depth.data_ptr() + span:
        raise EssentialsError("bfs_tree: pred_out must not overlap out")
    info = RunInfo()
    _check(lib().ess_bfs_tree(ctx.handle, g.handle, int(source), _p(depth), _p(pred), LOAD_BALANCE[lb],
                              DIRECTION[direction], alpha, beta, byref(info)), "ess_bfs_tree")
    return depth, pred, info.as_dict()


def sssp(ctx: Context, g: Graph, source: int, lb: str = "block_mapped", out=None):
    """gunrock::sssp::run (reference include/gunrock/algorithms/sssp.hxx:155-185). Returns (dist[float32], info)."""
    import torch
    dist = _out(g.n, torch.float32, g) if out is None else out
    info = RunInfo()
    _check(lib().ess_sssp(ctx.handle, g.handle, int(source), _p(dist), LOAD_BALANCE[lb], byref(info)), "ess_sssp")
    return dist, info.as_dict()


def sssp_near_far(ctx: Context, g: Graph, source: int, delta: float = 0.0, out=None):
    """SSSP through operators::advance::execute_near_far (near/far ordering in one persistent kernel)."""
    import torch
    dist = _out(g.n, torch.float32, g) if out is None else out
    info = RunInfo()
    _check(lib().ess_sssp_near_far(ctx.handle, g.handle, int(source), _p(dist), float(delta), byref(info)),
           "ess_sssp_near_far")
    d = info.as_dict()
    d.update(levels=int(info.reserved[0]), splits=int(info.reserved[1]), relaxations=int(info.reserved[2]))
    return dist, d


def sssp_delta(ctx: Context, g: Graph, source: int, delta: float = 0.0, out=None):
    """SSSP through gunrock::sssp::run_delta (dense active set + delta thresholds; for low-diameter graphs)."""
    import torch
    dist = _out(g.n, torch.float32, g) if out is None else out
    info = RunInfo()
    _check(lib().ess_sssp_delta(ctx.handle, g.handle, int(source), _p(dist), float(delta), byref(info)),
           "ess_sssp_delta")
    d = info.as_dict()
    d.update(rounds=int(info.reserved[0]), threshold_advances=int(info.reserved[1]),
             expanded_vertices=int(info.reserved[2]), passes=int(info.reserved[3]))
    return dist, d


def pagerank(ctx: Context, g: Graph, alpha: float = 0.85, tol: float = 1e-6, max_iterations: int = 1000,
             lb: str = "block_mapped", pull: bool | None = None, out=None):
    """gunrock::pr::run (reference include/gunrock/algorithms/pr.hxx:183-216). Returns (p[float32], info).

    `pull=None` (default) gathers over the in-edge view whenever the graph has one (a CSC, or a symmetric CSR): every
    vertex sums its contributions in one fixed order, and the ranks agree with the reference's CPU PageRank to 1e-6
    per element — this is the parity path. `pull=False` is the reference's formulation, an advance that scatters
    `atomic::add` over the out-edges with balancer `lb`; float additions then arrive in whatever order the hardware
    schedules them, so individual ranks can differ by up to ~1e-4 relative from run to run (1e-6 in L1), exactly as
    the reference's GPU PageRank does. Without an in-edge view the default is the scatter. The gather raises
    :class:`EssentialsError` when only one of the CSR and the CSC carries edge weights."""
    import torch
    p = _out(g.n, torch.float32, g) if out is None else out
    info = RunInfo()
    if pull is None:
        pull = bool(g.has_csc)
    _check(lib().ess_pagerank(ctx.handle, g.handle, alpha, tol, max_iterations, _p(p), LOAD_BALANCE[lb], int(pull),
                              byref(info)), "ess_pagerank")
    return p, info.as_dict()


def ppr(ctx: Context, g: Graph, seed: int, alpha: float = 0.15, epsilon: float = 1e-6, lb: str = "block_mapped",
        out=None):
    """gunrock::ppr::run (reference include/gunrock/algorithms/ppr.hxx:150-179)."""
    import torch
    p = _out(g.n, torch.float32, g) if out is None else out
    info = RunInfo()
    _check(lib().ess_ppr(ctx.handle, g.handle, int(seed), alpha, epsilon, _p(p), LOAD_BALANCE[lb], byref(info)),
           "ess_ppr")
    return p, info.as_dict()


def kcore(ctx: Context, g: Graph, lb: str = "block_mapped", out=None):
    """gunrock::kcore::run (reference include/gunrock/algorithms/kcore.hxx:202-222)."""
    import torch
    k = _out(g.n, torch.int32, g) if out is None else out
    info = RunInfo()
    _check(lib().ess_kcore(ctx.handle, g.handle, _p(k), LOAD_BALANCE[lb], byref(info)), "ess_kcore")
    return k, info.as_dict()


def color(ctx: Context, g: Graph, out=None):
    """gunrock::color::run (reference include/gunrock/algorithms/color.hxx:155-180)."""
    import torch
    c = _out(g.n, torch.int32, g) if out is None else out
    info = RunInfo()
    _check(lib().ess_color(ctx.handle, g.handle, _p(c), byref(info)), "ess_color")
    return c, info.as_dict()


def randoms(ctx: Context, n: int, begin: float, end: float, device="cuda"):
    """generate::random::uniform_distribution (reference include/gunrock/algorithms/generate/random.hxx:20-33)."""
    import torch
    out = torch.empty(n, dtype=torch.float32, device=device)
    _check(lib().ess_randoms(ctx.handle, _p(out), n, begin, end), "ess_randoms")
    return out


def _frontier_edges(g: Graph, frontier, backward: bool) -> int:
    """Σ out-degree (in-degree when `backward`) of the valid items of `frontier`: the most an advance can emit."""
    import torch
    view = g.csc if backward and g.csc is not None else g.csr
    f = frontier.to(view.offsets.device, torch.int64)
    f = f[f >= 0]
    return int((view.offsets[f + 1] - view.offsets[f]).sum()) if f.numel() else 0


def _probe_output(what: str, out, cap: int, produced: int, calls):
    if produced > cap:
        raise OutputOverflow(what, produced, cap, out[:cap], calls)
    return out[:produced], calls


def advance_probe(ctx: Context, g: Graph, frontier, lb: str = "merge_path", direction: str = "forward",
                  modulus: int = 3, count_calls: bool = True, capacity: int | None = None):
    """operators::advance::execute with the header's fixed test operator. Returns (kept neighbours, per-edge
    call counts or None).

    `capacity` sizes the output buffer handed to the operator (default: the frontier's Σdeg + 1, which always fits).
    A smaller buffer takes the operator's grow-and-relaunch path; if more neighbours are kept than it holds,
    :class:`OutputOverflow` is raised with the produced count and the prefix that fits."""
    import torch
    _need_cuda(frontier)
    calls = torch.zeros(max(g.m, 1), dtype=torch.int32, device=frontier.device) if count_calls else None
    n_out = c_int64(0)
    cap = _frontier_edges(g, frontier, direction == "backward") + 1 if capacity is None else int(capacity)
    out = torch.empty(max(cap, 1), dtype=torch.int32, device=frontier.device)
    _check(lib().ess_advance_probe(ctx.handle, g.handle, LOAD_BALANCE[lb], DIRECTION[direction], _p(frontier),
                                   int(frontier.numel()), _p(out), cap, byref(n_out), _p(calls), modulus),
           "ess_advance_probe")
    return _probe_output("ess_advance_probe", out, cap, n_out.value, calls)


def advance_unique_probe(ctx: Context, g: Graph, frontier, lb: str = "merge_path", modulus: int = 3,
                         capacity: int | None = None):
    """operators::advance::execute_unique (fused advance + uniquify) with the fixed test operator, run twice on the
    same bitmap. Returns (duplicate-free kept neighbours, per-edge call counts == 2 on every expanded edge).
    `capacity` as for :func:`advance_probe`; the operator's capacity guard still compares it with Σdeg."""
    import torch
    _need_cuda(frontier)
    calls = torch.zeros(max(g.m, 1), dtype=torch.int32, device=frontier.device)
    n_out = c_int64(0)
    cap = _frontier_edges(g, frontier, False) + 1 if capacity is None else int(capacity)
    out = torch.empty(max(cap, 1), dtype=torch.int32, device=frontier.device)
    _check(lib().ess_advance_unique_probe(ctx.handle, g.handle, LOAD_BALANCE[lb], _p(frontier), int(frontier.numel()),
                                          _p(out), cap, byref(n_out), _p(calls), modulus),
           "ess_advance_unique_probe")
    return _probe_output("ess_advance_unique_probe", out, cap, n_out.value, calls)


def filter_probe(ctx: Context, g: Graph, items, alg: str = "predicated", modulus: int = 3, in_place: bool = False):
    """operators::filter::execute with the header's fixed test operator. Returns (output, per-id call counts)."""
    import torch
    _need_cuda(items)
    calls = torch.zeros(max(g.n, 1), dtype=torch.int32, device=items.device)
    out = items if in_place else torch.empty(max(items.numel(), 1), dtype=torch.int32, device=items.device)
    n_out = c_int64(0)
    _check(lib().ess_filter_probe(ctx.handle, g.handle, FILTER[alg], _p(items), int(items.numel()), _p(out),
                                  byref(n_out), _p(calls), modulus), "ess_filter_probe")
    return out[: n_out.value], calls


def uniquify_probe(ctx: Context, g: Graph, items):
    """operators::uniquify::execute<unique>: ascending duplicate-free valid ids."""
    import torch
    out = torch.empty(max(min(int(items.numel()), g.n), 1), dtype=torch.int32, device=items.device)
    cnt = c_int64(0)
    _check(lib().ess_uniquify_probe(ctx.handle, g.handle, _p(items), int(items.numel()), _p(out), byref(cnt)),
           "ess_uniquify_probe")
    return out[: cnt.value]


ATOMIC_OPS = {"add": 0, "min": 1, "max": 2, "exch": 3}


def atomic_probe(ctx: Context, op: str, cell, values, serial: bool = False):
    """math::atomic::<op>(cell, values[i]) for every i; returns the OLD values each call saw (cell is updated in
    place). float32 or int32 tensors."""
    import torch
    _need_cuda(cell, values)
    assert cell.dtype == values.dtype and cell.dtype in (torch.float32, torch.int32) and cell.numel() == 1
    old = torch.empty_like(values)
    _check(lib().ess_atomic_probe(ctx.handle, ATOMIC_OPS[op], int(cell.dtype == torch.float32), _p(cell), _p(values),
                                  int(values.numel()), _p(old), int(serial)), "ess_atomic_probe")
    return old


def frontier_to_bitmap(ctx: Context, items, universe: int):
    import torch
    words = torch.empty((universe + 31) // 32 + 1, dtype=torch.int32, device=items.device)
    pop = c_int64(0)
    _check(lib().ess_frontier_to_bitmap(ctx.handle, _p(items), int(items.numel()), universe, _p(words), byref(pop)),
           "ess_frontier_to_bitmap")
    return words[: (universe + 31) // 32], pop.value


def bitmap_to_frontier(ctx: Context, words, universe: int):
    import torch
    out = torch.empty(max(universe, 1), dtype=torch.int32, device=words.device)
    cnt = c_int64(0)
    _check(lib().ess_bitmap_to_frontier(ctx.handle, _p(words), universe, _p(out), byref(cnt)),
           "ess_bitmap_to_frontier")
    return out[: cnt.value]


def transpose(g_csr):
    """CSR -> CSC on the device by counting sort (ess_transpose_csr)."""
    import torch
    from .graphgen import CSR
    n, m = int(g_csr.offsets.numel() - 1), int(g_csr.indices.numel())
    bits = 64 if g_csr.offsets.element_size() == 8 else 32
    off = torch.empty_like(g_csr.offsets)
    idx = torch.empty_like(g_csr.indices)
    val = None if g_csr.values is None else torch.empty_like(g_csr.values)
    _check(lib().ess_transpose_csr(n, m, bits, _p(g_csr.offsets), _p(g_csr.indices), _p(g_csr.values), _p(off),
                                   _p(idx), _p(val)), "ess_transpose_csr")
    return CSR(n, m, off, idx, val, g_csr.name + "-T", g_csr.symmetric)
