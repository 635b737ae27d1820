"""Python entry points of the B200-native rLap augmentor.

`approximate_cholesky` keeps the signature and the [E',3] float64 (row, col, weight) result of
the reference's rlap.ops.approximate_cholesky (rlap/ops.py:7-58); `identity` mirrors
rlap/ops.py:61-63. New: `prepare` / `schur_views` / `approximate_cholesky_batched` produce many
independent views (or the views of a batch of graphs) in one call, device resident.

All compute runs in the hand-written CUDA kernels behind the C ABI (include/rlap_b200.h); there is
no CPU implementation in this package. CPU tensors are accepted like in the reference: they are
copied to the current CUDA device and the result is returned on the input's device.
"""
import ctypes
import itertools
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch
from torch import Tensor

from . import _native

_O_V = ["random", "degree", "coarsen"]
_O_N = ["asc", "desc", "random"]

_seed_counter = itertools.count()
_base_seed = None
_DEBUG_FLAGS = 0   # profiling bits (128: barrier wait timers, 512: per-round prints); only a -DRLAP_DEBUG build of the library reads them


def manual_seed(seed: int) -> None:
    """Seed the stream of default per-call seeds (the reference has no seed control: it draws its
    permutations from std::random_device, preconditioner.cc:594)."""
    global _base_seed, _seed_counter
    _base_seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    _seed_counter = itertools.count()


def _next_seed() -> int:
    base = _base_seed if _base_seed is not None else (torch.initial_seed() & 0xFFFFFFFFFFFFFFFF)
    k = next(_seed_counter)
    # splitmix64 of (base, call index)
    z = (base + 0x9E3779B97F4A7C15 * (k + 1)) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("rlap_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


class Graph:
    """A coalesced, validated graph resident on the GPU (int32 ids, fp32 weights): what
    EdgeInfoMatrixReader::Read + the symmetry check leave behind in the reference
    (reader.cc:42-61, factorizers.cc:18-22). Shared, read-only, by every view taken from it."""

    def __init__(self, n, nnz, ptr, col, w, graph_ptr, device):
        self.n, self.nnz, self.ptr, self.col, self.w = n, nnz, ptr, col, w
        self.graph_ptr = graph_ptr
        self.device = device

    @property
    def num_graphs(self) -> int:
        return int(self.graph_ptr.shape[0] - 1)


def prepare(edge_index: Tensor, edge_weights: Optional[Tensor], num_nodes: int,
            graph_ptr: Optional[Union[Tensor, np.ndarray, Sequence[int]]] = None, validate: bool = True) -> Graph:
    """COO -> coalesced CSR on the device. Zero weights are dropped, duplicate edges summed, the
    adjacency must be symmetric (ValueError otherwise; the reference exit(0)s the process).
    graph_ptr (optional) splits the vertex range into independent graphs (a PyG-style batch)."""
    assert edge_index.shape[0] == 2
    dev = _require_cuda() if not edge_index.is_cuda else edge_index.device
    L = _native.lib()
    with torch.cuda.device(dev):
        ei = edge_index.to(device=dev, dtype=torch.int64).contiguous()
        E = int(ei.shape[1])
        w = None
        if edge_weights is not None:
            w = edge_weights.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
            assert w.numel() == E, "edge_weights must have one entry per edge"
        n = int(num_nodes)
        ptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
        col = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        cw = torch.empty(max(E, 1), dtype=torch.float32, device=dev)
        wsb = ctypes.c_size_t(0)
        _native.check(L.rlap_ingest_workspace_bytes(n, E, ctypes.byref(wsb)), "ingest_workspace_bytes")
        ws = torch.empty(wsb.value, dtype=torch.uint8, device=dev)
        nnz = ctypes.c_int64(0)
        st = L.rlap_ingest(ei[0].data_ptr(), ei[1].data_ptr(), 0 if w is None else w.data_ptr(), E, n,
                           ptr.data_ptr(), col.data_ptr(), cw.data_ptr(), ctypes.byref(nnz),
                           0 if validate else _native.FLAG_NO_VALIDATE, ws.data_ptr(), wsb.value, _stream_ptr())
        if st in (2, 3, 4, 9):
            raise ValueError("rlap_b200: " + L.rlap_status_string(st).decode())
        _native.check(st, "ingest")
    if graph_ptr is None:
        gp = np.array([0, n], dtype=np.int64)
    else:
        gp = np.ascontiguousarray(graph_ptr.detach().cpu().numpy() if isinstance(graph_ptr, Tensor) else graph_ptr,
                                  dtype=np.int64)
        assert gp[0] == 0 and gp[-1] == n, "graph_ptr must start at 0 and end at num_nodes"
    return Graph(n, int(nnz.value), ptr, col[: max(int(nnz.value), 1)], cw[: max(int(nnz.value), 1)], gp, dev)


def _keep_mask(keep, n: int, device) -> Tensor:
    """keep as a device uint8 [n] of 0 / 1; ValueError for a mask of another length, shape or dtype (a bool or integer
    mask with values other than 0 and 1 included)"""
    if isinstance(keep, Tensor):
        k = keep.detach()
    else:
        a = np.asarray(keep)
        if a.dtype.kind not in "biu":
            raise ValueError(f"keep must be a bool or 0/1 mask, got dtype {a.dtype}")
        k = torch.from_numpy(np.ascontiguousarray(a))
    if k.dtype != torch.bool and (k.is_floating_point() or k.is_complex()):
        raise ValueError(f"keep must be a bool or 0/1 mask, got dtype {k.dtype}")
    if k.dim() != 1 or k.shape[0] != n:
        raise ValueError(f"keep must have one entry per node ({n}), got shape {tuple(k.shape)}")
    k = k.to(device=device)
    if k.dtype != torch.bool:
        if n > 0 and bool(((k != 0) & (k != 1)).any()):
            raise ValueError("keep must be a bool or 0/1 mask")
    return k.to(torch.uint8).contiguous()


def schur_views(graph: Graph, num_remove, o_v: str, o_n: str, num_views: int = 1, seed: Optional[int] = None,
                view_base: int = 0, full_clique: bool = False, shared_order: bool = False, dtype=torch.float64,
                pool_cap: int = 0, scratch_cap: int = 0, return_stats: bool = False, colptr: bool = False,
                check_live: bool = False, weights: bool = True, relabel: bool = False, keep=None):
    """num_views independent randomized Schur-complement views of `graph`.

    Returns (edge_info, view_ptr): edge_info is [sum E'_v, 3] (row, col, weight) of `dtype`
    (float64 like the reference, or None for the packed form), views back to back, each sorted by
    (col, row); view_ptr is a host int64 tensor [num_views + 1]. With dtype=None returns
    ((row int32, col int32, w float32), view_ptr). num_remove: int or one value per graph.
    colptr=True (with dtype=None): the `col` array is replaced by the per-view column pointers, an int32 tensor
    [num_views, n + 1] (rows of a view are sorted by column, so col is implied; `expand_cols` rebuilds it on the
    host) - a third less to move for consumers behind a PCIe link. weights=False (with dtype=None): no weight array
    is written (w is None): the unweighted view the reference's GCL adapters keep.
    relabel=True: survivor compaction + relabelling inside the emission (what the reference's adapters do afterwards
    with torch.unique + subgraph(relabel_nodes=True), scripts/augmentor_benchmarks.py:149-155): the row / col ids of
    view v are ranks among that view's vertices with at least one edge, and the call returns one more value, `newid`
    int32 [num_views, n] (-1 for vertices without edges; `(newid[v] >= 0).nonzero()` is the sorted node list).
    keep: a bool or 0/1 mask of length n (tensor on any device, array or sequence), or None. A marked vertex is
    protected: no view eliminates it, and a graph with a protected vertex may lose every other vertex (num_remove is
    capped at its number of unprotected vertices instead of n_g - 1). With full_clique=True and num_remove >= that
    number the views are the exact Schur complement onto the protected set (a Kron reduction)."""
    assert o_v in _O_V
    assert o_n in _O_N
    L = _native.lib()
    dev = graph.device
    G = graph.num_graphs
    nr = np.ascontiguousarray(np.broadcast_to(np.asarray(num_remove, dtype=np.int64), (G,)))
    if seed is None:
        seed = _next_seed()
    flags = (_native.FLAG_FULL_CLIQUE if full_clique else 0) | (_native.FLAG_SHARED_ORDER if shared_order else 0)
    flags |= _native.FLAG_CHECK_LIVE if check_live else 0
    flags |= _DEBUG_FLAGS
    V = int(num_views)
    kmask = None if keep is None else _keep_mask(keep, graph.n, dev)
    if kmask is not None:
        flags |= _native.FLAG_KEEP
    if full_clique:  # test mode: cliques instead of trees, multi-edges pile up until a vertex goes
        pool_cap = pool_cap or 8 * graph.nnz + 4096
        scratch_cap = scratch_cap or (1 << 18)
    with torch.cuda.device(dev):
        stream = _stream_ptr()
        while True:
            wsb = ctypes.c_size_t(0)
            _native.check(L.rlap_schur_workspace_bytes(graph.n, graph.nnz, G, V, pool_cap, scratch_cap, flags, ctypes.byref(wsb)),
                          "schur_workspace_bytes")
            ws = torch.empty(wsb.value, dtype=torch.uint8, device=dev)
            rows = np.zeros(V, dtype=np.int64)
            stats = np.zeros(16, dtype=np.int64)
            args = (graph.n, graph.nnz, graph.ptr.data_ptr(), graph.col.data_ptr(), graph.w.data_ptr(), G,
                    graph.graph_ptr.ctypes.data, nr.ctypes.data, _native.OV[o_v], _native.ON[o_n],
                    seed & 0xFFFFFFFFFFFFFFFF, view_base, V, flags, pool_cap, scratch_cap, ws.data_ptr(), wsb.value,
                    rows.ctypes.data, stats.ctypes.data)
            if kmask is None:
                st = L.rlap_schur_eliminate(*args, stream)
            else:
                st = L.rlap_schur_eliminate_keep(*args, kmask.data_ptr(), stream)
            if st == _native.RLAP_ERR_POOL_OVERFLOW:
                pool_cap = 2 * int(stats[6])
                del ws
                continue
            if st == _native.RLAP_ERR_STAR_TOO_LARGE and scratch_cap < graph.nnz + 1:
                scratch_cap = graph.nnz + 1      # a star never holds more entries than the graph
                del ws
                continue
            _native.check(st, "schur_eliminate")
            break
        total = int(rows.sum())
        view_ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(rows)]).astype(np.int64))
        newid, nid_ptr = None, 0
        if relabel:
            newid = torch.empty(V * graph.n + 1, dtype=torch.int32, device=dev)
            _native.check(L.rlap_schur_relabel(graph.n, graph.nnz, V, ws.data_ptr(), wsb.value, newid.data_ptr(), 0, stream),
                          "schur_relabel")
            nid_ptr = newid.data_ptr()
        if dtype is None:
            orow = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
            ow = torch.empty(max(total, 1), dtype=torch.float32, device=dev) if weights else None
            if colptr:
                ocp = torch.empty((V, graph.n + 1), dtype=torch.int32, device=dev)
                _native.check(L.rlap_schur_colptr(graph.n, graph.nnz, V, ws.data_ptr(), wsb.value, ocp.data_ptr(), stream),
                              "schur_colptr")
            else:
                ocol = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
            _native.check(L.rlap_schur_emit_ids(graph.n, graph.nnz, graph.ptr.data_ptr(), graph.col.data_ptr(),
                                                graph.w.data_ptr(), V, ws.data_ptr(), wsb.value, orow.data_ptr(),
                                                0 if colptr else ocol.data_ptr(), ow.data_ptr() if weights else 0, 0,
                                                nid_ptr, stream), "schur_emit")
            out = (orow[:total], ocp if colptr else ocol[:total], ow[:total] if weights else None)
        else:
            o64 = torch.empty((max(total, 1), 3), dtype=torch.float64, device=dev)
            _native.check(L.rlap_schur_emit_ids(graph.n, graph.nnz, graph.ptr.data_ptr(), graph.col.data_ptr(),
                                                graph.w.data_ptr(), V, ws.data_ptr(), wsb.value, 0, 0, 0, o64.data_ptr(),
                                                nid_ptr, stream), "schur_emit")
            out = o64[:total]
            if dtype != torch.float64:
                out = out.to(dtype)
        # the library forgets the workspace before its memory goes back to the allocator
        L.rlap_schur_release(ws.data_ptr())
    if relabel:
        out = (out, newid[: V * graph.n].view(V, graph.n))
    if return_stats:
        names = ["rounds", "fills", "pool_used_max", "max_star", "raw_entries_read", "rows", "pool_cap", "elim_us",
                 "emit_count_us", "t_init_us", "t_phaseA_us", "t_phaseB_us", "t_phaseC_us", "t_elim_warp_us",
                 "t_elim_block_us", "check_mismatches"]
        return out, view_ptr, dict(zip(names, (int(x) for x in stats)))
    return out, view_ptr


def expand_cols(colptr_host: Tensor, view_ptr: Tensor, out: Optional[Tensor] = None, threads: int = 8) -> Tensor:
    """host side of schur_views(colptr=True): the int32 `col` array of the packed rows, rebuilt from a HOST copy of
    the column pointers [num_views, n + 1] and view_ptr with `threads` host threads (C, no Python loop)."""
    assert not colptr_host.is_cuda and colptr_host.dtype == torch.int32 and colptr_host.is_contiguous()
    V, n1 = colptr_host.shape
    vp = view_ptr.to(torch.int64).contiguous()
    total = int(vp[-1])
    if out is None:
        out = torch.empty(max(total, 1), dtype=torch.int32)
    assert out.dtype == torch.int32 and out.numel() >= total and out.is_contiguous()
    _native.check(_native.lib().rlap_expand_cols_host(colptr_host.data_ptr(), V, n1 - 1, vp.data_ptr(), out.data_ptr(),
                                                      int(threads)), "expand_cols_host")
    return out[:total]


def approximate_cholesky_batched(edge_index: Tensor, edge_weights: Optional[Tensor], num_nodes: int, num_remove,
                                 o_v: str, o_n: str, num_views: int = 1, graph_ptr=None, seed: Optional[int] = None,
                                 dtype=torch.float64, keep=None, **kw) -> Tuple[Tensor, Tensor]:
    """Batched variant: `num_views` views of one graph, or of every graph of a batch (graph_ptr),
    in one call. Returns (edge_info [sum E', 3], view_ptr [num_views + 1]). keep: protected vertices, as in
    schur_views."""
    g = prepare(edge_index, edge_weights, num_nodes, graph_ptr=graph_ptr)
    out, vp = schur_views(g, num_remove, o_v, o_n, num_views=num_views, seed=seed, dtype=dtype, keep=keep, **kw)
    if not edge_index.is_cuda and dtype is not None:
        out = out.to(edge_index.device)
    return out, vp


def approximate_cholesky(
    edge_index: Tensor,
    edge_weights: Optional[Tensor],
    num_nodes: int,
    num_remove: int,
    o_v: str,
    o_n: str,
    seed: Optional[int] = None,
    keep=None,
) -> Tensor:
    """
    Compute the randomized Schur complement of the graph Laplacian (same contract as the
    reference's rlap.ops.approximate_cholesky, rlap/ops.py:7-58).

    Parameters:
    -----------
    edge_index : Tensor [2, E] of node ids (both directions of every edge present).
    edge_weights : Tensor [E] or [1, E] of edge weights, or None for unit weights.
    num_nodes : total number of nodes.
    num_remove : number of nodes to eliminate (capped at num_nodes - 1, or at the number of unprotected nodes when
        keep marks at least one node).
    o_v : elimination order, one of ["random", "degree", "coarsen"].
    o_n : neighbour order, one of ["asc", "desc", "random"].
    seed : optional 64-bit seed (extension; the reference is unseedable).
    keep : optional bool or 0/1 mask of length num_nodes (extension): marked nodes are never eliminated.

    Returns:
    --------
    Tensor [E', 3] float64: rows (row, col, weight) of the sampled Schur complement over the
    surviving nodes, original node ids, both directions present, on edge_index's device.
    """
    assert edge_index.shape[0] == 2
    assert o_v in _O_V
    assert o_n in _O_N
    g = prepare(edge_index, edge_weights, num_nodes)
    out, _ = schur_views(g, int(num_remove), o_v, o_n, num_views=1, seed=seed, dtype=torch.float64, keep=keep)
    return out.to(edge_index.device)


def approximate_cholesky_host(edge_info: np.ndarray, num_nodes: int, num_remove: int, o_v: str, o_n: str,
                              seed: int = 0) -> np.ndarray:
    """Host-buffer call through rlap_approximate_cholesky_host: the exact shape of the reference's
    approximate_cholesky_cpu (py_api_binder.cc:54-69), [E,3] float64 in, [E',3] float64 out, all
    copies inside."""
    _require_cuda()
    L = _native.lib()
    ei = np.ascontiguousarray(edge_info, dtype=np.float64)
    assert ei.ndim == 2 and ei.shape[1] == 3
    out = ctypes.POINTER(ctypes.c_double)()
    rows = ctypes.c_int64(0)
    st = L.rlap_approximate_cholesky_host(ei.ctypes.data, ei.shape[0], num_nodes, num_remove, o_v.encode(),
                                          o_n.encode(), seed & 0xFFFFFFFFFFFFFFFF, ctypes.byref(out), ctypes.byref(rows))
    if st in (2, 3, 4, 9):
        raise ValueError("rlap_b200: " + L.rlap_status_string(st).decode())
    _native.check(st, "approximate_cholesky_host")
    res = np.ctypeslib.as_array(out, shape=(max(rows.value, 1), 3))[: rows.value].copy()
    L.rlap_free_host(out)
    return res


def identity(a: Tensor) -> Tensor:
    """Verification op of the reference (rlap/ops.py:61-63: a Torch -> Eigen -> Torch round trip).
    Here the boundary carries plain buffers, so the round trip is device -> device copy."""
    return a.clone()
