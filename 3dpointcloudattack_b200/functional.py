"""PyTorch autograd Functions over the C ABI of libpcdist.so (include/pcdist.h).

PyTorch is plumbing here: it owns device memory, the current stream and autograd; every
arithmetic step of the path runs in the hand-written sm_100a kernels.  Nothing in this
module computes a distance with torch ops and nothing falls back to CPU.
"""
from __future__ import annotations

import contextlib
import ctypes
import math
from collections import namedtuple

import torch

from . import _lib
from ._lib import (EDGE_CENTER, EDGE_DIFF, EDGE_NEIGHBOR, FORM_COL_ROW, FORM_ROW_COL, FORM_SUM_FIRST, NORM_FMA, NORM_MULSUM,
                   VALUE_SQRT_CLAMP, VALUE_SQUARED)

__all__ = ["nn1", "NN1Result", "time_next_sweep", "clear_cache", "knn", "ball_query", "edge_feature", "deterministic_edge_backward", "clip_points_", "lp_clip", "offset_proj", "find_offset", "farthest_point_sample", "fp32_peak_flops",
           "local_frames", "kappa", "graph_laplacian", "knn_outlier_loss", "sor", "SORResult", "sample_points", "PointSampler", "nn_dist64", "NNDist64Result",
           "shape_invariant_step_", "estimate_normals", "SI_STEP_SCALE", "si_sensitivity", "si_query_round_", "low_pass",
           "EDGE_CENTER", "EDGE_NEIGHBOR", "EDGE_DIFF",
           "FORM_ROW_COL", "FORM_COL_ROW", "FORM_SUM_FIRST", "NORM_MULSUM", "NORM_FMA",
           "VALUE_SQUARED", "VALUE_SQRT_CLAMP"]

_launch_count = 0   # number of C-ABI compute calls issued (bench.py reports launches)


def launches():
    return _launch_count


def _check_cloud(t, name, C=3):
    if not isinstance(t, torch.Tensor) or t.dim() != 3:
        raise ValueError(f"{name} must be a 3-D tensor [B, N, {C}] (a transposed view is fine)")
    if not t.is_cuda:
        raise RuntimeError(f"{name} is on {t.device}: this path runs on CUDA only (no CPU fallback)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if C is not None and t.shape[2] != C:
        raise ValueError(f"{name} must have {C} channels in its last logical dim, got {tuple(t.shape)}")


def _cloud_args(t):
    return [t.data_ptr(), t.stride(0), t.stride(1), t.stride(2)]


def _stream(dev=None):
    """raw cudaStream_t of the current stream (torch.cuda.current_stream() builds a Stream object: ~20 us per call)"""
    idx = torch.cuda.current_device() if dev is None or dev.index is None else dev.index
    return torch._C._cuda_getCurrentRawStream(idx)


_NULLCTX = contextlib.nullcontext()


def _on(dev):
    """device guard only when the tensor's device is not the current one (the guard costs ~10 us)"""
    if dev.index is None or torch.cuda.current_device() == dev.index:
        return _NULLCTX
    return torch.cuda.device(dev)


def _ptr(t):
    return None if t is None else t.data_ptr()


# ----------------------------------------------------------------------------------- NN-1
NN1Result = namedtuple("NN1Result", "row_min row_arg col_min col_arg row_sum row_max col_sum col_max "
                                    "row_argmax col_argmax")
# row_* : minima over the columns j for every row i (and their per-sample scaled sum / max / first argmax)
# col_* : minima over the rows i for every column j


class _Token:
    """Marks a cached NN-1 result whose autograd graph has been consumed by backward()."""
    __slots__ = ("consumed",)

    def __init__(self):
        self.consumed = False


_tiling = (0, 0)          # (rows per lane, column tile) override for the next calls; (0, 0) = heuristic (tests / tuning)
_sweep_events = None     # (start, stop) torch.cuda.Event pair consumed by the next _NN1.forward (bench.py's roofline)


def time_next_sweep(start_event, stop_event):
    """Measurement helper: the next nn1() call on this thread records the two torch.cuda.Event
    objects immediately before / after its sweep kernel launch (passed per call through the C ABI;
    the library itself keeps no state).  The event between the kernels costs that call the
    programmatic overlap of the chain, nothing else."""
    global _sweep_events
    _sweep_events = None if start_event is None else (start_event, stop_event)


def force_tiling(rows_per_lane=0, col_tile=0):
    """Tests / tuning sweeps: force the sweep's tile shape for the following nn1() calls (0, 0 = heuristic)."""
    global _tiling
    _tiling = (int(rows_per_lane), int(col_tile))


class _NN1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rows, cols, form, norm, swap_norms, transform, row_scale, col_scale, token):
        global _launch_count, _sweep_events
        lib = _lib.load()
        B, N, _ = rows.shape
        M = cols.shape[1]
        dev = rows.device
        need_r, need_c = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        ev, _sweep_events = _sweep_events, None
        with _on(dev):
            row_min = torch.empty((B, N), dtype=torch.float32, device=dev)
            col_min = torch.empty((B, M), dtype=torch.float32, device=dev)
            row_arg = torch.empty((B, N), dtype=torch.int32, device=dev)
            col_arg = torch.empty((B, M), dtype=torch.int32, device=dev)
            stats = torch.empty((4, B), dtype=torch.float32, device=dev)
            stats_i = torch.empty((2, B), dtype=torch.int32, device=dev)
            ws_bytes = lib.pcd_nn1_workspace_bytes(B, N, M, 0)
            ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
            # gradient buffers of the coming backward: the forward's last kernel clears them on the way, so the
            # backward is ONE launch (atomics into zeroed memory) instead of memset + memset + kernel
            grad_rows = torch.empty((B, N, 3), dtype=torch.float32, device=dev) if need_r and (B * N * 3) % 4 == 0 else None
            grad_cols = torch.empty((B, M, 3), dtype=torch.float32, device=dev) if need_c and (B * M * 3) % 4 == 0 else None
            st = lib.pcd_nn1_forward(*_cloud_args(rows), *_cloud_args(cols), B, N, M,
                                     form, norm, int(swap_norms), transform, row_scale, col_scale,
                                     row_min.data_ptr(), row_arg.data_ptr(), col_min.data_ptr(), col_arg.data_ptr(),
                                     stats.data_ptr(), stats_i.data_ptr(),
                                     _ptr(grad_rows), 0 if grad_rows is None else grad_rows.numel(),
                                     _ptr(grad_cols), 0 if grad_cols is None else grad_cols.numel(),
                                     ws.data_ptr(), ws_bytes, _tiling[0], _tiling[1], 0,
                                     None if ev is None else ev[0].cuda_event, None if ev is None else ev[1].cuda_event,
                                     _stream(dev))
            _lib.check(st, "pcd_nn1_forward")
        _launch_count += 3
        ctx.save_for_backward(rows, cols, row_arg, col_arg, row_min, col_min, stats_i)
        ctx.cfg = (int(swap_norms), transform, row_scale, col_scale)
        ctx.token = token
        ctx.zeroed = [grad_rows, grad_cols]      # valid for ONE backward (retain_graph re-runs allocate afresh)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(row_arg, col_arg, stats_i)
        return row_min, row_arg, col_min, col_arg, stats[0], stats[1], stats[2], stats[3], stats_i

    @staticmethod
    def backward(ctx, g_row_min, _ga, g_col_min, _gb, g_row_sum, g_row_max, g_col_sum, g_col_max, _gc):
        global _launch_count
        rows, cols, row_arg, col_arg, row_min, col_min, stats_i = ctx.saved_tensors
        swap_norms, transform, row_scale, col_scale = ctx.cfg
        ctx.token.consumed = True          # the graph is (normally) freed after this: never serve it again
        need_r, need_c = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (need_r or need_c):
            return (None,) * 9
        lib = _lib.load()
        B, N, _ = rows.shape
        M = cols.shape[1]
        dev = rows.device
        with _on(dev):
            c = lambda t: None if t is None else t.contiguous()
            g_row, g_col = c(g_row_min), c(g_col_min)
            # [B] upstream gradients are read through their stride: autograd hands out expanded
            # (stride 0) views for sum()/mean() and we do not want a copy kernel per gradient
            w = [g_row_sum, g_row_max, g_col_sum, g_col_max]
            w_strides = (ctypes.c_int64 * 4)(*[0 if t is None else t.stride(0) for t in w])
            zr, zc = ctx.zeroed
            ctx.zeroed = [None, None]
            prezeroed = (not need_r or zr is not None) and (not need_c or zc is not None)
            grad_rows = (zr if prezeroed else torch.empty((B, N, 3), dtype=torch.float32, device=dev)) if need_r else None
            grad_cols = (zc if prezeroed else torch.empty((B, M, 3), dtype=torch.float32, device=dev)) if need_c else None
            gr = _cloud_args(grad_rows) if need_r else [None, 0, 0, 0]
            gc = _cloud_args(grad_cols) if need_c else [None, 0, 0, 0]
            st = lib.pcd_nn1_backward(*_cloud_args(rows), *_cloud_args(cols), B, N, M, swap_norms, transform,
                                      row_arg.data_ptr(), col_arg.data_ptr(), row_min.data_ptr(), col_min.data_ptr(),
                                      _ptr(g_row), _ptr(g_col),
                                      _ptr(w[0]), _ptr(w[1]), stats_i[0].data_ptr(),
                                      _ptr(w[2]), _ptr(w[3]), stats_i[1].data_ptr(),
                                      w_strides, row_scale, col_scale, *gr, *gc, int(prezeroed), _stream(dev))
            _lib.check(st, "pcd_nn1_backward")
        _launch_count += 1
        return grad_rows, grad_cols, None, None, None, None, None, None, None


_nn1_cache = {"key": None, "val": None, "refs": None, "token": None}


def _tensor_key(t):
    # identity of the autograd root (the base of a view), storage, version counter and geometry:
    # two `x.permute(0, 2, 1)` views of the same unmodified x hit the same entry.
    root = t._base if t._is_view() else t
    return (id(root), t.data_ptr(), t._version, tuple(t.shape), tuple(t.stride()), t.requires_grad)


def nn1(rows, cols, form, norm, swap_norms=False, transform=VALUE_SQUARED, row_sum_scale=1.0,
        col_sum_scale=1.0, cache=True) -> NN1Result:
    """One NN-1 sweep of every sample: row/column minima of d(i,j), lowest-index argmins and
    per-sample (scaled) sum / max (see pcd_nn1_forward in include/pcdist.h).

    rows [B,N,3], cols [B,M,3]: fp32 CUDA tensors, any strides (pass `x.transpose(1, 2)` for a
    channel-first [B,3,N] cloud).  A one-entry cache returns the previous result when called
    again with the very same tensors (same storage, same version counter) and mode -- the
    reference's losses recompute the same adv->ori nearest neighbours up to six times per
    iteration (attack/GeoA3/GeoA3_attack.py:134-166, Chamfer then Hausdorff in CW).

    The cache is only consulted while an autograd graph is being recorded (grad mode on and one
    of the clouds requires grad) and its entry dies with the first backward() through it: one
    entry = one forward pass of one iteration.  Under no_grad nothing is cached -- in-place
    writes through `.data` (the clip / projection steps of the attack loops) do not bump the
    version counter, so a cached no_grad result could be stale.  Code that mutates a cloud
    through `.data` BETWEEN two calls inside the same recorded forward must call clear_cache().
    """
    _check_cloud(rows, "rows"); _check_cloud(cols, "cols")
    if rows.shape[0] != cols.shape[0]:
        raise ValueError("rows and cols must have the same batch dimension.")
    if rows.device != cols.device:
        raise ValueError("rows and cols must be on the same device")
    if rows.shape[1] == 0 or cols.shape[1] == 0 or rows.shape[0] == 0:
        raise ValueError("empty clouds are not supported (the reference's min() raises as well)")
    key = None
    cache = cache and torch.is_grad_enabled() and (rows.requires_grad or cols.requires_grad)
    if cache:
        key = (_tensor_key(rows), _tensor_key(cols), form, norm, bool(swap_norms), transform,
               float(row_sum_scale), float(col_sum_scale))
        if _nn1_cache["key"] == key and not _nn1_cache["token"].consumed:
            return _nn1_cache["val"]
    token = _Token()
    out = _NN1.apply(rows, cols, form, norm, bool(swap_norms), transform, float(row_sum_scale),
                     float(col_sum_scale), token)
    res = NN1Result(out[0], out[1], out[2], out[3], out[4], out[5], out[6], out[7], out[8][0], out[8][1])
    if cache:
        _nn1_cache["key"] = key
        _nn1_cache["val"] = res
        _nn1_cache["refs"] = (rows, cols)      # keeps the ids in the key from being recycled
        _nn1_cache["token"] = token
    return res


def clear_cache():
    _nn1_cache["key"] = None
    _nn1_cache["val"] = None
    _nn1_cache["refs"] = None
    _nn1_cache["token"] = None


# -------------------------------------------------------------------------------- k-NN
KNN_AUTO, KNN_BOUND_SELECT, KNN_SELECT_ONLY = 0, 1, 2
_knn_strategy = KNN_AUTO


def force_knn_strategy(strategy=KNN_AUTO):
    """Tests / tuning: pick the xyz k-NN pipeline of the following calls explicitly (pcd_knn_strategy in include/pcdist.h)."""
    global _knn_strategy
    _knn_strategy = int(strategy)


class _KNN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rows, cols, K, form, norm, swap_norms, want_dists):
        global _launch_count
        lib = _lib.load()
        B, N, C = rows.shape
        M = cols.shape[1]
        dev = rows.device
        with _on(dev):
            dists = torch.empty((B, N, K), dtype=torch.float32, device=dev)
            idx = torch.empty((B, N, K), dtype=torch.int32, device=dev)
            ws_bytes = lib.pcd_knn_workspace_bytes(B, N, M, C, K)
            ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev)
            st = lib.pcd_knn_forward(*_cloud_args(rows), *_cloud_args(cols), B, N, M, C, K,
                                     form, norm, int(swap_norms), dists.data_ptr(), idx.data_ptr(),
                                     ws.data_ptr(), ws_bytes, _knn_strategy, _stream(dev))
            _lib.check(st, "pcd_knn_forward")
        _launch_count += 2
        ctx.save_for_backward(rows, cols, idx)
        ctx.cfg = (int(swap_norms), K)
        ctx.mark_non_differentiable(idx)
        return dists, idx

    @staticmethod
    def backward(ctx, g_dists, _gi):
        global _launch_count
        rows, cols, idx = ctx.saved_tensors
        swap_norms, K = ctx.cfg
        need_r, need_c = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if g_dists is None or not (need_r or need_c):
            return (None,) * 7
        B, N, C = rows.shape
        M = cols.shape[1]
        if C != 3:
            raise NotImplementedError("gradients of k-NN distances are provided for 3-channel clouds only "
                                      "(the reference differentiates kNN distances on xyz only)")
        lib = _lib.load()
        dev = rows.device
        with _on(dev):
            g = g_dists.contiguous()
            grad_rows = torch.empty((B, N, 3), dtype=torch.float32, device=dev) if need_r else None
            grad_cols = torch.empty((B, M, 3), dtype=torch.float32, device=dev) if need_c else None
            gr = _cloud_args(grad_rows) if need_r else [None, 0, 0, 0]
            gc = _cloud_args(grad_cols) if need_c else [None, 0, 0, 0]
            st = lib.pcd_knn_backward(*_cloud_args(rows), *_cloud_args(cols), B, N, M, K, swap_norms,
                                      idx.data_ptr(), g.data_ptr(), *gr, *gc, _stream(dev))
            _lib.check(st, "pcd_knn_backward")
        _launch_count += 2
        return grad_rows, grad_cols, None, None, None, None, None


def knn(rows, cols, K, form=FORM_COL_ROW, norm=NORM_MULSUM, swap_norms=False):
    """K smallest d(i,j) per row, ascending by (distance, index): (dists[B,N,K] fp32,
    idx[B,N,K] int32).  rows [B,N,C], cols [B,M,C] with 1 <= C <= 128 (any strides)."""
    _check_cloud(rows, "rows", C=None); _check_cloud(cols, "cols", C=None)
    if rows.shape[0] != cols.shape[0]:
        raise ValueError("rows and cols must have the same batch dimension.")
    if rows.shape[2] != cols.shape[2]:
        raise ValueError("rows and cols must have the same point dimension.")
    K = int(K)
    if not 1 <= K <= min(cols.shape[1], _lib.KNN_MAX_K):
        raise ValueError(f"K={K} out of range: need 1 <= K <= min(M={cols.shape[1]}, {_lib.KNN_MAX_K})")
    if not 1 <= rows.shape[2] <= _lib.KNN_MAX_C:
        raise ValueError(f"C={rows.shape[2]} out of range 1..{_lib.KNN_MAX_C}")
    return _KNN.apply(rows, cols, K, form, norm, bool(swap_norms), True)


# --------------------------------------------------------------------------- ball query
def ball_query(radius, nsample, xyz, new_xyz):
    """model/pointnet2_utils.py:84-104 semantics -> idx [B,S,nsample] int32."""
    global _launch_count
    _check_cloud(xyz, "xyz"); _check_cloud(new_xyz, "new_xyz")
    lib = _lib.load()
    B, N, _ = xyz.shape
    S = new_xyz.shape[1]
    dev = xyz.device
    with _on(dev):
        idx = torch.empty((B, S, int(nsample)), dtype=torch.int32, device=dev)
        r2 = torch.tensor(float(radius) ** 2, dtype=torch.float32).item()   # fp32(radius**2), as the reference compares
        st = lib.pcd_ball_query(*_cloud_args(xyz.detach()), *_cloud_args(new_xyz.detach()), B, N, S, r2,
                                int(nsample), idx.data_ptr(), _stream(dev))
        _lib.check(st, "pcd_ball_query")
    _launch_count += 1
    return idx


# ------------------------------------------------ k-NN graph edge features, farthest point sampling
_edge_bwd_gather = False


def deterministic_edge_backward(enabled=True):
    """Select the backward of edge_feature.  False (default): scatter with shared-memory atomics, 3.4 TB/s, summation
    order not fixed (as the reference's index backward).  True: gather over the inverted graph, the same bits on every
    run, ~1.8x the time of that kernel (shapes the gather form does not cover -- N > 4096, 4 not dividing N*k -- fall
    back to the atomics).  Returns the previous setting."""
    global _edge_bwd_gather
    prev, _edge_bwd_gather = _edge_bwd_gather, bool(enabled)
    return prev


class _EdgeFeature(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, idx, ops):
        global _launch_count
        lib = _lib.load()
        B, C, N = x.shape
        k = idx.shape[2]
        dev = x.device
        c_ops = (ctypes.c_int * len(ops))(*ops)
        with _on(dev):
            out = torch.empty((B, len(ops) * C, N, k), dtype=torch.float32, device=dev)
            st = lib.pcd_edge_feature_forward(x.data_ptr(), idx.data_ptr(), B, C, N, k, len(ops), c_ops,
                                              out.data_ptr(), _stream(dev))
            _lib.check(st, "pcd_edge_feature_forward")
        _launch_count += 1
        ctx.save_for_backward(idx)
        ctx.cfg = (ops, C)
        return out

    @staticmethod
    def backward(ctx, g):
        global _launch_count
        if g is None or not ctx.needs_input_grad[0]:
            return None, None, None
        (idx,) = ctx.saved_tensors
        ops, C = ctx.cfg
        lib = _lib.load()
        B, _, N, k = g.shape
        dev = g.device
        c_ops = (ctypes.c_int * len(ops))(*ops)
        with _on(dev):
            g = g.contiguous()
            gx = torch.empty((B, C, N), dtype=torch.float32, device=dev)
            # gather form (inverted graph in a workspace) where the shape allows it, else shared-memory atomics
            ws_bytes = int(lib.pcd_edge_feature_backward_workspace(B, N, k, len(ops))) if _edge_bwd_gather else 0
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
            st = lib.pcd_edge_feature_backward(g.data_ptr(), idx.data_ptr(), B, C, N, k, len(ops), c_ops,
                                               gx.data_ptr(), ws.data_ptr() if ws_bytes else None, ws_bytes, _stream(dev))
            _lib.check(st, "pcd_edge_feature_backward")
        _launch_count += 2 if ws_bytes else 1
        return gx, None, None


def edge_feature(x, idx, ops):
    """Edge features of a k-NN graph (pcd_edge_feature_forward in include/pcdist.h):
    x [B,C,N] fp32 channel-first, idx [B,N,k] integer with entries in [0,N), ops a tuple of
    EDGE_CENTER / EDGE_NEIGHBOR / EDGE_DIFF -> out [B, len(ops)*C, N, k]; differentiable in x."""
    if not isinstance(x, torch.Tensor) or x.dim() != 3:
        raise ValueError("x must be a 3-D tensor [B, C, N]")
    if not x.is_cuda:
        raise RuntimeError(f"x is on {x.device}: this path runs on CUDA only (no CPU fallback)")
    if x.dtype != torch.float32:
        raise TypeError(f"x must be float32, got {x.dtype}")
    if idx.dim() != 3 or idx.shape[0] != x.shape[0] or idx.shape[1] != x.shape[2]:
        raise ValueError(f"idx must be [B, N, k] matching x {tuple(x.shape)}, got {tuple(idx.shape)}")
    ops = tuple(int(o) for o in ops)
    if not 1 <= len(ops) <= 4 or any(o not in (EDGE_CENTER, EDGE_NEIGHBOR, EDGE_DIFF) for o in ops):
        raise ValueError("ops must hold 1..4 of EDGE_CENTER / EDGE_NEIGHBOR / EDGE_DIFF")
    idx32 = idx.detach().to(device=x.device, dtype=torch.int32).contiguous()
    return _EdgeFeature.apply(x.contiguous(), idx32, ops)


def farthest_point_sample(xyz, npoint, start=None):
    """model/pointnet2_utils.py:59-81 as one persistent CTA per sample (pcd_fps): xyz [B,N,3]
    (any strides), start [B] integer tensor or None (= index 0, model/curvenet_util.py:81)
    -> centroids [B,npoint] int32 with centroids[:,0] = start."""
    global _launch_count
    _check_cloud(xyz, "xyz")
    lib = _lib.load()
    B, N, _ = xyz.shape
    npoint = int(npoint)
    if npoint < 1:
        raise ValueError("npoint must be >= 1")
    dev = xyz.device
    with _on(dev):
        st32 = None if start is None else start.detach().to(device=dev, dtype=torch.int32).contiguous()
        out = torch.empty((B, npoint), dtype=torch.int32, device=dev)
        x = xyz.detach()
        st = lib.pcd_fps(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2), B, N, npoint, _ptr(st32),
                         out.data_ptr(), _stream(dev))
        _lib.check(st, "pcd_fps")
    _launch_count += 1
    return out


# ------------------------------------------------ k-NN outlier / smoothing loss with a fused epilogue
class _KnnOutlierLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pc, k, alpha, form, norm, swap_norms):
        global _launch_count
        lib = _lib.load()
        B, N, _ = pc.shape
        dev = pc.device
        K1 = k + 1
        with _on(dev):
            x = pc.detach()
            dists = torch.empty((B, N, K1), dtype=torch.float32, device=dev)
            idx = torch.empty((B, N, K1), dtype=torch.int32, device=dev)
            ws_bytes = lib.pcd_knn_workspace_bytes(B, N, N, 3, K1)
            ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev)
            st = lib.pcd_knn_forward(*_cloud_args(x), *_cloud_args(x), B, N, N, 3, K1, form, norm, int(swap_norms),
                                     dists.data_ptr(), idx.data_ptr(), ws.data_ptr(), ws_bytes, _knn_strategy, _stream(dev))
            _lib.check(st, "pcd_knn_forward")
            value = torch.empty((B, N), dtype=torch.float32, device=dev)
            mask = torch.empty((B, N), dtype=torch.float32, device=dev)
            loss = torch.empty((B,), dtype=torch.float32, device=dev)
            thr = torch.empty((B,), dtype=torch.float32, device=dev)
            grad = torch.empty((B, N, 3), dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
            st = lib.pcd_knn_outlier_forward(dists.data_ptr(), B, N, K1, 1, float(alpha), value.data_ptr(), mask.data_ptr(),
                                             loss.data_ptr(), thr.data_ptr(), _ptr(grad), _stream(dev))
            _lib.check(st, "pcd_knn_outlier_forward")
        _launch_count += 3
        ctx.zeroed = grad                           # valid for ONE backward
        ctx.save_for_backward(pc, idx, mask)
        ctx.mark_non_differentiable(value, mask, thr)
        return loss, value, mask, thr

    @staticmethod
    def backward(ctx, g_loss, _gv, _gm, _gt):
        global _launch_count
        if g_loss is None or not ctx.needs_input_grad[0]:
            return (None,) * 6
        pc, idx, mask = ctx.saved_tensors
        lib = _lib.load()
        B, N, _ = pc.shape
        dev = pc.device
        with _on(dev):
            grad, ctx.zeroed = ctx.zeroed, None
            pre = grad is not None
            if not pre:
                grad = torch.empty((B, N, 3), dtype=torch.float32, device=dev)
            st = lib.pcd_knn_outlier_backward(*_cloud_args(pc), idx.data_ptr(), mask.data_ptr(), g_loss.data_ptr(), g_loss.stride(0),
                                              B, N, idx.shape[2], 1, grad.data_ptr(), int(pre), _stream(dev))
            _lib.check(st, "pcd_knn_outlier_backward")
        _launch_count += 1
        return grad, None, None, None, None, None


def knn_outlier_loss(pc, k, alpha, form=FORM_COL_ROW, norm=NORM_MULSUM, swap_norms=False):
    """Self k-NN select + fused outlier-loss epilogue (pcd_knn_outlier_forward in include/pcdist.h):
    pc [B,N,3] (any strides) -> (loss [B] differentiable, value [B,N], mask [B,N], threshold [B])."""
    _check_cloud(pc, "pc")
    k = int(k)
    if not 1 <= k + 1 <= min(pc.shape[1], _lib.KNN_MAX_K):
        raise ValueError(f"k={k} out of range for N={pc.shape[1]}")
    return _KnnOutlierLoss.apply(pc, k, float(alpha), form, norm, bool(swap_norms))


# ------------------------------------------------ statistical outlier removal (SOR defence), float64
SORResult = namedtuple("SORResult", "value threshold keep kept_idx lengths")
# value [B,N] f64 mean distance to the k nearest neighbours; threshold [B] f64; keep [B,N] bool;
# kept_idx [B,N] int64 kept point indices ascending, then -1; lengths [B] int64 number of kept points


def sor(pc, k=2, alpha=1.1, lengths=None, col_split=0):
    """Statistical outlier removal in float64 (pcd_sor_forward_len in include/pcdist.h; the statistic of
    attack/SIadv/baselines/defense/drop_points/SOR.py:24-54): pc [B,N,3] fp32 (any strides) -> SORResult.
    lengths: None (all N points) or an integer tensor [B]; sample i is pc[i, :lengths[i]], clamped to [0, N] on the
    device.  A sample with fewer than k + 1 points has no statistic: NaN values and threshold, nothing kept.  Rows past
    a sample's length get value NaN, keep False.  col_split > 0 forces the number of column ranges per row tile
    (testing and tuning only; results do not change).  Two kernels (three when the columns are split), no host
    synchronisation; pc is detached (the statistic carries no gradient)."""
    value, thr, keep, kept, kept_n = _sor32(pc, k, alpha, lengths, col_split)
    return SORResult(value, thr, keep.view(torch.bool), kept.long(), kept_n.long())


def _sor32(pc, k, alpha, lengths, col_split=0):
    """sor's launches -> (value, threshold, keep uint8, kept_idx int32, lengths int32), the C ABI's types"""
    global _launch_count
    _check_cloud(pc, "pc")
    k, alpha = int(k), float(alpha)
    B, N, _ = pc.shape
    if not 1 <= k <= _lib.SOR_MAX_K or (lengths is None and N < k + 1):
        raise ValueError(f"SOR needs 1 <= k <= {_lib.SOR_MAX_K} and N >= k + 1, got k={k}, N={N}")
    if not math.isfinite(alpha):
        raise ValueError(f"alpha must be finite, got {alpha}")
    if B == 0:
        raise ValueError("pc holds no sample")
    if N == 0:
        raise ValueError("pc holds no point")
    col_split = int(col_split)
    if col_split < 0:
        raise ValueError(f"col_split must be >= 0, got {col_split}")
    lib = _lib.load()
    dev = pc.device
    with _on(dev):
        x = pc.detach()
        len32 = _lengths32(lengths, B, N, "lengths", dev)
        value = torch.empty((B, N), dtype=torch.float64, device=dev)
        thr = torch.empty((B,), dtype=torch.float64, device=dev)
        keep = torch.empty((B, N), dtype=torch.uint8, device=dev)
        kept = torch.empty((B, N), dtype=torch.int32, device=dev)
        kept_n = torch.empty((B,), dtype=torch.int32, device=dev)
        ws_bytes = lib.pcd_sor_workspace_bytes(B, N, k, col_split)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
        st = lib.pcd_sor_forward_len(*_cloud_args(x), B, N, k, alpha, _ptr(len32), col_split, value.data_ptr(),
                                     thr.data_ptr(), keep.data_ptr(), kept.data_ptr(), kept_n.data_ptr(), _ptr(ws),
                                     ws_bytes, _stream(dev))
        _lib.check(st, "pcd_sor_forward_len")
    _launch_count += 3 if ws_bytes else 2       # a workspace means split columns: the merge is one more launch
    return value, thr, keep, kept, kept_n


def sample_points(n, N, npoint, sampler, table=None):
    """Uniform draws without replacement, per sample, on the device (pcd_sample_points in include/pcdist.h): the
    resampling of SORDefense.process_data and the SRS defence, without numpy and without a host synchronisation.
    n: None (N points in every sample) or an integer tensor [B] of valid counts, clamped to [0, N] on the device;
    N: the padded size; sampler: a PointSampler (seed, first_sample, device-side draw counter).  -> int64 [B, npoint]:
      n > npoint  npoint distinct points in random order    (np.random.choice(n, npoint, replace=False))
      n < npoint  arange(n) npoint // n times, then npoint % n distinct points in random order
      n == npoint arange(n);  n == 0  -1 everywhere
    table: None or an integer tensor [B, >= N] (SOR's kept_idx): every drawn value v becomes table[b, v].  B is n's
    length, or table's when n is None.  One launch; the sampler's counter advances by one in stream order, so the call
    is graph-capturable and a replayed graph draws afresh.  The draws follow numpy's in distribution, not its bits."""
    global _launch_count
    if not isinstance(sampler, PointSampler):
        raise TypeError(f"sampler must be a PointSampler, got {type(sampler).__name__}")
    N, npoint = int(N), int(npoint)
    if n is None and table is None:
        raise ValueError("sample_points needs n or table to know the batch size")
    B = int(n.shape[0]) if n is not None else int(table.shape[0])
    if B < 1 or N < 1 or npoint < 1:
        raise ValueError(f"sample_points needs B, N, npoint >= 1, got B={B}, N={N}, npoint={npoint}")
    if N > _lib.SAMPLE_MAX_N:
        raise ValueError(f"sample_points supports N <= {_lib.SAMPLE_MAX_N}, got N={N}")
    dev = sampler.state.device
    if table is not None:
        if not isinstance(table, torch.Tensor) or table.dim() != 2 or table.shape[0] != B or table.shape[1] < N \
                or table.dtype.is_floating_point or table.dtype == torch.bool:
            raise ValueError(f"table must be an integer tensor [{B}, >= {N}], got {table!r:.80}")
        if table.device != dev:
            raise ValueError(f"table is on {table.device} and the sampler on {dev}")
        if table.dtype != torch.int32 or table.stride(1) != 1:
            table = table.to(torch.int32).contiguous()
    lib = _lib.load()
    with _on(dev):
        len32 = _lengths32(n, B, N, "n", dev)
        out = torch.empty((B, npoint), dtype=torch.int64, device=dev)
        st = lib.pcd_sample_points(B, N, npoint, _ptr(len32), _ptr(table), table.stride(0) if table is not None else 0,
                                   sampler.seed, sampler.first_sample, sampler.state.data_ptr(), out.data_ptr(),
                                   _stream(dev))
        _lib.check(st, "pcd_sample_points")
    _launch_count += 1
    return out


class PointSampler:
    """Seed and device-side draw counter of sample_points.  Draw c of global sample first_sample + b is a pure function
    of (seed, first_sample + b, c, n, npoint), so a run sharded over ranks (each with the first_sample of its shard)
    draws what the unsharded run draws, as sharding.per_sample_noise does for the initial noise.
    state: int64 [2] on the device; state[0] is the draw counter (each sample_points call adds one, on the stream),
    state[1] scratch of the kernel (0 between calls)."""

    def __init__(self, seed, first_sample=0, device=None):
        seed, first_sample = int(seed), int(first_sample)
        if not 0 <= seed < 2 ** 64:
            raise ValueError(f"seed must be in [0, 2**64), got {seed}")
        if first_sample < 0:
            raise ValueError(f"first_sample must be >= 0, got {first_sample}")
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if device.type != "cuda":
            raise RuntimeError(f"PointSampler on {device}: the sampler runs on CUDA only (no CPU fallback)")
        self.seed, self.first_sample = seed, first_sample
        self.state = torch.zeros(2, dtype=torch.int64, device=device)

    @property
    def counter(self):
        """the draw counter: a 0-d view of state[0] on the device"""
        return self.state[0]

    def reset(self, counter=0):
        """set the draw counter (stream-ordered; no synchronisation)"""
        self.state[0].fill_(int(counter))
        self.state[1].zero_()
        return self


# ------------------------------------------------ exact float64 nearest-neighbour distances (Chamfer / Hausdorff metrics)
NNDist64Result = namedtuple("NNDist64Result", "a_min a_arg b_min b_arg a_mean_sq a_mean a_max_sq a_max a_argmax "
                                              "b_mean_sq b_mean b_max_sq b_max b_argmax")
# a_min [B,N] f64 squared distance of each a point to its nearest valid b point, a_arg [B,N] int64 its index (NaN / -1
# past a's length); b_min / b_arg [B,M] the same from b to a.  Per sample [B], over the valid rows: a_mean_sq = mean of
# a_min, a_mean = mean of sqrt(a_min), a_max_sq = max of a_min, a_max = sqrt(a_max_sq), a_argmax = its first index; b_*
# the same for b.


def _lengths32(lengths, B, n, name, dev):
    if lengths is None:
        return None
    if not isinstance(lengths, torch.Tensor) or lengths.dtype.is_floating_point or lengths.dtype.is_complex \
            or lengths.dtype == torch.bool or tuple(lengths.shape) != (B,):
        raise ValueError(f"{name} must be None or an integer tensor of shape ({B},), got {lengths!r:.80}")
    lengths = lengths.detach().to(dev)
    if lengths.dtype != torch.int32:
        lengths = lengths.clamp(0, n).to(torch.int32)     # clamped first: a cast alone would wrap values past 2^31
    return lengths.contiguous()


def nn_dist64(a, b, a_lengths=None, b_lengths=None, col_split=0):
    """Exact float64 nearest-neighbour distances between a [B,N,3] and b [B,M,3] fp32 (any strides), both directions,
    with per-sample means and maxima (pcd_nn_dist64_forward in include/pcdist.h) -> NNDist64Result.
    a_lengths / b_lengths: None (all points) or an integer tensor [B]; sample i uses a[i, :a_lengths[i]] and
    b[i, :b_lengths[i]], clamped to [0, N] / [0, M] on the device.  Two kernels, no host synchronisation, no autograd.
    col_split > 0 forces the number of column ranges per row tile (testing and tuning only; results do not change)."""
    global _launch_count
    _check_cloud(a, "a")
    _check_cloud(b, "b")
    if a.device != b.device:
        raise ValueError(f"a is on {a.device} and b on {b.device}")
    B, N, _ = a.shape
    M = b.shape[1]
    if b.shape[0] != B:
        raise ValueError(f"a and b hold {B} and {b.shape[0]} samples")
    if B == 0 or N == 0 or M == 0:
        raise ValueError(f"nn_dist64 needs B, N, M >= 1, got B={B}, N={N}, M={M}")
    col_split = int(col_split)
    if col_split < 0:
        raise ValueError(f"col_split must be >= 0, got {col_split}")
    lib = _lib.load()
    dev = a.device
    with _on(dev):
        la = _lengths32(a_lengths, B, N, "a_lengths", dev)
        lb = _lengths32(b_lengths, B, M, "b_lengths", dev)
        a_min = torch.empty((B, N), dtype=torch.float64, device=dev)
        a_arg = torch.empty((B, N), dtype=torch.int32, device=dev)
        b_min = torch.empty((B, M), dtype=torch.float64, device=dev)
        b_arg = torch.empty((B, M), dtype=torch.int32, device=dev)
        stats = torch.empty((2, B, 4), dtype=torch.float64, device=dev)
        argmax = torch.empty((2, B), dtype=torch.int32, device=dev)
        ws_bytes = lib.pcd_nn_dist64_workspace_bytes(B, N, M, col_split)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        st = lib.pcd_nn_dist64_forward(*_cloud_args(a.detach()), *_cloud_args(b.detach()), B, N, M, _ptr(la), _ptr(lb),
                                       col_split, a_min.data_ptr(), a_arg.data_ptr(), b_min.data_ptr(), b_arg.data_ptr(),
                                       stats.data_ptr(), argmax.data_ptr(), ws.data_ptr(), ws_bytes, _stream(dev))
        _lib.check(st, "pcd_nn_dist64_forward")
        argmax = argmax.long()
        res = NNDist64Result(a_min, a_arg.long(), b_min, b_arg.long(), *stats[0].unbind(1), argmax[0],
                             *stats[1].unbind(1), argmax[1])
    _launch_count += 2
    return res


# ------------------------------------------------ local geometry on a k-NN graph (SURVEY 8f row 4)
def _idx32(idx, dev):
    return idx.detach().to(device=dev, dtype=torch.int32).contiguous()


def local_frames(pc, idx, skip_first=True, normals=True, frames=False):
    """Per-point covariance eigen-frame of the k-NN patch (pcd_local_frames in include/pcdist.h;
    attack/GeoA3/utility.py:43-92, :119-152).  pc [B,N,3] fp32 (any strides), idx [B,N,K1] integer
    (self-kNN of pc; column 0 is dropped when skip_first) -> (normal [B,N,3] or None,
    evecs [B,N,3,3] rows by ascending eigenvalue or None, evals [B,N,3] or None).  No gradient."""
    global _launch_count
    _check_cloud(pc, "pc")
    lib = _lib.load()
    B, N, _ = pc.shape
    dev = pc.device
    idx32 = _idx32(idx, dev)
    if idx32.dim() != 3 or idx32.shape[:2] != (B, N):
        raise ValueError(f"idx must be [B, N, K], got {tuple(idx32.shape)} for pc {tuple(pc.shape)}")
    K1 = idx32.shape[2]
    if K1 - int(bool(skip_first)) < 1:
        raise ValueError("need at least one neighbour")
    with _on(dev):
        normal = torch.empty((B, N, 3), dtype=torch.float32, device=dev) if normals else None
        evecs = torch.empty((B, N, 3, 3), dtype=torch.float32, device=dev) if frames else None
        evals = torch.empty((B, N, 3), dtype=torch.float32, device=dev) if frames else None
        x = pc.detach()
        st = lib.pcd_local_frames(*_cloud_args(x), idx32.data_ptr(), B, N, K1, int(bool(skip_first)),
                                  _ptr(normal), *([normal.stride(0), normal.stride(1), normal.stride(2)] if normals else [0, 0, 0]),
                                  _ptr(evecs), _ptr(evals), _stream(dev))
        _lib.check(st, "pcd_local_frames")
    _launch_count += 1
    return normal, evecs, evals


class _Kappa(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pc, normal, nidx, idx, skip_first):
        global _launch_count
        lib = _lib.load()
        B, N, _ = pc.shape
        dev = pc.device
        with _on(dev):
            kappa = torch.empty((B, N), dtype=torch.float32, device=dev)
            st = lib.pcd_kappa_forward(*_cloud_args(pc), *_cloud_args(normal), _ptr(nidx), idx.data_ptr(), B, N, idx.shape[2],
                                       int(skip_first), kappa.data_ptr(), _stream(dev))
            _lib.check(st, "pcd_kappa_forward")
        _launch_count += 1
        ctx.save_for_backward(pc, normal, idx)
        ctx.nidx, ctx.skip_first = nidx, skip_first
        return kappa

    @staticmethod
    def backward(ctx, g):
        global _launch_count
        if g is None or not ctx.needs_input_grad[0]:
            return None, None, None, None, None
        pc, normal, idx = ctx.saved_tensors
        lib = _lib.load()
        B, N, _ = pc.shape
        dev = pc.device
        with _on(dev):
            grad = torch.empty((B, N, 3), dtype=torch.float32, device=dev)
            g = g.contiguous()
            st = lib.pcd_kappa_backward(*_cloud_args(pc), *_cloud_args(normal), _ptr(ctx.nidx), idx.data_ptr(), B, N, idx.shape[2],
                                        int(ctx.skip_first), g.data_ptr(), grad.data_ptr(), _stream(dev))
            _lib.check(st, "pcd_kappa_backward")
        _launch_count += 2
        return grad, None, None, None, None


def kappa(pc, normal, idx, nidx=None, skip_first=True):
    """mean_j |<unit(q_j - p_i), n>| over the k-NN patch (pcd_kappa_forward; loss_utils.py:60-90, :116-125).
    pc [B,N,3] (any strides, differentiable), normal [B,N,3] (any strides, constant), idx [B,N,K1] self-kNN of pc,
    nidx [B,N] optional: take the normal of point nidx[b,i] instead of i (the adv->ori neighbour) -> [B,N]."""
    _check_cloud(pc, "pc"); _check_cloud(normal, "normal")
    if pc.shape != normal.shape:
        raise ValueError("pc and normal must have the same shape")
    dev = pc.device
    idx32 = _idx32(idx, dev)
    if idx32.dim() != 3 or idx32.shape[:2] != pc.shape[:2]:
        raise ValueError(f"idx must be [B, N, K], got {tuple(idx32.shape)}")
    n32 = None if nidx is None else _idx32(nidx.reshape(pc.shape[0], pc.shape[1]), dev)
    return _Kappa.apply(pc, normal.detach(), n32, idx32, bool(skip_first))


def graph_laplacian(pc, idx):
    """Dense L = D - A of the symmetrised k-NN graph with Gaussian weights (pcd_graph_laplacian;
    attack/AOF/TAOF_attack.py:31-52 up to the eigensolver).  pc [B,N,3] (any strides), idx [B,N,K] -> [B,N,N]."""
    global _launch_count
    _check_cloud(pc, "pc")
    lib = _lib.load()
    B, N, _ = pc.shape
    dev = pc.device
    idx32 = _idx32(idx, dev)
    if idx32.dim() != 3 or idx32.shape[:2] != (B, N):
        raise ValueError(f"idx must be [B, N, K], got {tuple(idx32.shape)}")
    with _on(dev):
        L = torch.empty((B, N, N), dtype=torch.float32, device=dev)
        x = pc.detach()
        st = lib.pcd_graph_laplacian(*_cloud_args(x), idx32.data_ptr(), B, N, idx32.shape[2], L.data_ptr(), _stream(dev))
        _lib.check(st, "pcd_graph_laplacian")
    _launch_count += 3
    return L


def fp32_peak_flops(iters=2048):
    """Measured fp32 FMA peak of the current device (FLOP/s) -- roofline denominator: the larger of
    the scalar-FFMA and packed-FFMA2 probe kernels, best of three timed launches each (CUDA events)."""
    lib = _lib.load()
    scratch = torch.empty(64, dtype=torch.float32, device="cuda")
    flop = ctypes.c_double(0.0)
    best = 0.0
    for variant in (0, 1):
        for rep in range(4):                                  # first = warm-up
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st = lib.pcd_fp32_probe_launch(variant, int(iters), scratch.data_ptr(), ctypes.byref(flop), _stream())
            _lib.check(st, "pcd_fp32_probe_launch")
            e1.record()
            e1.synchronize()
            if rep:
                best = max(best, flop.value / (e0.elapsed_time(e1) * 1e-3))
    return best


# ------------------------------------------------ projection / clipping epilogues of the attack loops
CLIP_LINF, CLIP_PROJECT_LINF, CLIP_L2 = 0, 1, 2


def _check_cf(t, name):
    """channel-first contiguous fp32 CUDA cloud [B,3,K]"""
    if not isinstance(t, torch.Tensor) or t.dim() != 3 or t.shape[1] != 3:
        raise ValueError(f"{name} must be a [B, 3, K] tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} is on {t.device}: this path runs on CUDA only (no CPU fallback)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def clip_points_(pc, ori, budget, mode=CLIP_LINF, normal=None):
    """IN PLACE clip of the perturbation pc - ori (pcd_clip_points in include/pcdist.h): CLIP_LINF = ClipPointsLinf,
    CLIP_PROJECT_LINF = ProjectInnerClipLinf (needs normal), CLIP_L2 = ClipPointsL2 (clip_utils.py:5-136).
    pc, ori, normal: [B,3,K] fp32 contiguous.  Returns pc.  Not differentiable (the reference clips under no_grad)."""
    global _launch_count
    _check_cf(pc, "pc"); _check_cf(ori, "ori")
    if ori.shape != pc.shape or ori.device != pc.device:
        raise ValueError("pc and ori must have the same shape and device")
    if mode == CLIP_PROJECT_LINF:
        if normal is None:
            raise ValueError("CLIP_PROJECT_LINF needs the normals")
        _check_cf(normal, "normal")
        if normal.shape != pc.shape or normal.device != pc.device:
            raise ValueError("normal must match pc")
    lib = _lib.load()
    B, _, K = pc.shape
    with _on(pc.device):
        st = lib.pcd_clip_points(pc.data_ptr(), ori.data_ptr(), _ptr(normal) if mode == CLIP_PROJECT_LINF else None, B, K,
                                 int(mode), float(budget), _stream(pc.device))
        _lib.check(st, "pcd_clip_points")
    _launch_count += 1
    return pc


def lp_clip(offset, cc_linf):
    """attack/GeoA3/GeoA3_attack.py:92-101 as one launch (pcd_lp_clip): offset [B,3,K] -> clipped copy.  No gradient."""
    global _launch_count
    _check_cf(offset, "offset")
    lib = _lib.load()
    B, _, K = offset.shape
    with _on(offset.device):
        out = torch.empty_like(offset)
        st = lib.pcd_lp_clip(offset.data_ptr(), B, K, float(cc_linf), out.data_ptr(), _stream(offset.device))
        _lib.check(st, "pcd_lp_clip")
    _launch_count += 1
    return out


def _offset_gather(fn_name, a, table, idx):
    global _launch_count
    _check_cf(a, "offset"); _check_cf(table, "table")
    B, _, K = a.shape
    M = table.shape[2]
    idx32 = _idx32(idx, a.device).reshape(B, -1)
    if table.shape[0] != B or idx32.shape[1] != K or table.device != a.device:
        raise ValueError(f"shapes do not match: {tuple(a.shape)}, {tuple(table.shape)}, idx {tuple(idx.shape)}")
    lib = _lib.load()
    with _on(a.device):
        out = torch.empty_like(a)
        st = getattr(lib, fn_name)(a.data_ptr(), table.data_ptr(), idx32.data_ptr(), B, K, M, out.data_ptr(), _stream(a.device))
        _lib.check(st, fn_name)
    _launch_count += 1
    return out


def offset_proj(offset, ori_normal, idx):
    """GeoA3_attack.py:62-81 after its knn_points(K=1) (pcd_offset_proj): offset [B,3,K], ori_normal [B,3,M],
    idx [B,K] or [B,K,1] integer (nearest original point) -> projected offsets [B,3,K].  No gradient."""
    return _offset_gather("pcd_offset_proj", offset, ori_normal, idx)


def find_offset(adv, ori, idx):
    """GeoA3_attack.py:83-89 after its knn_points(K=1) (pcd_find_offset): adv - ori[:, :, idx].  No gradient."""
    return _offset_gather("pcd_find_offset", adv, ori, idx)


# ------------------------------------------------ the SI-Adv shape-invariant step and the normals it re-estimates
SI_STEP_SCALE = math.sqrt(3 * 1024)     # the reference's hard-coded step scale (SIadv_attack.py), whatever N is


def shape_invariant_step_(pc, ori, normal, grad, step_size, eps, step_scale=SI_STEP_SCALE, split=0):
    """One step of SI-Adv's shape_invariant_ifgm IN PLACE on pc (pcd_si_step in include/pcdist.h; get_spin_axis_matrix,
    get_transformed_point_cloud, get_original_point_cloud of attack/SIadv/SIadv_attack.py): the gradient restricted to
    every point's tangent plane, normalised over the sample, a step of step_size * step_scale against it, and the
    reference's clip of the perturbation to eps, which on [B,N,3] clouds bounds each axis's norm over the whole cloud.
    pc, ori, normal, grad [B,N,3] fp32 (any strides; grad = dL/d pc; the projection g - (g.n)n does not depend on the
    sign of the normal).  -> gnorm [B], the per-sample norm of the tangent gradient.  One launch, no gradient, no host
    synchronisation.  split > 0 forces the CTAs per sample (testing; the results do not change)."""
    global _launch_count
    for t, name in ((pc, "pc"), (ori, "ori"), (normal, "normal"), (grad, "grad")):
        _check_cloud(t, name)
        if t.shape != pc.shape or t.device != pc.device:
            raise ValueError(f"{name} {tuple(t.shape)} on {t.device} does not match pc {tuple(pc.shape)} on {pc.device}")
    B, N, _ = pc.shape
    if not 1 <= N <= _lib.SI_MAX_N:
        raise ValueError(f"shape_invariant_step_ supports 1 <= N <= {_lib.SI_MAX_N}, got N={N}")
    if not float(eps) >= 0:
        raise ValueError(f"eps must be >= 0, got {eps}")
    split = int(split)
    if split < 0 or split > _lib.SI_MAX_SPLIT or split & (split - 1):
        raise ValueError(f"split must be 0 or a power of two <= {_lib.SI_MAX_SPLIT}, got {split}")
    if any(t.data_ptr() == pc.data_ptr() for t in (ori, normal, grad)) and B:
        raise ValueError("pc is updated in place and must not alias ori, normal or grad")
    lib = _lib.load()
    dev = pc.device
    with _on(dev):
        gnorm = torch.empty((B,), dtype=torch.float32, device=dev)
        st = lib.pcd_si_step(*_cloud_args(pc), *_cloud_args(ori), *_cloud_args(normal), *_cloud_args(grad), B, N,
                             float(step_size), float(step_scale), float(eps), split, gnorm.data_ptr(), _stream(dev))
        _lib.check(st, "pcd_si_step")
    torch.autograd.graph.increment_version(pc)      # written through its pointer: autograd must see the change
    _launch_count += 1
    return gnorm


def estimate_normals(pc, k=20):
    """Unit normals [B,N,3] of pc [B,N,3] (any strides): the eigenvector of the smallest eigenvalue of the covariance of
    each point's k nearest neighbours, the point itself included (knn, then local_frames with skip_first=False; three
    launches, no gradient).  It stands in for SI-Adv's get_normal_vector (open3d estimate_normals with
    KDTreeSearchParamKNN(knn=20) on the host).  The sign of a normal and the order among neighbours at equal distance
    are this library's, not open3d's; every consumer here is sign-free."""
    _check_cloud(pc, "pc")
    k = int(k)
    if not 2 <= k <= min(pc.shape[1], _lib.KNN_MAX_K):
        raise ValueError(f"k={k} out of range: need 2 <= k <= min(N={pc.shape[1]}, {_lib.KNN_MAX_K})")
    x = pc.detach()
    with torch.no_grad():
        _, idx = knn(x, x, k)
    return local_frames(x, idx, skip_first=False)[0]


# ------------------------------------------------ SI-Adv's query-based attack: the sensitivity map and one query round
def si_sensitivity(grad, normal):
    """The sensitivity map of SI-Adv's query-based attack (pcd_si_sensitivity in include/pcdist.h): grad (a surrogate's
    dL/d cloud) and normal [B,N,3] fp32 (any strides) -> (order int32 [B,N]: the points by descending tangent-gradient
    length, ties by the lower index; dir [B,N,2]: the unit tangent direction of each point's gradient in its frame).
    A point whose length is NaN ranks last with dir (0, 0).  One launch, then a stable torch.sort; no gradient."""
    global _launch_count
    for t, name in ((grad, "grad"), (normal, "normal")):
        _check_cloud(t, name)
    if normal.shape != grad.shape or normal.device != grad.device:
        raise ValueError(f"normal {tuple(normal.shape)} on {normal.device} does not match grad {tuple(grad.shape)} on "
                         f"{grad.device}")
    B, N, _ = grad.shape
    if N < 1:
        raise ValueError("si_sensitivity needs N >= 1")
    lib = _lib.load()
    dev = grad.device
    with _on(dev):
        s = torch.empty((B, N), dtype=torch.float32, device=dev)
        dir = torch.empty((B, N, 2), dtype=torch.float32, device=dev)
        st = lib.pcd_si_sensitivity(*_cloud_args(grad.detach()), *_cloud_args(normal.detach()), B, N, s.data_ptr(),
                                    dir.data_ptr(), _stream(dev))
        _lib.check(st, "pcd_si_sensitivity")
        order = torch.sort(s, dim=1, descending=True, stable=True)[1].to(torch.int32)
    _launch_count += 1
    return order, dir


def si_query_round_(logits, target, ori, normal, order, dir, cloud, trial, state, best, step_size, eps, max_query,
                    targeted=False, active=None):
    """One round of SI-Adv's query-based attack for every sample, IN PLACE on cloud, trial, state, best and active
    (pcd_si_query_round in include/pcdist.h), after the black box has scored the trials: logits [B,C] fp32 (any
    strides, C >= 2), target [B] int64.  Each active sample takes or rejects its trial, and the next trial moves one point
    of the cloud by +-step_size in its tangent plane, clipped to eps.
    ori, normal, cloud, trial [B,N,3] fp32 (any strides); order int32 [B,N] and dir [B,N,2] from si_sensitivity;
    state int32 [B,4] = (sigma, cursor, queries, status: 0 active, 1 success, 2 failed), best [B] fp32; active: None or
    an int32 [1] tensor that every sample ending in this round decrements.  One launch, no host synchronisation."""
    global _launch_count
    for t, name in ((ori, "ori"), (normal, "normal"), (cloud, "cloud"), (trial, "trial")):
        _check_cloud(t, name)
        if t.shape != ori.shape or t.device != ori.device:
            raise ValueError(f"{name} {tuple(t.shape)} on {t.device} does not match ori {tuple(ori.shape)} on {ori.device}")
    B, N, _ = ori.shape
    dev = ori.device
    if not 1 <= N <= _lib.SI_MAX_N:
        raise ValueError(f"si_query_round_ supports 1 <= N <= {_lib.SI_MAX_N}, got N={N}")
    if not isinstance(logits, torch.Tensor) or logits.dim() != 2 or logits.shape[0] != B or logits.shape[1] < 2 \
            or logits.dtype != torch.float32 or logits.device != dev:
        raise ValueError(f"logits must be float32 [{B}, C >= 2] on {dev}, got {logits!r:.80}")
    for t, name, shape, dtype in ((target, "target", (B,), torch.int64), (order, "order", (B, N), torch.int32),
                                  (dir, "dir", (B, N, 2), torch.float32), (state, "state", (B, 4), torch.int32),
                                  (best, "best", (B,), torch.float32)):
        if not isinstance(t, torch.Tensor) or tuple(t.shape) != shape or t.dtype != dtype or t.device != dev \
                or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous {dtype} tensor {shape} on {dev}, got {t!r:.80}")
    if active is not None and (not isinstance(active, torch.Tensor) or active.dtype != torch.int32
                               or active.numel() != 1 or active.device != dev):
        raise ValueError(f"active must be None or an int32 tensor of one element on {dev}")
    if not math.isfinite(float(step_size)) or not float(eps) >= 0 or int(max_query) < 1:
        raise ValueError(f"need a finite step_size, eps >= 0 and max_query >= 1, got {step_size}, {eps}, {max_query}")
    if cloud.data_ptr() == trial.data_ptr() and B:
        raise ValueError("cloud and trial must not be the same memory")
    lib = _lib.load()
    with _on(dev):
        st = lib.pcd_si_query_round(logits.data_ptr(), logits.stride(0), logits.stride(1), logits.shape[1],
                                    target.data_ptr(), *_cloud_args(ori), *_cloud_args(normal), order.data_ptr(),
                                    dir.data_ptr(), *_cloud_args(cloud), *_cloud_args(trial), state.data_ptr(),
                                    best.data_ptr(), B, N, float(step_size), float(eps), int(max_query), int(bool(targeted)),
                                    _ptr(active), _stream(dev))
        _lib.check(st, "pcd_si_query_round")
    for t in (cloud, trial, state, best) + (() if active is None else (active,)):
        torch.autograd.graph.increment_version(t)      # written through its pointer: autograd must see the change
    _launch_count += 1


# ------------------------------------------------ AOF's low-frequency projection
def _low_pass_launch(basis, x, split):
    global _launch_count
    lib = _lib.load()
    B, N, _ = x.shape
    dev = x.device
    with _on(dev):
        y = torch.empty_like(x)                      # x's layout: [B,N,3] or a transposed [B,3,N]
        st = lib.pcd_low_pass(basis.data_ptr(), basis.stride(0), basis.shape[1], *_cloud_args(x), B, N, *_cloud_args(y),
                              split, _stream(dev))
        _lib.check(st, "pcd_low_pass")
    _launch_count += 1
    return y


class _LowPass(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, basis, split):
        ctx.save_for_backward(basis)
        ctx.split = split
        return _low_pass_launch(basis, x.detach(), split)

    @staticmethod
    def backward(ctx, g):
        basis, = ctx.saved_tensors
        return _low_pass_launch(basis, g, ctx.split), None, None    # P = V^T V is symmetric


def low_pass(x, basis, split=None):
    """AOF's low-frequency component y = V^T (V x) per sample and channel (pcd_low_pass in include/pcdist.h):
    x [B,N,3] fp32 (any strides; y has x's layout), basis V [B,Kl,N] fp32 with rows contiguous along N (a sample stride
    of 0, e.g. V.expand(B, -1, -1), shares one basis), 1 <= Kl <= N.  Differentiable in x: the backward is the same
    projection of the incoming gradient, one launch each way; no host synchronisation, so it can be captured in a CUDA
    graph.  The basis gets no gradient.  split forces the CTAs per sample (testing; the results do not change)."""
    _check_cloud(x, "x")
    B, N, _ = x.shape
    if not 1 <= N <= _lib.LP_MAX_N:
        raise ValueError(f"low_pass supports 1 <= N <= {_lib.LP_MAX_N}, got N={N}")
    if not isinstance(basis, torch.Tensor) or basis.dim() != 3 or basis.shape[0] != B or basis.shape[2] != N \
            or not 1 <= basis.shape[1] <= N:
        raise ValueError(f"basis must be [{B}, Kl, {N}] with 1 <= Kl <= {N}, got "
                         f"{tuple(basis.shape) if isinstance(basis, torch.Tensor) else basis!r}")
    if basis.dtype != torch.float32 or basis.device != x.device:
        raise ValueError(f"basis must be float32 on {x.device}, got {basis.dtype} on {basis.device}")
    if basis.stride(2) != 1 or (basis.shape[1] > 1 and basis.stride(1) != N) or basis.stride(0) < 0:
        raise ValueError(f"basis rows must be contiguous along N, got strides {basis.stride()}")
    split = 0 if split is None else int(split)
    if split < 0 or split > _lib.LP_MAX_SPLIT or split & (split - 1):
        raise ValueError(f"split must be None, 0 or a power of two <= {_lib.LP_MAX_SPLIT}, got {split}")
    return _LowPass.apply(x, basis.detach(), split)
