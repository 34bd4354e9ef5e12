"""Drop-in for the reference's `pcdet/ops/pointnet2/pointnet2_batch/pointnet2_utils.py`.

Same public names, positional signatures, return dtypes and autograd behaviour
(reference pointnet2_utils.py:36,65,101,133,181,225,256,287-384); every native call goes through the
C-ABI of include/spsk.h (libspsk.so, hand-written sm_100a CUDA) on torch's current stream.  Differences,
all deliberate: preconditions raise instead of `assert`/`exit(-1)`; kernels are stream-explicit; FPS
keeps its running minima on chip (no `temp` tensor unless n > 131072).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Tuple

import torch
import torch.nn as nn
from torch.autograd import Function

from ._lib import GroupDesc, PwDesc, SaMmaDesc, check, lib

__all__ = [
    "farthest_point_sample", "furthest_point_sample", "furthest_point_sample_with_dist", "gather_operation",
    "three_nn", "three_interpolate", "grouping_operation", "ball_query", "ball_query_dilated",
    "QueryAndGroup", "QueryDilatedAndGroup", "GroupAll",
    "score_topk", "gather_rows", "ball_query_msg",
]

current_ovf_tag = 0   # fp16 range-guard tag stamped on the tensor-core launches (set by the calling module, 0 = untagged)


def fp16_overflow(clear: bool = True) -> int:
    """Bit mask of the modules (tags) whose tensor-core kernels stored a value beyond the fp16 range since the last clear.
    SYNCHRONISES the current device (include/spsk.h: spsk_fp16_overflow_poll)."""
    m = C.c_uint(0)
    check(lib.spsk_fp16_overflow_poll(C.byref(m), 1 if clear else 0), "fp16_overflow_poll")
    return int(m.value)


FPS_DISTMAT_ONCHIP_MAX_N = 16384  # distance-matrix mode (F-FPS) and the forced dense kernels keep 16 minima per thread on chip, no clusters
FPS_ONCHIP_MAX_N = 131072  # <= 16384: one CTA per scene; <= 131072: one 2/4/8-CTA cluster per scene; above: a 16-CTA cluster
# (<= 262144) where the device can schedule one, else the streaming kernel over the `temp` scratch, which is allocated from here on


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def deterministic_grads() -> bool:
    """Backward of gather / group / three_interpolate through the sorted segment reduction (spsk_scatter_grad: no atomics,
    bit-reproducible) instead of the reference-style atomicAdd scatters.  On when torch.use_deterministic_algorithms(True)
    is set or SPSK_DETERMINISTIC_GRAD=1."""
    return torch.are_deterministic_algorithms_enabled() or os.environ.get("SPSK_DETERMINISTIC_GRAD", "0") == "1"


def scatter_grad(grad_out: torch.Tensor, idx: torch.Tensor, n: int, weight: torch.Tensor = None, div: int = 1) -> torch.Tensor:
    """grad_points[b, c, idx[b, l]] += weight[b, l] * grad_out[b, c, l // div] without atomics (include/spsk.h).
    grad_out (B, C, cols) f32, idx (B, L) i32, weight (B, L) f32 or None -> (B, C, n)."""
    B, Cc, cols = grad_out.shape
    L = idx.shape[1]
    out = torch.empty((B, Cc, n), dtype=torch.float32, device=grad_out.device)
    need = int(lib.spsk_scatter_grad_workspace_bytes(B, n, L))
    if need < 0:
        raise RuntimeError("scatter_grad: problem too large")
    ws = torch.empty(max(need, 8), dtype=torch.uint8, device=grad_out.device)
    with torch.cuda.device(grad_out.device):
        check(lib.spsk_scatter_grad(B, Cc, n, L, cols, div, grad_out.data_ptr(), idx.data_ptr(),
                                    weight.data_ptr() if weight is not None else None, out.data_ptr(), ws.data_ptr(),
                                    ws.numel(), _stream()), "scatter_grad")
    return out


def _chk(t: torch.Tensor, name: str, dtype: torch.dtype, ndim: int) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise RuntimeError(f"{name} must be {dtype}, got {t.dtype}")
    if t.dim() != ndim:
        raise RuntimeError(f"{name} must have {ndim} dims, got shape {tuple(t.shape)}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")


class FarthestPointSampling(Function):
    """reference: pointnet2_utils.py:10-33 (FarthestPointSampling)."""

    @staticmethod
    def forward(ctx, xyz: torch.Tensor, npoint: int) -> torch.Tensor:
        _chk(xyz, "xyz", torch.float32, 3)
        B, N, _ = xyz.shape
        if xyz.shape[2] != 3:
            raise RuntimeError("xyz must be (B, N, 3)")
        output = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
        temp = None
        dense = os.environ.get("SPSK_FPS", "")[:1] == "d"   # cross-check mode: the unpruned kernels, no clusters
        if N > (FPS_DISTMAT_ONCHIP_MAX_N if dense else FPS_ONCHIP_MAX_N):
            temp = torch.full((B, N), 1e10, dtype=torch.float32, device=xyz.device)
        with torch.cuda.device(xyz.device):
            check(lib.spsk_farthest_point_sampling(B, N, npoint, xyz.data_ptr(), temp.data_ptr() if temp is not None else None,
                                                   output.data_ptr(), _stream()), "farthest_point_sampling")
        return output

    @staticmethod
    def backward(ctx, a=None):
        return None, None


farthest_point_sample = furthest_point_sample = FarthestPointSampling.apply


class FurthestPointSamplingWithDist(Function):
    """reference: pointnet2_utils.py:39-62 (FurthestPointSamplingWithDist); xyz is a (B,N,N) distance matrix."""

    @staticmethod
    def forward(ctx, xyz: torch.Tensor, npoint: int) -> torch.Tensor:
        _chk(xyz, "dist", torch.float32, 3)
        B, N, N2 = xyz.shape
        if N != N2:
            raise RuntimeError("distance matrix must be (B, N, N)")
        output = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
        temp = None
        if N > FPS_DISTMAT_ONCHIP_MAX_N:
            temp = torch.full((B, N), 1e10, dtype=torch.float32, device=xyz.device)
        with torch.cuda.device(xyz.device):
            check(lib.spsk_furthest_point_sampling_with_dist(B, N, npoint, xyz.data_ptr(),
                                                             temp.data_ptr() if temp is not None else None,
                                                             output.data_ptr(), _stream()), "furthest_point_sampling_with_dist")
        return output

    @staticmethod
    def backward(ctx, a=None):
        return None, None


furthest_point_sample_with_dist = FurthestPointSamplingWithDist.apply


class GatherOperation(Function):
    """reference: pointnet2_utils.py:67-98 (GatherOperation)."""

    @staticmethod
    def forward(ctx, features: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
        _chk(features, "features", torch.float32, 3)
        _chk(idx, "idx", torch.int32, 2)
        B, npoint = idx.shape
        _, Cc, N = features.shape
        output = torch.empty((B, Cc, npoint), dtype=torch.float32, device=features.device)
        with torch.cuda.device(features.device):
            check(lib.spsk_gather_points(B, Cc, N, npoint, features.data_ptr(), idx.data_ptr(), output.data_ptr(), _stream()),
                  "gather_points")
        ctx.for_backwards = (idx, Cc, N)
        return output

    @staticmethod
    def backward(ctx, grad_out):
        idx, Cc, N = ctx.for_backwards
        B, npoint = idx.shape
        g = grad_out.detach().contiguous()
        if deterministic_grads():
            return scatter_grad(g, idx, N), None
        grad_features = torch.zeros((B, Cc, N), dtype=torch.float32, device=grad_out.device)
        with torch.cuda.device(g.device):
            check(lib.spsk_gather_points_grad(B, Cc, N, npoint, g.data_ptr(), idx.data_ptr(), grad_features.data_ptr(), _stream()),
                  "gather_points_grad")
        return grad_features, None


gather_operation = GatherOperation.apply


class ThreeNN(Function):
    """reference: pointnet2_utils.py:104-130 (ThreeNN); returns (sqrt(dist2), idx)."""

    @staticmethod
    def forward(ctx, unknown: torch.Tensor, known: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        _chk(unknown, "unknown", torch.float32, 3)
        _chk(known, "known", torch.float32, 3)
        B, N, _ = unknown.shape
        m = known.shape[1]
        dist2 = torch.empty((B, N, 3), dtype=torch.float32, device=unknown.device)
        idx = torch.empty((B, N, 3), dtype=torch.int32, device=unknown.device)
        with torch.cuda.device(unknown.device):
            check(lib.spsk_three_nn(B, N, m, unknown.data_ptr(), known.data_ptr(), dist2.data_ptr(), idx.data_ptr(), _stream()),
                  "three_nn")
        ctx.mark_non_differentiable(idx)
        return torch.sqrt(dist2), idx

    @staticmethod
    def backward(ctx, a=None, b=None):
        return None, None


three_nn = ThreeNN.apply

# include/spsk.h: spsk_three_nn runs the grid kernel for n >= THREE_NN_GRID_MIN_N and THREE_NN_GRID_MIN_M <= m <=
# THREE_NN_GRID_MAX_M, the all-pairs kernel otherwise (bit-identical results)
THREE_NN_GRID_MIN_N = 1024  # SPSK_THREE_NN_GRID_MIN_N
THREE_NN_GRID_MIN_M = 1024  # SPSK_THREE_NN_GRID_MIN_M
THREE_NN_GRID_MAX_M = 131072  # SPSK_THREE_NN_GRID_MAX_M


class ThreeInterpolate(Function):
    """reference: pointnet2_utils.py:136-178 (ThreeInterpolate)."""

    @staticmethod
    def forward(ctx, features: torch.Tensor, idx: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
        _chk(features, "features", torch.float32, 3)
        _chk(idx, "idx", torch.int32, 3)
        _chk(weight, "weight", torch.float32, 3)
        B, c, m = features.shape
        n = idx.shape[1]
        ctx.three_interpolate_for_backward = (idx, weight, m)
        output = torch.empty((B, c, n), dtype=torch.float32, device=features.device)
        with torch.cuda.device(features.device):
            check(lib.spsk_three_interpolate(B, c, m, n, features.data_ptr(), idx.data_ptr(), weight.data_ptr(),
                                             output.data_ptr(), _stream()), "three_interpolate")
        return output

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        idx, weight, m = ctx.three_interpolate_for_backward
        B, c, n = grad_out.shape
        g = grad_out.detach().contiguous()
        if deterministic_grads():
            return scatter_grad(g, idx.view(B, -1), m, weight=weight.contiguous().view(B, -1), div=3), None, None
        grad_features = torch.zeros((B, c, m), dtype=torch.float32, device=grad_out.device)
        with torch.cuda.device(g.device):
            check(lib.spsk_three_interpolate_grad(B, c, n, m, g.data_ptr(), idx.data_ptr(), weight.data_ptr(),
                                                  grad_features.data_ptr(), _stream()), "three_interpolate_grad")
        return grad_features, None, None


three_interpolate = ThreeInterpolate.apply


class GroupingOperation(Function):
    """reference: pointnet2_utils.py:184-222 (GroupingOperation)."""

    @staticmethod
    def forward(ctx, features: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
        _chk(features, "features", torch.float32, 3)
        _chk(idx, "idx", torch.int32, 3)
        B, nfeatures, nsample = idx.shape
        _, Cc, N = features.shape
        output = torch.empty((B, Cc, nfeatures, nsample), dtype=torch.float32, device=features.device)
        with torch.cuda.device(features.device):
            check(lib.spsk_group_points(B, Cc, N, nfeatures, nsample, features.data_ptr(), idx.data_ptr(),
                                        output.data_ptr(), _stream()), "group_points")
        ctx.for_backwards = (idx, N)
        return output

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        idx, N = ctx.for_backwards
        B, Cc, npoint, nsample = grad_out.shape
        g = grad_out.detach().contiguous()
        if deterministic_grads():
            return scatter_grad(g.view(B, Cc, -1), idx.view(B, -1), N), None
        grad_features = torch.zeros((B, Cc, N), dtype=torch.float32, device=grad_out.device)
        with torch.cuda.device(g.device):
            check(lib.spsk_group_points_grad(B, Cc, N, npoint, nsample, g.data_ptr(), idx.data_ptr(),
                                             grad_features.data_ptr(), _stream()), "group_points_grad")
        return grad_features, None


grouping_operation = GroupingOperation.apply


class BallQuery(Function):
    """reference: pointnet2_utils.py:228-253 (BallQuery); note the (radius, nsample, xyz, new_xyz) order."""

    @staticmethod
    def forward(ctx, radius: float, nsample: int, xyz: torch.Tensor, new_xyz: torch.Tensor) -> torch.Tensor:
        _chk(new_xyz, "new_xyz", torch.float32, 3)
        _chk(xyz, "xyz", torch.float32, 3)
        B, N, _ = xyz.shape
        npoint = new_xyz.shape[1]
        if GRID_BQ_MIN_N < N <= GRID_MAX_N:
            # the brute-force scan reads all N points for every centre whose ball holds fewer than nsample of them; the grid
            # kernel writes empty rows as zeros, which is what the zero-filled output below would hold
            return ball_query_msg([radius], [nsample], xyz, new_xyz, grid=True)[0]
        idx = torch.zeros((B, npoint, nsample), dtype=torch.int32, device=xyz.device)
        with torch.cuda.device(xyz.device):
            check(lib.spsk_ball_query(B, N, npoint, float(radius), int(nsample), new_xyz.data_ptr(), xyz.data_ptr(),
                                      idx.data_ptr(), _stream()), "ball_query")
        return idx

    @staticmethod
    def backward(ctx, a=None):
        return None, None, None, None


ball_query = BallQuery.apply


class BallQueryDilated(Function):
    """reference: pointnet2_utils.py:258-284 (BallQueryDilated)."""

    @staticmethod
    def forward(ctx, max_radius: float, min_radius: float, nsample: int, xyz: torch.Tensor, new_xyz: torch.Tensor) -> torch.Tensor:
        _chk(new_xyz, "new_xyz", torch.float32, 3)
        _chk(xyz, "xyz", torch.float32, 3)
        B, N, _ = xyz.shape
        npoint = new_xyz.shape[1]
        idx = torch.zeros((B, npoint, nsample), dtype=torch.int32, device=xyz.device)
        with torch.cuda.device(xyz.device):
            check(lib.spsk_ball_query_dilated(B, N, npoint, float(max_radius), float(min_radius), int(nsample),
                                              new_xyz.data_ptr(), xyz.data_ptr(), idx.data_ptr(), _stream()), "ball_query_dilated")
        return idx

    @staticmethod
    def backward(ctx, a=None):
        return None, None, None, None, None


ball_query_dilated = BallQueryDilated.apply


def _group(xyz, new_xyz, features, idx, use_xyz):
    """reference: pointnet2_utils.py:308-320 (shared tail of QueryAndGroup / QueryDilatedAndGroup)."""
    xyz_trans = xyz.transpose(1, 2).contiguous()
    grouped_xyz = grouping_operation(xyz_trans, idx)  # (B, 3, npoint, nsample)
    grouped_xyz = grouped_xyz - new_xyz.transpose(1, 2).unsqueeze(-1)
    if features is not None:
        grouped_features = grouping_operation(features, idx)
        if use_xyz:
            return torch.cat([grouped_xyz, grouped_features], dim=1)  # (B, C + 3, npoint, nsample)
        return grouped_features
    assert use_xyz, "Cannot have not features and not use xyz as a feature!"
    return grouped_xyz


class QueryAndGroup(nn.Module):
    """reference: pointnet2_utils.py:289-322."""

    def __init__(self, radius: float, nsample: int, use_xyz: bool = True):
        super().__init__()
        self.radius, self.nsample, self.use_xyz = radius, nsample, use_xyz

    def forward(self, xyz: torch.Tensor, new_xyz: torch.Tensor, features: torch.Tensor = None) -> torch.Tensor:
        idx = ball_query(self.radius, self.nsample, xyz, new_xyz)
        return _group(xyz, new_xyz, features, idx, self.use_xyz)


class QueryDilatedAndGroup(nn.Module):
    """reference: pointnet2_utils.py:324-359; (radius_in, radius_out) are forwarded as (max_radius, min_radius)."""

    def __init__(self, radius_in: float, radius_out: float, nsample: int, use_xyz: bool = True):
        super().__init__()
        self.radius_in, self.radius_out, self.nsample, self.use_xyz = radius_in, radius_out, nsample, use_xyz

    def forward(self, xyz: torch.Tensor, new_xyz: torch.Tensor, features: torch.Tensor = None) -> torch.Tensor:
        idx = ball_query_dilated(self.radius_in, self.radius_out, self.nsample, xyz, new_xyz)
        return _group(xyz, new_xyz, features, idx, self.use_xyz)


class GroupAll(nn.Module):
    """reference: pointnet2_utils.py:361-384."""

    def __init__(self, use_xyz: bool = True):
        super().__init__()
        self.use_xyz = use_xyz

    def forward(self, xyz: torch.Tensor, new_xyz: torch.Tensor, features: torch.Tensor = None):
        grouped_xyz = xyz.transpose(1, 2).unsqueeze(2)
        if features is not None:
            grouped_features = features.unsqueeze(2)
            if self.use_xyz:
                return torch.cat([grouped_xyz, grouped_features], dim=1)  # (B, 3 + C, 1, N)
            return grouped_features
        return grouped_xyz


# ---------------------------------------------------------------------------------------------------
# fused entry points (no counterpart function in the reference: they replace chains of torch ops in
# pointnet2_modules.py; see include/spsk.h section 2)
# ---------------------------------------------------------------------------------------------------

def score_topk(cls_features: torch.Tensor, npoint: int, stds: torch.Tensor | None = None,
               return_scores: bool = False):
    """ctr/cls-aware (reference pointnet2_modules.py:287-291) or, with `stds`, SPSNet stability-aware
    (:293-303) down-sampling indices: (B, npoint) int32, descending score, ties by ascending index.  One kernel launch
    for N up to 262144 (one CTA per scene up to 16384 points, a thread-block cluster of up to 16 CTAs above)."""
    _chk(cls_features, "cls_features", torch.float32, 3)
    B, N, nc = cls_features.shape
    if stds is not None:
        _chk(stds, "stds", torch.float32, 2)
        if tuple(stds.shape) != (B, N):
            raise RuntimeError(f"stds must be (B, N)=({B},{N}), got {tuple(stds.shape)}")
    idx = torch.empty((B, npoint), dtype=torch.int32, device=cls_features.device)
    scores = torch.empty((B, npoint), dtype=torch.float32, device=cls_features.device) if return_scores else None
    with torch.cuda.device(cls_features.device):
        check(lib.spsk_score_topk(B, N, nc, npoint, cls_features.data_ptr(), stds.data_ptr() if stds is not None else None,
                                  idx.data_ptr(), scores.data_ptr() if scores is not None else None, _stream()), "score_topk")
    return (idx, scores) if return_scores else idx


def gather_rows(points: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """out[b, j, :] = points[b, idx[b, j], :] for point-major (B, N, C) tensors (new_xyz = xyz[idx])."""
    _chk(points, "points", torch.float32, 3)
    _chk(idx, "idx", torch.int32, 2)
    B, N, Cc = points.shape
    M = idx.shape[1]
    out = torch.empty((B, M, Cc), dtype=torch.float32, device=points.device)
    with torch.cuda.device(points.device):
        check(lib.spsk_gather_rows(B, N, M, Cc, points.data_ptr(), idx.data_ptr(), out.data_ptr(), _stream()), "gather_rows")
    return out


GRID_MIN_N = 2048  # below this the brute-force scan (early exit, smem tiles) is as fast as building a grid
GRID_MAX_N = 262144  # include/spsk.h: SPSK_BQ_GRID_MAX_N
GRID_BQ_MIN_N = 65536  # BallQuery (single radius) takes the grid kernel above this many points


def ball_query_msg(radii, nsamples, xyz: torch.Tensor, new_xyz: torch.Tensor, grid=None):
    """All scales of an MSG layer in ONE pass; returns a list of (B, npoint, nsample_s) int32 tensors,
    identical to [ball_query(r, ns, xyz, new_xyz) for r, ns in zip(radii, nsamples)].  grid=None picks the
    uniform-grid kernel for GRID_MIN_N <= n <= GRID_MAX_N and the brute-force scan otherwise (same results)."""
    _chk(new_xyz, "new_xyz", torch.float32, 3)
    _chk(xyz, "xyz", torch.float32, 3)
    S = len(radii)
    B, N, _ = xyz.shape
    M = new_xyz.shape[1]
    outs = [torch.empty((B, M, int(ns)), dtype=torch.int32, device=xyz.device) for ns in nsamples]
    r = (C.c_float * S)(*[float(x) for x in radii])
    n = (C.c_int * S)(*[int(x) for x in nsamples])
    ptrs = (C.c_void_p * S)(*[o.data_ptr() for o in outs])
    use_grid = (GRID_MIN_N <= N <= GRID_MAX_N) if grid is None else bool(grid)
    with torch.cuda.device(xyz.device):
        if use_grid:
            nbytes = int(lib.spsk_ball_query_grid_workspace_bytes(B, N))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=xyz.device)
            check(lib.spsk_ball_query_msg_grid(B, N, M, S, r, n, new_xyz.data_ptr(), xyz.data_ptr(), ptrs, ws.data_ptr(),
                                               nbytes, _stream()), "ball_query_msg_grid")
        else:
            check(lib.spsk_ball_query_msg(B, N, M, S, r, n, new_xyz.data_ptr(), xyz.data_ptr(), ptrs, _stream()), "ball_query_msg")
    return outs


def grouped_linear(*, xyz, new_xyz, features, idx, use_xyz, in_rows, wt, bias, relu, pool, out_pooled=None, co_off=0):
    """One shared-MLP layer over grouped rows (include/spsk.h: spsk_grouped_linear).
    gather mode when in_rows is None.  Returns out_rows (R, c_out) for pool == 0, else out_pooled."""
    B, M, ns = idx.shape
    N = xyz.shape[1]
    c_in, c_out = wt.shape
    g = GroupDesc()
    g.b, g.n, g.m, g.nsample = B, N, M, ns
    g.c_feat = features.shape[1] if features is not None else 0
    g.use_xyz = 1 if use_xyz else 0
    g.xyz = xyz.data_ptr()
    g.new_xyz = new_xyz.data_ptr()
    g.features = features.data_ptr() if features is not None else None
    g.idx = idx.data_ptr()
    out_rows = None
    if pool == 0:
        out_rows = torch.empty((B * M * ns, c_out), dtype=torch.float32, device=idx.device)
    c_total = out_pooled.shape[1] if out_pooled is not None else 0
    with torch.cuda.device(idx.device):
        check(lib.spsk_grouped_linear(C.byref(g), 1 if in_rows is None else 0,
                                      in_rows.data_ptr() if in_rows is not None else None, c_in,
                                      wt.data_ptr(), bias.data_ptr() if bias is not None else None, c_out,
                                      1 if relu else 0, pool,
                                      out_rows.data_ptr() if out_rows is not None else None,
                                      out_pooled.data_ptr() if out_pooled is not None else None,
                                      c_total, co_off, _stream()), "grouped_linear")
    return out_rows if pool == 0 else out_pooled


def pointwise_linear(x: torch.Tensor, wt: torch.Tensor, bias, relu: bool) -> torch.Tensor:
    """Conv1d(kernel_size=1) [+ folded BN] [+ ReLU] on a channel-major (B, C_in, M) tensor."""
    _chk(x, "x", torch.float32, 3)
    B, c_in, M = x.shape
    if wt.shape[0] != c_in:
        raise RuntimeError(f"weight (c_in={wt.shape[0]}) does not match input channels {c_in}")
    c_out = wt.shape[1]
    out = torch.empty((B, c_out, M), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.spsk_pointwise_linear(B, M, x.data_ptr(), c_in, wt.data_ptr(), bias.data_ptr() if bias is not None else None,
                                        c_out, 1 if relu else 0, out.data_ptr(), _stream()), "pointwise_linear")
    return out


# ---------------------------------------------------------------------------------------------------
# tensor-core path (tcgen05): host-side packing + launch  (include/spsk.h "tensor-core path")
# ---------------------------------------------------------------------------------------------------

def _ceil(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def _canonical_tile(block: torch.Tensor) -> torch.Tensor:
    """(rows, k) -> flat fp16 in the K-major no-swizzle UMMA layout: 8-row x 8-half core matrices, k-groups
    contiguous inside an 8-row group:  half(r, k) = (r/8)*(kw*8) + (k/8)*64 + (r%8)*8 + (k%8)."""
    rows, kw = block.shape
    return block.reshape(rows // 8, 8, kw // 8, 8).permute(0, 2, 1, 3).contiguous().reshape(-1)


def _pack_chunks(Wt: torch.Tensor, ncols: int) -> torch.Tensor:
    """All cout chunks of one width at once: Wt (nchunk*ncols, vk) fp16 -> the chunks' tiles, chunk-major then k, every tile
    `ncols x kw` (kw = 64, the last one vk % 64) in the canonical layout of `_canonical_tile`.  Two strided copies per call instead
    of one per tile: training re-packs the weights every step."""
    nch, vk = Wt.shape[0] // ncols, Wt.shape[1]
    nfk = vk // 64
    kr = vk - nfk * 64
    parts = []
    if nfk:
        parts.append(Wt[:, :nfk * 64].reshape(nch, ncols // 8, 8, nfk, 8, 8).permute(0, 3, 1, 4, 2, 5).reshape(nch, -1))
    if kr:
        parts.append(Wt[:, nfk * 64:].reshape(nch, ncols // 8, 8, 1, kr // 8, 8).permute(0, 3, 1, 4, 2, 5).reshape(nch, -1))
    return (parts[0] if len(parts) == 1 else torch.cat(parts, dim=1)).reshape(-1)


def _pack_layer(Wv: torch.Tensor) -> list:
    """Wv (vk, cp) fp16 -> flat tiles of (<= 128 couts) x (<= 64 k), cout-chunk major then k (include/spsk.h: wtiles)."""
    Wt = Wv.t()
    cp = Wt.shape[0]
    nfc = cp // 128
    out = []
    if nfc:
        out.append(_pack_chunks(Wt[:nfc * 128], 128))
    if cp - nfc * 128:
        out.append(_pack_chunks(Wt[nfc * 128:], cp - nfc * 128))
    return out


class MmaChain:
    """A folded Conv/BN/ReLU chain packed for spsk_sa_mma_forward (layout: include/spsk.h).

    plain mode : fp16 operands; layer-0 input order [features (ceil8(c_feat)), x, y, z, 0...] (the reference's order
                 is [x, y, z, features], pointnet2_utils.py:315 -- a pure row permutation of W0)
    split mode : chosen automatically for narrow chains (every width <= 64, c_feat <= 8: IA-SSD layer 0); weights
                 become [Wh; Wl] and the kernel evaluates Xh.Wh + Xl.Wh + Xh.Wl  (fp32-grade)
    """

    def __init__(self, chain, c_feat: int, use_xyz: bool, split: bool | None = None, pair: bool | None = None):
        dev = chain[0][0].device
        self.nlayers = len(chain)
        self.c_feat, self.use_xyz = c_feat, use_xyz
        widths = [wt.shape[1] for wt, _, _ in chain]
        can_split = c_feat <= 8 and all(_ceil(w, 16) <= 64 for w in widths[:-1]) and self.nlayers <= 4
        self.split = can_split if split is None else (bool(split) and can_split)
        # CTA-pair kernel (tcgen05 cta_group::2, sa_mma_pair.cu) for wide chains: opt-in (SPSK_SA_PAIR=1 or pair=True).
        # Measured on B200 (round 1): correct, 4x fewer MMA issues per row, but with the activations of 128 rows per CTA
        # still filling shared memory the 2-stage weight ring plus the cross-CTA forwarding hops make it 25-45 % slower
        # than the single-CTA kernel (layer 5 scale 2: 388 vs 288 us) -- see DESIGN.md section 4.3.
        can_pair = (not self.split) and len(widths) >= 2
        want_pair = can_pair and os.environ.get("SPSK_SA_PAIR", "0") == "1" and (max(widths) >= 512 or widths[-1] >= 256)
        self.pair = want_pair if pair is None else (bool(pair) and can_pair)
        self.cpad8 = _ceil(c_feat, 8) if c_feat > 0 else 0
        k0 = self.cpad8 + (8 if use_xyz else 0)
        self.ok = 1 <= self.nlayers <= 4 and all(relu for _, _, relu in chain) and k0 > 0
        kin = 16 if self.split else _ceil(max(k0, 16), 16)
        self.kpad, self.cpad = [], []
        tiles, biases = [], []
        for l, (wt, bias, _relu) in enumerate(chain):
            cin, cout = wt.shape
            last = l == self.nlayers - 1
            cp = _ceil(cout, (256 if self.pair else 128) if last else 16)
            W = torch.zeros((kin, cp), dtype=torch.float32, device=dev)
            if l == 0:
                xr = 3 if use_xyz else 0  # reference row order: xyz first
                fo = 0
                xo = (8 if c_feat else 0) if self.split else self.cpad8
                if c_feat:
                    W[fo:fo + c_feat, :cout] = wt[xr:xr + c_feat]
                if use_xyz:
                    W[xo:xo + 3, :cout] = wt[0:3]
            else:
                W[:cin, :cout] = wt
            if self.split:
                Wh = W.half()
                Wl = (W - Wh.float()).half()
                Wv = torch.cat([Wh, Wl], dim=0)   # Wh serves two of the three products (Xh.Wh, Xl.Wh), stored once
            else:
                Wv = W.half()
            vk = Wv.shape[0]
            if self.pair:
                # 256-wide cout chunks; inside a chunk the rows of pair rank 0 then rank 1 (half of the chunk each; the last
                # layer's chunks are always 256 wide: 128 couts per CTA), each as tiles of <= 64 k
                for c0 in range(0, cp, 256):
                    cw = min(256, cp - c0)
                    for rk in range(2):
                        r0 = c0 + rk * (cw // 2)
                        for k0_ in range(0, vk, 64):
                            kw = min(64, vk - k0_)
                            tiles.append(_canonical_tile(Wv[k0_:k0_ + kw, r0:r0 + cw // 2].t()))
            else:
                tiles += _pack_layer(Wv)
            bv = torch.zeros(cp, dtype=torch.float32, device=dev)
            bv[:cout] = bias
            biases.append(bv)
            self.kpad.append(kin)
            self.cpad.append(cp)
            if kin > 1024 or (not last and cp > 1024):
                self.ok = False
            kin = cp
            self.cout_last = cout
        # split chains: layer 0 (<= 11 real inputs) CAN be evaluated in fp32 by the gather threads (include/spsk.h: l0_fused; its
        # fp32 weights [16][cpad0] + bias ride behind the fp16 tiles).  Opt-in (SPSK_SA_L0_FUSED=1): measured on B200 it is
        # 8-12 % SLOWER than running layer 0 as one more tensor-core job -- the gather/epilogue warps' instruction issue, not
        # the hand-off latency, bounds these chains, and the fusion adds ~300 instructions per row to exactly those warps.
        self.l0_fused = bool(self.split and self.nlayers >= 2 and self.cpad[0] <= 32 and os.environ.get("SPSK_SA_L0_FUSED", "0") == "1")
        if self.l0_fused:
            wt0, b0, _ = chain[0]
            cp0 = self.cpad[0]
            W0 = torch.zeros((16, cp0), dtype=torch.float32, device=dev)
            xr = 3 if use_xyz else 0
            if c_feat:
                W0[0:c_feat, :wt0.shape[1]] = wt0[xr:xr + c_feat]
            if use_xyz:
                xo = 8 if c_feat else 0
                W0[xo:xo + 3, :wt0.shape[1]] = wt0[0:3]
            bb0 = torch.zeros(cp0, dtype=torch.float32, device=dev)
            bb0[:wt0.shape[1]] = b0
            tiles.append(torch.cat([W0.reshape(-1), bb0]).contiguous().view(torch.float16))
        self.wtiles = torch.cat(tiles).contiguous()
        self.bias = torch.cat(biases).contiguous()
        self.ctas_per_sm = self.nstages = self.resident = self.smem = 0
        if self.ok:
            d = self._desc()
            v = [C.c_int(0) for _ in range(4)]
            self.ok = lib.spsk_sa_mma_config(C.byref(d), *[C.byref(x) for x in v]) == 0
            self.smem, self.ctas_per_sm, self.nstages, self.resident = [int(x.value) for x in v]

    def _desc(self) -> SaMmaDesc:
        d = SaMmaDesc()
        d.nlayers = self.nlayers
        for l in range(self.nlayers):
            d.kpad[l] = self.kpad[l]
            d.cpad[l] = self.cpad[l]
        d.split = 1 if self.split else 0
        d.ovf_tag = current_ovf_tag
        d.pair = 1 if self.pair else 0
        d.l0_fused = 1 if self.l0_fused else 0
        d.c_feat = self.c_feat
        d.use_xyz = 1 if self.use_xyz else 0
        d.cout_last = self.cout_last
        d.wtiles = self.wtiles.data_ptr()
        d.bias = self.bias.data_ptr()
        return d


def make_twin(features: torch.Tensor, cpad8: int) -> torch.Tensor:
    """(B, C, N) f32 -> (B, N, cpad8) fp16 point-major, zero padded."""
    _chk(features, "features", torch.float32, 3)
    B, Cc, N = features.shape
    twin = torch.empty((B, N, cpad8), dtype=torch.float16, device=features.device)
    with torch.cuda.device(features.device):
        check(lib.spsk_make_twin(B, Cc, N, cpad8, features.data_ptr(), twin.data_ptr(), _stream()), "make_twin")
    return twin


def sa_mma_stats_parts(idx: torch.Tensor, n: int, chain: MmaChain) -> int:
    """Partial-sum slices a batch-statistics pass of `chain` over these centres writes (include/spsk.h)."""
    B, M, ns = idx.shape
    d = chain._desc()
    d.b, d.n, d.m, d.nsample = B, n, M, ns
    v = C.c_int(0)
    check(lib.spsk_sa_mma_stats_parts(C.byref(d), C.byref(v)), "sa_mma_stats_parts")
    return int(v.value)


def sa_mma_forward(*, xyz, new_xyz, idx, chain: MmaChain, twin=None, features=None, out_pooled=None, co_off=0,
                   out16=None, co16=0, n16=None, o16lo=0, stats=None):
    """One fused MSG scale (include/spsk.h: spsk_sa_mma_forward).  `twin` (B, N, ld) fp16 in plain mode, `features`
    (B, C, N) fp32 in split mode; results go to out_pooled[:, co_off:co_off+cout, :] (fp32, (B, C_total, M)) and/or
    out16[:, co16:co16+n16] (fp16, (B*M, ld16)); with o16lo > 0 the fp16 residuals go to out16[:, o16lo+co16 : ...]."""
    B, M, ns = idx.shape
    d = chain._desc()
    d.b, d.n, d.m, d.nsample = B, xyz.shape[1], M, ns
    d.xyz, d.new_xyz, d.idx = xyz.data_ptr(), new_xyz.data_ptr(), idx.data_ptr()
    if chain.c_feat:
        if chain.split:
            _chk(features, "features", torch.float32, 3)
            d.features = features.data_ptr()
        else:
            if twin is None or twin.dtype != torch.float16 or not twin.is_contiguous() or twin.shape[2] < chain.cpad8:
                raise RuntimeError("sa_mma_forward: twin must be a contiguous (B, N, >=ceil8(C)) fp16 tensor")
            d.twin, d.ldtwin = twin.data_ptr(), twin.shape[2]
    if out_pooled is not None:
        d.out_cm, d.c_total, d.co_off = out_pooled.data_ptr(), out_pooled.shape[1], co_off
    if out16 is not None:
        d.out16, d.ld16, d.co16 = out16.data_ptr(), out16.shape[-1], co16
        d.n16 = chain.cout_last if n16 is None else n16
        d.o16lo = int(o16lo)
    if stats is not None:
        # batch-statistics pass (training-mode BN): stats (parts, cpad_last, 2) float64 (the call zeroes the slices it uses); nothing else is written
        if stats.dtype != torch.float64 or not stats.is_contiguous() or stats.dim() != 3 or stats.shape[1] != chain.cpad[-1] or stats.shape[2] != 2:
            raise RuntimeError("sa_mma_forward: stats must be a contiguous (parts, cpad_last, 2) float64 tensor")
        d.stats, d.stats_parts = stats.data_ptr(), stats.shape[0]
    with torch.cuda.device(idx.device):
        check(lib.spsk_sa_mma_forward(C.byref(d), _stream()), "sa_mma_forward")
    if stats is not None:
        return stats
    return out_pooled if out_pooled is not None else out16


class PwLayer:
    """One folded Conv1d(k=1)[+BN][+ReLU] layer packed for spsk_pw_mma_forward: W (c_out x K) as 128-cout x 64-k
    fp16 tiles (16 KB each, canonical K-major layout), zero padded to cover ceil128(max(c_out, n16)) couts.
    split=True packs, per (cout chunk, k chunk), the Wh tile followed by the Wl tile, for inputs carried as hi + lo
    fp16 halves (y = xh.Wh + xl.Wh + xh.Wl)."""

    def __init__(self, wt: torch.Tensor, bias: torch.Tensor, relu: bool, split: bool = False):
        dev = wt.device
        self.c_in, self.c_out = wt.shape
        self.relu = bool(relu)
        self.split = bool(split)
        self.k = _ceil(self.c_in, 16)
        self.n16 = _ceil(self.c_out, 16)
        ncov = _ceil(max(self.c_out, self.n16), 128)
        n_cc, n_kc = ncov // 128, _ceil(self.k, 64) // 64
        Wt = torch.zeros((ncov, n_kc * 64), dtype=torch.float32, device=dev)
        Wt[:self.c_out, :self.c_in] = wt.t()

        def tiles(M):  # (ncov, n_kc*64) -> (cc, kc, rg, kg, r, k) canonical 16 KB tiles
            return M.view(n_cc, 16, 8, n_kc, 8, 8).permute(0, 3, 1, 4, 2, 5).contiguous()

        if self.split:
            Wh = Wt.half()
            Wl = (Wt - Wh.float()).half()
            # per (cc, kc): the Wh tile immediately followed by the Wl tile (one 32 KB bulk copy per pipeline step)
            T = torch.stack([tiles(Wh), tiles(Wl)], dim=2)
        else:
            T = tiles(Wt.half())
        self.wtiles = T.reshape(-1).contiguous()
        self.bias = torch.zeros(ncov, dtype=torch.float32, device=dev)
        self.bias[:self.c_out] = bias


def pw_mma_forward(x16: torch.Tensor, layer: PwLayer, *, xlo=0, out_cm=None, m=0, co_off=0, want16=False, want16_lo=False, out_pm=None):
    """y = act(x16 @ W^T + b) on the tensor cores.  x16: (rows, ldx) fp16 point-major with zeros in columns >= c_in
    (split layers: hi in [0, k), lo in [xlo, xlo + k)).  Returns (out_cm, out16, out_pm); out16 = (rows, ceil16(c_out))
    fp16 when want16, or (rows, 2 * ceil16(c_out)) = [hi | lo] when want16_lo."""
    if x16.dtype != torch.float16 or x16.dim() != 2 or not x16.is_contiguous() or not x16.is_cuda:
        raise RuntimeError("pw_mma_forward: x16 must be a contiguous CUDA (rows, ldx) fp16 tensor")
    rows, ldx = x16.shape
    if ldx < layer.k or (layer.split and (xlo < layer.k or xlo + layer.k > ldx)):
        raise RuntimeError(f"pw_mma_forward: input width {ldx} (lo at {xlo}) does not hold the padded c_in {layer.k}")
    d = PwDesc()
    d.rows, d.k, d.ldx, d.n, d.relu = rows, layer.k, ldx, layer.c_out, 1 if layer.relu else 0
    d.split, d.xlo = (1, int(xlo)) if layer.split else (0, 0)
    d.ovf_tag = current_ovf_tag
    d.x, d.wtiles, d.bias = x16.data_ptr(), layer.wtiles.data_ptr(), layer.bias.data_ptr()
    if out_cm is not None:
        d.out_cm, d.m, d.c_total, d.co_off = out_cm.data_ptr(), m, out_cm.shape[1], co_off
    out16 = None
    if want16 or want16_lo:
        ld16 = layer.n16 * (2 if want16_lo else 1)
        out16 = torch.empty((rows, ld16), dtype=torch.float16, device=x16.device)
        d.out16, d.ld16, d.n16 = out16.data_ptr(), ld16, layer.n16
        d.o16lo = layer.n16 if want16_lo else 0
    if out_pm is not None:
        d.out_pm, d.ldpm = out_pm.data_ptr(), out_pm.shape[-1]
    with torch.cuda.device(x16.device):
        check(lib.spsk_pw_mma_forward(C.byref(d), _stream()), "pw_mma_forward")
    return out_cm, out16, out_pm
