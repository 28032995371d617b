"""Tensor-level wrappers over the C-ABI (torch supplies device memory and the current stream only).

Every function takes/returns CUDA fp32 tensors in the reference's layouts; index tensors are
int64 where the reference's callers see them (torch.topk output, gcn3d.py:21) and int32 inside
the fused encoder.  No function here computes anything in PyTorch.
"""
import ctypes

import torch

from . import _lib
from ._lib import GemmArgs, OutSeg


# large contractions go to the tcgen05 3xTF32 kernel; small / odd ones (K = 3, M = batch) to the fp32 FMA kernel
TC_ENABLED = True

# bench.py sets this to a dict to time every C-ABI call with CUDA events on the launching stream
EVENT_LOG = None


# device of the op being assembled: set by _f32c / _idx from the op's own tensors, so that the stream handed to the
# C-ABI and the launch itself belong to the tensors' device, not to whatever device happens to be current
_DEV = None


def _run(name, cfn, *args):
    log = EVENT_LOG
    if _DEV is not None and _DEV.index is not None and _DEV.index != torch.cuda.current_device():
        with torch.cuda.device(_DEV):
            _lib.check(cfn(*args), "tgp_" + name)
        return
    if log is None:
        _lib.check(cfn(*args), "tgp_" + name)
        return
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    rc = cfn(*args)
    b.record()
    log.setdefault(name, []).append((a, b))
    _lib.check(rc, "tgp_" + name)


def _ptr(t):
    """device address of a tensor handed to the C-ABI.  A host tensor is refused here, before anything is launched: a
    kernel given a host address faults the whole CUDA context, asynchronously, long after the call returned."""
    if not t.is_cuda:
        raise RuntimeError("expected a CUDA tensor (tg-pose_b200 has no CPU path)")
    return t.data_ptr()


def _p(t):
    return ctypes.c_void_p(_ptr(t)) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream(_DEV).cuda_stream)


def _f32c(t, name):
    global _DEV
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (tg-pose_b200 has no CPU path)")
    _DEV = t.device
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _idx(t, name):
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA index tensor")
    if t.dtype not in (torch.int64, torch.int32):
        t = t.long()
    t = t.contiguous()
    return t, (64 if t.dtype == torch.int64 else 32)


# --------------------------------------------------------------------------------------- kNN
def knn_xyz(xyz, k, want64=True, want32=False):
    """get_neighbor_index on (B,N,3), gcn3d.py:14-23.  Returns (idx64 or None, idx32 or None)."""
    xyz = _f32c(xyz, "knn_xyz")
    B, N, D = xyz.shape
    assert D == 3
    i64 = torch.empty((B, N, k), dtype=torch.int64, device=xyz.device) if want64 else None
    i32 = torch.empty((B, N, k), dtype=torch.int32, device=xyz.device) if want32 else None
    _run("knn_xyz", _lib.load().tgp_knn_xyz, _p(xyz), B, N, k, _p(i64), _p(i32), _stream())
    return i64, i32


def knn_feat(x, k, want64=True, want32=False, x_split=None):
    """get_neighbor_index on (B,N,D) features (RF-F), gcn3d.py:14-23,201-206.  x_split: the same features already
    split as a tensor-core operand (B*N, 2*kpad(D)), if a producer's epilogue wrote it."""
    x = _f32c(x, "knn_feat")
    B, N, D = x.shape
    lib = _lib.load()
    if x_split is not None and (x_split.numel() == 0 or x_split.shape != (B * N, 2 * kpad(D))):
        x_split = None
    ws_bytes = lib.tgp_knn_feat_workspace(B, N, D, 1 if x_split is not None else 0)
    ws = torch.empty((ws_bytes + 3) // 4, dtype=torch.float32, device=x.device)
    i64 = torch.empty((B, N, k), dtype=torch.int64, device=x.device) if want64 else None
    i32 = torch.empty((B, N, k), dtype=torch.int32, device=x.device) if want32 else None
    _run("knn_feat", lib.tgp_knn_feat, _p(x), _p(x_split), B, N, D, k, _p(i64), _p(i32), _p(ws), ws_bytes, _stream())
    return i64, i32


def nearest(target, source, want64=True, want32=False):
    """get_nearest_index, gcn3d.py:26-35 -> (B,N,1)."""
    target, source = _f32c(target, "nearest"), _f32c(source, "nearest")
    B, N, _ = target.shape
    M = source.shape[1]
    i64 = torch.empty((B, N, 1), dtype=torch.int64, device=target.device) if want64 else None
    i32 = torch.empty((B, N, 1), dtype=torch.int32, device=target.device) if want32 else None
    _run("nearest", _lib.load().tgp_nearest, _p(target), _p(source), B, N, M, _p(i64), _p(i32), _stream())
    return i64, i32


# --------------------------------------------------------------------------------------- gathers
def gather_rows(tensor, index):
    """indexing_neighbor_new, gcn3d.py:38-46: (B,N,C),(B,M,k) -> (B,M,k,C)."""
    tensor = _f32c(tensor, "gather_rows")
    index, bits = _idx(index, "gather_rows")
    B, N = tensor.shape[0], tensor.shape[1]
    C = tensor.numel() // (B * N)
    _, M, k = index.shape
    out = torch.empty((B, M, k, C), dtype=torch.float32, device=tensor.device)
    _run("gather_rows", _lib.load().tgp_gather_rows, _p(tensor), _p(index), bits, B, N, M, k, C, _p(out), _stream())
    return out


def select_rows(tensor, rows):
    """tensor[:, rows, :] with one row list for the whole batch (gcn3d.py:243-244)."""
    tensor = _f32c(tensor, "select_rows")
    rows = rows.to(device=tensor.device, dtype=torch.int64).contiguous()
    B, N, C = tensor.shape
    M = rows.numel()
    out = torch.empty((B, M, C), dtype=torch.float32, device=tensor.device)
    _run("select_rows", _lib.load().tgp_select_rows, _p(tensor), _p(rows), B, N, M, C, _p(out), _stream())
    return out


def direction_norm(xyz, idx):
    """get_neighbor_direction_norm, gcn3d.py:48-58 -> (B,N,k,3)."""
    xyz = _f32c(xyz, "direction_norm")
    idx, bits = _idx(idx, "direction_norm")
    B, N, k = idx.shape
    out = torch.empty((B, N, k, 3), dtype=torch.float32, device=xyz.device)
    _run("direction_norm", _lib.load().tgp_direction_norm, _p(xyz), _p(idx), bits, B, N, k, _p(out), _stream())
    return out


def gather_max(f, idx, rows=None, want_arg=False):
    """max_j f[b, idx[b, rows[m], j], :] -> (B,M,C) (+ uint8 arg)."""
    f = _f32c(f, "gather_max")
    idx, bits = _idx(idx, "gather_max")
    B, N, C = f.shape
    k = idx.shape[2]
    if rows is not None:
        rows = rows.to(device=f.device, dtype=torch.int64).contiguous()
        M = rows.numel()
    else:
        M = N
    out = torch.empty((B, M, C), dtype=torch.float32, device=f.device)
    arg = torch.empty((B, M, C), dtype=torch.uint8, device=f.device) if want_arg else None
    _run("gather_max", _lib.load().tgp_gather_max, _p(f), _p(idx), bits, _p(rows), B, N, M, k, C, _p(out), _p(arg), _stream())
    return (out, arg) if want_arg else out


def orl_global(f, idx, want_arg=False):
    """get_ORL_global before .repeat, gcn3d.py:210-217 -> (B,C)."""
    f = _f32c(f, "orl_global")
    idx, bits = _idx(idx, "orl_global")
    B, N, C = f.shape
    k = idx.shape[2]
    g = torch.empty((B, C), dtype=torch.float32, device=f.device)
    arg = torch.empty((B, N, C), dtype=torch.uint8, device=f.device) if want_arg else None
    lib = _lib.load()
    ws_bytes = lib.tgp_orl_workspace(B, N, C)
    ws = torch.empty((ws_bytes + 3) // 4, dtype=torch.float32, device=f.device)
    _run("orl_global", lib.tgp_orl_global, _p(f), _p(idx), bits, B, N, k, C, _p(g), _p(arg), _p(ws), ws_bytes, _stream())
    return (g, arg) if want_arg else g


def concat_rows(sources, B, N, want_raw=True, want_split=False, mixed=False):
    """[src_0 | src_1 | ...] per point.  sources: list of (tensor2d (rows, C), idx or None, n_src):
    idx None & n_src > 0: identity rows; idx (B,N) int32: gather from a cloud of n_src rows; n_src == 0: per-cloud row.
    Returns (raw (B*N, total) or None, split (B*N, 2*kpad(total)) or None)."""
    dev = sources[0][0].device
    arr = (_lib.ConcatSrc * len(sources))()
    total = 0
    keep = []
    for i, (t, idx, n_src) in enumerate(sources):
        assert t.stride(-1) == 1 and t.dim() == 2
        if idx is not None:
            idx = idx.to(torch.int32).contiguous()
            keep.append(idx)
        arr[i] = _lib.ConcatSrc(_ptr(t), t.shape[1], t.stride(0), _ptr(idx) if idx is not None else None, n_src)
        total += t.shape[1]
    M = B * N
    raw = torch.empty((M, total), dtype=torch.float32, device=dev) if want_raw else None
    kp = mixed_kpad(total) if mixed else kpad(total)
    spl = torch.empty((M, 2 * kp), dtype=torch.float32, device=dev) if want_split else None
    _run("concat_rows", _lib.load().tgp_concat_rows, arr, len(sources), B, N, _p(raw), total, _p(spl), kp,
         1 if mixed else 0, _stream())
    return raw, spl


# --------------------------------------------------------------------------------------- graph convs
def _split_buf(M, C, device):
    kp = kpad(C)
    return (torch.zeros if kp != C else torch.empty)((M, 2 * kp), dtype=torch.float32, device=device)


def surface_conv(xyz, idx, directions, S, C, want_arg=False, want_split=False, full=False):
    """HSlayer_surface.graph_conv, gcn3d.py:91-106 -> (B,N,C) [, arg][, split operand (B*N, 2*Kp)]."""
    xyz = _f32c(xyz, "surface_conv")
    directions = _f32c(directions, "surface_conv")
    idx, bits = _idx(idx, "surface_conv")
    B, N, k = idx.shape
    out = torch.empty((B, N, C), dtype=torch.float32, device=xyz.device)
    arg = torch.empty((B, N, S * C), dtype=torch.uint8, device=xyz.device) if want_arg else None
    spl = _split_buf(B * N, C, xyz.device) if want_split else None
    _run("surface_conv_fwd", _lib.load().tgp_surface_conv_fwd, _p(xyz), _p(idx), bits, _p(directions), B, N, k, S, C,
         _p(out), _p(arg), _p(spl), _stream())
    if full or want_split:
        return out, arg, spl
    return (out, arg) if want_arg else out


def edge_records(xyz, idx):
    xyz = _f32c(xyz, "edge_records")
    idx, bits = _idx(idx, "edge_records")
    B, N, k = idx.shape
    rec = torch.empty((B, k, N, 4), dtype=torch.float32, device=xyz.device)     # neighbour-major
    _run("edge_records", _lib.load().tgp_edge_records, _p(xyz), _p(idx), bits, B, N, k, _p(rec), _stream())
    return rec


def layer_conv(rec, directions, centre, support_slab, B, N, S, C, want_arg=False, want_split=False, full=False):
    """HS_layer.graph_conv after the projection, gcn3d.py:157-180 -> (B,N,C).
    centre: (B*N, C) view (any row stride); support_slab: [C/4][B*N][S*4]; rec (B,k,N,4) from edge_records."""
    k = rec.shape[1]
    directions = _f32c(directions, "layer_conv")
    out = torch.empty((B, N, C), dtype=torch.float32, device=rec.device)
    arg = torch.empty((C // 4, B * N, S * 4), dtype=torch.uint8, device=rec.device) if want_arg else None
    assert centre.stride(-1) == 1
    spl = _split_buf(B * N, C, rec.device) if want_split else None
    _run("layer_conv_fwd", _lib.load().tgp_layer_conv_fwd, _p(rec), _p(directions), _p(centre), centre.stride(0),
         _p(support_slab), B, N, k, S, C, _p(out), _p(arg), _p(spl), _stream())
    if full or want_split:
        return out, arg, spl
    return (out, arg) if want_arg else out


# --------------------------------------------------------------------------------------- gemm
def tc_eligible(M, K, Ncols):
    return TC_ENABLED and M >= 256 and K >= 16 and Ncols >= 16


def split_tf32(x2d, src_is_kn=False):
    """[tf32(x) | x - tf32(x)] operand for the tensor-core GEMM: (rows, 2*Kp).  x2d: (rows,K) (row-strided
    views allowed) or, with src_is_kn, (K, rows)."""
    assert x2d.stride(-1) == 1
    rows, K = (x2d.shape[1], x2d.shape[0]) if src_is_kn else (x2d.shape[0], x2d.shape[1])
    lib = _lib.load()
    Kp = lib.tgp_split_kpad(K)
    dst = torch.empty((rows, 2 * Kp), dtype=torch.float32, device=x2d.device)
    _run("split_tf32", lib.tgp_split_tf32, _p(x2d), rows, K, x2d.stride(0), 1 if src_is_kn else 0, _p(dst), _stream())
    return dst


class ParamCache:
    """Derived weight tensors (packed / tf32-split) cached per parameter OBJECT and version.
    Keys use id() guarded by weak references: a data_ptr-only key goes stale when a freed parameter's
    storage is reused by a new module."""

    def __init__(self):
        self._d = {}

    def get(self, params, tag, build):
        import weakref
        key = (tag,) + tuple(id(p) for p in params)
        ver = tuple((p._version, p.data_ptr()) for p in params)
        ent = self._d.get(key)
        if ent is not None and ent[0] == ver and all(r() is p for r, p in zip(ent[1], params)):
            return ent[2]
        if len(self._d) > 512:
            self._d = {k: v for k, v in self._d.items() if all(r() is not None for r in v[1])}
        val = build()
        self._d[key] = (ver, tuple(weakref.ref(p) for p in params), val)
        return val


PARAM_CACHE = ParamCache()


def gemm(A, Bmat, b_is_nk, segs, bias=None, group_bias=None, rows_per_group=0, res1=None, res2=None,
         scale=None, shift=None, relu=False, K=None, Ncols=None, A_split=None, B_split=None, neg_slope=None, tc=None,
         mixed=False, a_kp=0, a_group_cols=0, res1_idx=None, res2_idx=None, algo_flops=None):
    """C = A @ B (+ epilogue) written to `segs` = [(col_begin, col_end, tensor, mode, slab_width)].
    A: (M,K) with unit column stride; Bmat: (K,Ncols) or, if b_is_nk, (Ncols,K); both may be row-strided views."""
    assert Bmat.stride(-1) == 1
    if A is None:
        assert A_split is not None and K is not None, "gemm: A=None needs A_split and K"
        M = A_split.shape[0]
        tc = True
    else:
        assert A.stride(-1) == 1
        M = A.shape[0]
    if K is None:
        K = A.shape[1]
    if Ncols is None:
        Ncols = Bmat.shape[0] if b_is_nk else Bmat.shape[1]
    if tc is None:
        tc = tc_eligible(M, K, Ncols)
    if tc:
        if A_split is None:
            A_split = split_tf32(A[:, :K] if A.shape[1] != K else A)
        if B_split is None:
            B_split = split_tf32(Bmat.detach(), src_is_kn=not b_is_nk)   # callers with persistent weights pass a cached split
    else:
        A_split = B_split = None
    a = GemmArgs()
    if A is not None:
        a.A, a.lda = _ptr(A), A.stride(0)
    a.Bmat, a.ldb, a.b_is_nk = _ptr(Bmat), Bmat.stride(0), 1 if b_is_nk else 0
    if A_split is not None and B_split is not None:
        a.A_split, a.B_split = _ptr(A_split), _ptr(B_split)
    a.mixed = int(mixed)          # 0: 3xTF32 operands, 1: mixed, 2: mixed with a w16 weight operand (third pass fp16(a).lo16(b))
    a.a_kp, a.a_group_cols = int(a_kp), int(a_group_cols)      # block-diagonal contraction (tgp_gemm_args.a_group_cols)
    if mixed:
        assert A_split is not None and B_split is not None, "mixed operands must be supplied (split_mixed / mode-4 epilogue)"
    a.M, a.K, a.Ncols = M, K, Ncols
    a.bias = _ptr(bias) if bias is not None else None
    a.group_bias = _ptr(group_bias) if group_bias is not None else None
    a.rows_per_group = rows_per_group
    if res1 is not None:
        assert res1.stride(-1) == 1
        a.res1, a.ld_res1 = _ptr(res1), res1.stride(0)
    if res2 is not None:
        assert res2.stride(-1) == 1
        a.res2, a.ld_res2 = _ptr(res2), res2.stride(0)
    for nm, ix, rs_ in (("res1_idx", res1_idx, res1), ("res2_idx", res2_idx, res2)):
        if ix is not None:      # gathered residual: output row m adds row ix[m] of the residual matrix
            assert rs_ is not None and ix.dtype == torch.int32 and ix.is_contiguous() and ix.numel() == M
            setattr(a, nm, _ptr(ix))
    a.scale = _ptr(scale) if scale is not None else None
    a.shift = _ptr(shift) if shift is not None else None
    a.relu = 1 if relu else 0
    a.neg_slope = _ptr(neg_slope) if neg_slope is not None else None
    a.nseg = len(segs)
    for i, (c0, c1, t, mode, sw) in enumerate(segs):
        a.seg[i] = OutSeg(c0, c1, mode, sw, t.stride(0) if mode in (0, 2, 4, 5) else 0, _ptr(t))
    name = "gemm_tc" if A_split is not None and B_split is not None else "gemm"
    if EVENT_LOG is not None:
        # algo_flops: flops of the REFERENCE's contraction this launch stands for, when the launch is a factored piece of it
        EVENT_LOG.setdefault("__gemm_shapes__", []).append((name, M, K, Ncols, bool(mixed), algo_flops))
    _run(name, _lib.load().tgp_gemm, ctypes.byref(a), _stream())


def decode_max(enc_i32):
    """inverse of the order-preserving int encoding written by a column-max GEMM segment (mode 3) -> fp32 (new tensor)."""
    out = torch.empty(enc_i32.shape, dtype=torch.float32, device=enc_i32.device)
    _run("decode_max", _lib.load().tgp_decode_max, _p(enc_i32), enc_i32.numel(), _p(out), _stream())
    return out


def kpad(K):
    return _lib.load().tgp_split_kpad(K)


def mixed_kpad(K):
    return _lib.load().tgp_mixed_kpad(K)


def split_mixed(x2d, w16=False):
    """MIXED tensor-core operand of a row-major (rows, K) matrix (include/tgpose_b200.h, tgp_gemm_args.mixed):
    (rows, 2*mixed_kpad(K)) fp32 slots = 16-bit slots [fp16(x) | bf16(x) | bf16(x - fp16(x)) | unused].
    w16: the weight operand of a mixed = 2 contraction (residual slot in fp16, tgp_split_mixed_w16)."""
    assert x2d.stride(-1) == 1
    rows, K = x2d.shape
    dst = torch.empty((rows, 2 * mixed_kpad(K)), dtype=torch.float32, device=x2d.device)
    lib = _lib.load()
    _run("split_mixed", lib.tgp_split_mixed_w16 if w16 else lib.tgp_split_mixed, _p(x2d), rows, K, x2d.stride(0), _p(dst), _stream())
    return dst


def mixed_buf(M, C, device):
    kp = mixed_kpad(C)
    return (torch.zeros if kp != C else torch.empty)((M, 2 * kp), dtype=torch.float32, device=device)


def linear_fused(x2d, weight_nk, want_raw=True, want_split=False, x_split=None, w_split=None, **kw):
    """x (M,K) @ weight (Ncols,K)^T with the fused epilogue; returns (raw (M,Ncols) or None, split (M,2*Kp) or None).
    The split form is the next contraction's tensor-core operand, written by this one's epilogue."""
    M, Ncols = x2d.shape[0], weight_nk.shape[0]
    segs, raw, spl = [], None, None
    if want_raw:
        raw = torch.empty((M, Ncols), dtype=torch.float32, device=x2d.device)
        segs.append((0, Ncols, raw, 0, 0))
    if want_split:
        kp = kpad(Ncols)
        # padding columns of the operand must be zero: allocate zeroed only when there is padding
        spl = (torch.zeros if kp != Ncols else torch.empty)((M, 2 * kp), dtype=torch.float32, device=x2d.device)
        segs.append((0, Ncols, spl, 2, kp))
    gemm(x2d, weight_nk, True, segs, A_split=x_split, B_split=w_split, **kw)
    return raw, spl


def linear_nk(x2d, weight_nk, **kw):
    """x (M,K) @ weight (Ncols,K)^T -> new (M,Ncols) tensor; epilogue options as in gemm()."""
    out = torch.empty((x2d.shape[0], weight_nk.shape[0]), dtype=torch.float32, device=x2d.device)
    gemm(x2d, weight_nk, True, [(0, weight_nk.shape[0], out, 0, 0)], **kw)
    return out


# --------------------------------------------------------------------------------------- chamfer
def chamfer_forward(xyz1, xyz2, dist1, dist2, idx1, idx2, sums=None):
    B, n, _ = xyz1.shape
    m = xyz2.shape[1]
    _run("chamfer_fwd", _lib.load().tgp_chamfer_fwd, _p(xyz1), _p(xyz2), B, n, m, _p(dist1), _p(dist2), _p(idx1), _p(idx2),
                                           _p(sums), _stream())


def dcd(dist1, dist2, idx1, idx2, alpha, n_lambda, want_coef=True, non_reg=False):
    """calc_dcd tail (TDA_loss_sym_recon.py:411-450) -> loss (B), [d loss / d dist1 (B,n), d loss / d dist2 (B,m)]."""
    B, n = dist1.shape
    m = dist2.shape[1]
    loss = torch.empty(B, dtype=torch.float32, device=dist1.device)
    c1 = torch.empty_like(dist1) if want_coef else None
    c2 = torch.empty_like(dist2) if want_coef else None
    _run("dcd", _lib.load().tgp_dcd, _p(dist1), _p(dist2), _p(idx1), _p(idx2), B, n, m, float(alpha), float(n_lambda),
         1 if non_reg else 0, _p(loss), _p(c1), _p(c2), _stream())
    return loss, c1, c2


def chamfer_backward(xyz1, xyz2, gd1, gd2, idx1, idx2, g1, g2):
    B, n, _ = xyz1.shape
    m = xyz2.shape[1]
    _run("chamfer_bwd", _lib.load().tgp_chamfer_bwd, _p(xyz1), _p(xyz2), _p(gd1), _p(gd2), _p(idx1), _p(idx2), B, n, m,
                                           _p(g1), _p(g2), _stream())


# --------------------------------------------------------------------------------------- backward (SURVEY 8a')
def _ws(nbytes, device):
    return torch.empty((max(int(nbytes), 4) + 3) // 4, dtype=torch.float32, device=device)


def act_bwd(grad2d, y2d=None, scale=None, relu=False, out=None):
    """gz = grad * [y > 0] * scale: backward of a fused (affine, ReLU) epilogue.  2-D row-strided views allowed."""
    M, C = grad2d.shape
    assert grad2d.stride(1) == 1 and (y2d is None or y2d.stride(1) == 1)
    if out is None:
        out = torch.empty((M, C), dtype=torch.float32, device=grad2d.device)
    assert out.stride(1) == 1
    _run("act_bwd", _lib.load().tgp_act_bwd, _p(grad2d), grad2d.stride(0), _p(y2d), y2d.stride(0) if y2d is not None else 0,
         _p(scale), 1 if relu else 0, M, C, _p(out), out.stride(0), _stream())
    return out


def colsum(x2d, rows_per_group=None):
    """column sums per group of rows_per_group consecutive rows -> (M / rows_per_group, C)."""
    M, C = x2d.shape
    assert x2d.stride(1) == 1
    rpg = M if rows_per_group is None else rows_per_group
    lib = _lib.load()
    nb = lib.tgp_colsum_workspace(M, C, rpg)
    ws = _ws(nb, x2d.device)
    out = torch.empty((M // rpg, C), dtype=torch.float32, device=x2d.device)
    _run("colsum", lib.tgp_colsum, _p(x2d), x2d.stride(0), M, C, rpg, _p(out), _p(ws), nb, _stream())
    return out


def gather_max_bwd(grad, idx, arg, N, dfeat, rows=None, per_cloud=False, scale=1.0):
    """dfeat[b, idx[b, rows[m], arg[b,m,c]], c] += scale * grad[b,m,c]   (grad (B,C) if per_cloud)."""
    idx, bits = _idx(idx, "gather_max_bwd")
    grad = _f32c(grad, "gather_max_bwd")
    B, M, C = arg.shape
    k = idx.shape[2]
    if rows is not None:
        rows = rows.to(device=grad.device, dtype=torch.int64).contiguous()
    assert dfeat.is_contiguous() and dfeat.shape == (B, N, C)
    _run("gather_max_bwd", _lib.load().tgp_gather_max_bwd, _p(grad), 1 if per_cloud else 0, float(scale), _p(idx), bits,
         _p(rows), _p(arg), B, N, M, k, C, _p(dfeat), _stream())
    return dfeat


def scatter_add_rows(grad, index, N):
    """backward of gather_rows: (B,M,k,C) scattered into a new zero (B,N,C)."""
    grad = _f32c(grad, "scatter_add_rows")
    index, bits = _idx(index, "scatter_add_rows")
    B, M, k = index.shape
    C = grad.numel() // (B * M * k)
    out = torch.zeros((B, N, C), dtype=torch.float32, device=grad.device)
    _run("scatter_add_rows", _lib.load().tgp_scatter_add_rows, _p(grad), _p(index), bits, B, N, M, k, C, _p(out), _stream())
    return out


def layer_conv_bwd(rec, directions, support_slab, arg_slab, grad2d, B, N, S, C, d_support):
    """-> d_directions (3,S*C); d_support: a (B*N, S*C) row-strided view that is overwritten (slab column order)."""
    k = rec.shape[1]
    directions = _f32c(directions, "layer_conv_bwd")
    lib = _lib.load()
    nb = lib.tgp_layer_conv_bwd_workspace(B, S, C)
    ws = _ws(nb, rec.device)
    dd = torch.empty((3, S * C), dtype=torch.float32, device=rec.device)
    assert grad2d.stride(1) == 1 and d_support.stride(1) == 1
    _run("layer_conv_bwd", lib.tgp_layer_conv_bwd, _p(rec), _p(directions), _p(support_slab), _p(arg_slab), _p(grad2d),
         grad2d.stride(0), B, N, k, S, C, _p(d_support), d_support.stride(0), _p(dd), _p(ws), nb, _stream())
    return dd


def surface_conv_bwd(xyz, idx, directions, arg, grad2d, S, C):
    """-> d_directions (3,S*C)."""
    xyz = _f32c(xyz, "surface_conv_bwd")
    directions = _f32c(directions, "surface_conv_bwd")
    idx, bits = _idx(idx, "surface_conv_bwd")
    B, N, k = idx.shape
    lib = _lib.load()
    nb = lib.tgp_surface_conv_bwd_workspace(B, N, S, C)
    ws = _ws(nb, xyz.device)
    dd = torch.empty((3, S * C), dtype=torch.float32, device=xyz.device)
    assert grad2d.stride(1) == 1
    _run("surface_conv_bwd", lib.tgp_surface_conv_bwd, _p(xyz), _p(idx), bits, _p(directions), _p(arg), _p(grad2d),
         grad2d.stride(0), B, N, k, S, C, _p(dd), _p(ws), nb, _stream())
    return dd


def split_mixed_t(x2d):
    """TRANSPOSED, K-blocked mixed operand of a row-major (rows, K) matrix (include/tgpose_b200.h, tgp_split_mixed_t):
    a flat buffer of tgp_split_mixed_t_bytes(rows, K) bytes."""
    assert x2d.stride(1) == 1
    rows, K = x2d.shape
    nbytes = _lib.load().tgp_split_mixed_t_bytes(rows, K)
    dst = torch.empty(nbytes // 4, dtype=torch.float32, device=x2d.device)
    _run("split_mixed_t", _lib.load().tgp_split_mixed_t, _p(x2d), rows, K, x2d.stride(0), _p(dst), _stream())
    return dst


def split_tf32_t(x2d):
    """TRANSPOSED, K-blocked [tf32 | residual] operand of a row-major (rows, K) matrix for the 3xTF32 weight-gradient
    contraction (include/tgpose_b200.h, tgp_split_tf32_t): flat buffer of tgp_split_tf32_t_bytes(rows, K) bytes."""
    assert x2d.stride(1) == 1
    rows, K = x2d.shape
    nbytes = _lib.load().tgp_split_tf32_t_bytes(rows, K)
    dst = torch.empty(nbytes // 4, dtype=torch.float32, device=x2d.device)
    _run("split_tf32_t", _lib.load().tgp_split_tf32_t, _p(x2d), rows, K, x2d.stride(0), _p(dst), _stream())
    return dst


GEMM_TN_ROWMAJOR = True     # mixed weight gradients read the row-major operands in place (MN-major MMA operands)


def gemm_tn(A2d, B2d, out=None, tc=None, mixed=False, A_mixed=None, B_mixed=None):
    """A^T B: (M,K1),(M,K2) -> (K1,K2), the weight-gradient contraction.  Large shapes run on the tensor cores
    (split-K over M; 3xTF32 on transposed splits, or -- mixed -- fp16+bf16 operands read IN PLACE from the row-major mixed
    splits, which the forward / dX contractions have usually produced already: pass them as A_mixed / B_mixed), small /
    skinny ones on the exact fp32 FMA kernel."""
    M, K1 = A2d.shape
    K2 = B2d.shape[1]
    assert B2d.shape[0] == M and A2d.stride(1) == 1 and B2d.stride(1) == 1
    if out is None:
        out = torch.empty((K1, K2), dtype=torch.float32, device=A2d.device)
    assert out.stride(1) == 1
    lib = _lib.load()
    if tc is None:
        tc = TC_ENABLED and M >= 512 and K1 >= 16 and K2 >= 16
    if tc and mixed and GEMM_TN_ROWMAJOR:
        Am = A_mixed if (A_mixed is not None and A_mixed.numel()) else split_mixed(A2d)
        same = B2d.data_ptr() == A2d.data_ptr() and B2d.shape == A2d.shape and B2d.stride() == A2d.stride()
        Bm = B_mixed if (B_mixed is not None and B_mixed.numel()) else (Am if same else split_mixed(B2d))
        kpa, kpb = Am.shape[1] // 2, Bm.shape[1] // 2          # a mixed row is 2*Kp fp32 slots = 4*Kp 16-bit slots
        assert Am.shape[0] == M and Bm.shape[0] == M and kpa >= K1 and kpb >= K2
        nb = lib.tgp_gemm_tn_tc_workspace(M, K1, K2)
        ws = _ws(nb, A2d.device)
        _run("gemm_tn_tc", lib.tgp_gemm_tn_tc_rm, _p(Am), kpa, _p(Bm), kpb, M, K1, K2, _p(out), out.stride(0), _p(ws), nb, _stream())
    elif tc:
        spl = split_mixed_t if mixed else split_tf32_t
        At = spl(A2d)
        Bt = At if (B2d.data_ptr() == A2d.data_ptr() and B2d.shape == A2d.shape and B2d.stride() == A2d.stride()) \
            else spl(B2d)
        nb = lib.tgp_gemm_tn_tc_workspace(M, K1, K2)
        ws = _ws(nb, A2d.device)
        _run("gemm_tn_tc", lib.tgp_gemm_tn_tc, _p(At), _p(Bt), M, K1, K2, _p(out), out.stride(0), 1 if mixed else 0,
             _p(ws), nb, _stream())
    else:
        nb = lib.tgp_gemm_tn_workspace(M, K1, K2)
        ws = _ws(nb, A2d.device)
        _run("gemm_tn", lib.tgp_gemm_tn, _p(A2d), A2d.stride(0), _p(B2d), B2d.stride(0), M, K1, K2, _p(out),
             out.stride(0), _p(ws), nb, _stream())
    return out


def matmul_kn(x2d, w_kn, **kw):
    """x (M,K) @ w (K,Ncols) -> new (M,Ncols) (w row-major, e.g. dY @ W for a Conv1d weight W (out,in))."""
    out = torch.empty((x2d.shape[0], w_kn.shape[1]), dtype=torch.float32, device=x2d.device)
    gemm(x2d, w_kn, False, [(0, w_kn.shape[1], out, 0, 0)], **kw)
    return out


# --------------------------------------------------------------------------------------- heads in training
def colsumsq_dev(x2d, mu):
    """sum over rows of (x - mu)^2 -> (C,)."""
    M, C = x2d.shape
    assert x2d.stride(1) == 1
    lib = _lib.load()
    nb = lib.tgp_bn_workspace(M, C)
    ws = _ws(nb, x2d.device)
    out = torch.empty(C, dtype=torch.float32, device=x2d.device)
    _run("colsumsq_dev", lib.tgp_colsumsq_dev, _p(x2d), x2d.stride(0), M, C, _p(mu), _p(out), _p(ws), nb, _stream())
    return out


def affine_act(z2d, scale, shift, slope, want_raw=True, want_split=False, mixed=False):
    """act(z * scale + shift) -> (raw (M,C) or None, split operand or None): (M, 2*kpad(C)) [tf32 | residual], or the
    MIXED layout (M, 2*mixed_kpad(C)) when mixed."""
    M, C = z2d.shape
    assert z2d.stride(1) == 1
    raw = torch.empty((M, C), dtype=torch.float32, device=z2d.device) if want_raw else None
    spl = None
    if want_split:
        spl = mixed_buf(M, C, z2d.device) if mixed else _split_buf(M, C, z2d.device)
    _run("affine_act", _lib.load().tgp_affine_act, _p(z2d), z2d.stride(0), _p(scale), _p(shift), float(slope), M, C,
         _p(raw), C, _p(spl), mixed_kpad(C) if mixed else kpad(C), 1 if mixed else 0, _stream())
    return raw, spl


def bn_bwd(dy2d, y2d, z2d, mean, invstd, gamma, slope, want_mixed=False, scale=None, shift=None):
    """-> (dz (M,C), dbeta (C,), dgamma (C,)) of y = act(BN_train(z)); with want_mixed also dz as the mixed operand of
    the dx contraction (4th result; None when the shape does not take the 128-bit kernel)."""
    M, C = z2d.shape
    dy2d = dy2d if dy2d.stride(1) == 1 else dy2d.contiguous()
    lib = _lib.load()
    nb = lib.tgp_bn_workspace(M, C)
    ws = _ws(nb, z2d.device)
    dz = torch.empty((M, C), dtype=torch.float32, device=z2d.device)
    dbeta = torch.empty(C, dtype=torch.float32, device=z2d.device)
    dgamma = torch.empty(C, dtype=torch.float32, device=z2d.device)
    dzm = None
    if want_mixed and C % 4 == 0 and all(t.stride(0) % 4 == 0 and t.data_ptr() % 16 == 0 for t in (dy2d, y2d, z2d)):
        dzm = mixed_buf(M, C, z2d.device)
    _run("bn_bwd", lib.tgp_bn_bwd, _p(dy2d), dy2d.stride(0), _p(y2d), y2d.stride(0), _p(z2d), z2d.stride(0), _p(mean),
         _p(invstd), _p(gamma), _p(scale), _p(shift), float(slope), M, C, _p(dz), C, _p(dzm), _p(dbeta), _p(dgamma), _p(ws),
         nb, _stream())
    if want_mixed:
        return dz, dbeta, dgamma, dzm
    return dz, dbeta, dgamma
