"""Tensor-level wrappers over the C ABI (one Python function per exported kernel).

Everything here takes/returns CUDA torch tensors, allocates outputs with torch (device memory is
PyTorch's job) and enqueues work on torch's current stream.  No math is done in PyTorch.
"""
from __future__ import annotations

from ctypes import byref
from typing import Optional

import torch

from . import native as nv
from .native import ACT_GELU, ACT_NONE, ACT_RELU, GemmOut, LinearArgs, LnArgs, Operand  # noqa: F401


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


class Split:
    """split-bf16 matrix: planes [2, rows, pitch] (hi, lo), logical width `cols`."""

    __slots__ = ("t", "rows", "cols", "pitch")

    def __init__(self, rows: int, cols: int, device, pitch: Optional[int] = None, zero: bool = False):
        self.rows, self.cols = rows, cols
        self.pitch = pitch if pitch is not None else _round_up(cols, 64)
        alloc = torch.zeros if zero else torch.empty
        self.t = alloc((2, rows, self.pitch), dtype=torch.bfloat16, device=device)

    @property
    def plane(self) -> int:
        return self.rows * self.pitch

    def ptr(self, col: int = 0, row: int = 0) -> int:
        return self.t.data_ptr() + 2 * (row * self.pitch + col)

    def operand(self, rows=None, k=None, col=0, row=0, nb1=0, b1_stride=0, nb2=0, b2_stride=0) -> Operand:
        return Operand(self.ptr(col, row), self.plane, rows if rows is not None else self.rows,
                       k if k is not None else self.cols, self.pitch, nb1, nb2, b1_stride, b2_stride)

    def float(self) -> torch.Tensor:  # debugging / tests only
        return (self.t[0].float() + self.t[1].float())[:, : self.cols]


def pack_weight(w: torch.Tensor) -> Split:
    """fp32 [N,K] -> split-bf16 (done once at model load)."""
    w = w.detach().float().contiguous()
    s = Split(w.shape[0], w.shape[1], w.device)
    split_f32(w, s)
    return s


# ------------------------------------------------------------------------------------------------
def fps(xyz: torch.Tensor, num_samples: int):
    B, N, _ = xyz.shape
    idx = torch.empty((B, num_samples), dtype=torch.int64, device=xyz.device)
    centers = torch.empty((B, num_samples, 3), dtype=torch.float32, device=xyz.device)
    nbytes = nv.lib().psam_fps_workspace_bytes(B, N, num_samples)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=xyz.device) if nbytes else None
    nv.check(nv.lib().psam_fps_f32(nv.ptr(xyz), B, N, num_samples, nv.ptr(idx), nv.ptr(centers), nv.ptr(ws), nv.stream()), "fps")
    return idx, centers


def knn(query: torch.Tensor, key: torch.Tensor, k: int, want_d2: bool = False):
    B, Q, _ = query.shape
    N = key.shape[1]
    idx = torch.empty((B, Q, k), dtype=torch.int64, device=query.device)
    d2 = torch.empty((B, Q, k), dtype=torch.float32, device=query.device) if want_d2 else None
    nv.check(nv.lib().psam_knn_f32(nv.ptr(query), nv.ptr(key), B, Q, N, k, nv.ptr(idx), nv.ptr(d2), nv.stream()), "knn")
    return idx, d2


def group_gather(xyz, feats, centers, knn_idx, radius=None, center_idx=None):
    """center_idx [B,G] int64: centralize_features=True (C more channels feats[idx] - feats[center])."""
    B, N, _ = xyz.shape
    B2, _, C = feats.shape
    _, G, K = knn_idx.shape
    out = torch.empty((B2, G, K, 3 + C + (C if center_idx is not None else 0)), dtype=torch.float32, device=xyz.device)
    nv.check(nv.lib().psam_group_gather_f32(nv.ptr(xyz), nv.ptr(feats), nv.ptr(centers), nv.ptr(knn_idx), nv.ptr(center_idx), B, B2 // B,
                                            N, G, K, C, float(radius) if radius else 0.0, nv.ptr(out), nv.stream()), "group_gather")
    return out


def nn_index(query, key):
    """Nearest key of every query point, one cloud at a time (first index on ties): idx [B,Nq] int64."""
    B, Nq, _ = query.shape
    Nk = key.shape[1]
    idx = torch.empty((B, Nq), dtype=torch.int64, device=query.device)
    dist = torch.empty((B, Nq), dtype=torch.float32, device=query.device)
    for b in range(B):
        nv.check(nv.lib().psam_nn_distance_f32(nv.ptr(query[b]), nv.ptr(key[b]), Nq, Nk, nv.ptr(dist[b]), nv.ptr(idx[b]), nv.stream()),
                 "nn_distance")
    return idx


def voronoi_features(xyz, centers, nn_idx, feats, want_split: bool = False):
    """[unit direction to the nearest centre, distance, features] per point: fp32 [B2,N,4+C] (+ split copy, pitch 64)."""
    B, N, _ = xyz.shape
    B2, _, C = feats.shape
    out = torch.empty((B2, N, 4 + C), dtype=torch.float32, device=xyz.device)
    sp = Split(B2 * N, 4 + C, xyz.device) if want_split else None
    nv.check(nv.lib().psam_voronoi_features_f32(nv.ptr(xyz), nv.ptr(centers), nv.ptr(nn_idx), nv.ptr(feats), B, B2 // B, N,
                                                centers.shape[1], C, nv.ptr(out), sp.ptr() if sp is not None else None,
                                                sp.plane if sp is not None else 0, sp.pitch if sp is not None else 0, nv.stream()),
             "voronoi_features")
    return (out, sp) if want_split else out


def scatter_amax(x, nn_idx, G: int):
    """x [B,N,D], nn_idx [B,N] -> [B,G,D] maximum per Voronoi cell (empty cells 0)."""
    B, N, D = x.shape
    y = torch.empty((B, G, D), dtype=torch.float32, device=x.device)
    nv.check(nv.lib().psam_scatter_amax_f32(nv.ptr(x), nv.ptr(nn_idx), B, N, G, D, nv.ptr(y), nv.stream()), "scatter_amax")
    return y


def knn3_interp(xyz, centers):
    B, N, _ = xyz.shape
    G = centers.shape[1]
    idx = torch.empty((B, N, 3), dtype=torch.int64, device=xyz.device)
    w = torch.empty((B, N, 3), dtype=torch.float32, device=xyz.device)
    nv.check(nv.lib().psam_knn3_interp_f32(nv.ptr(xyz), nv.ptr(centers), B, N, G, nv.ptr(idx), nv.ptr(w), nv.stream()), "knn3_interp")
    return idx, w


def nn_distance(query: torch.Tensor, key: torch.Tensor):
    """Squared distance from each query [n1,3] to its nearest key [n2,3]."""
    q, k = query.float().contiguous(), key.float().contiguous()
    d = torch.empty(q.shape[0], dtype=torch.float32, device=q.device)
    nv.check(nv.lib().psam_nn_distance_f32(nv.ptr(q), nv.ptr(k), q.shape[0], k.shape[0], nv.ptr(d), None, nv.stream()), "nn_distance")
    return d


def border_prompt(coords: torch.Tensor, gt_masks: torch.Tensor, pred_logits: Optional[torch.Tensor] = None,
                  pred_masks: Optional[torch.Tensor] = None, from_error_region: bool = False,
                  status: Optional[torch.Tensor] = None):
    """Batched farthest-from-border prompt sampling (psam_border_prompt_f32).  coords [B,N,3], gt_masks [B,M,N] bool,
    prediction as logits [B*M,N] or bool masks [B*M,N] or neither.  Returns (xyz [B*M,1,3], labels [B*M,1] bool, status)."""
    B, M, N = gt_masks.shape
    c = coords.float().contiguous()
    g = gt_masks.contiguous().view(torch.uint8) if gt_masks.dtype == torch.bool else gt_masks.to(torch.uint8).contiguous()
    lg = pred_logits.float().contiguous() if pred_logits is not None else None
    pm = None
    if pred_masks is not None:
        pm = pred_masks.contiguous().view(torch.uint8) if pred_masks.dtype == torch.bool else pred_masks.to(torch.uint8).contiguous()
    dev = c.device
    xyz = torch.empty((B * M, 1, 3), dtype=torch.float32, device=dev)
    lab = torch.empty((B * M, 1), dtype=torch.uint8, device=dev)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(nv.lib().psam_border_prompt_workspace_bytes(B, M, N), dtype=torch.uint8, device=dev)
    nv.check(nv.lib().psam_border_prompt_f32(nv.ptr(c), nv.ptr(g), nv.ptr(lg), nv.ptr(pm), B, M, N, int(from_error_region), nv.ptr(xyz),
                                             nv.ptr(lab), nv.ptr(status), nv.ptr(ws), nv.stream()), "border_prompt")
    return xyz, lab.view(torch.bool), status


GEMM_TILE_HINT = 0  # 0 = latency-optimal tiles, 1 = SM-time-optimal tiles (set by PipelinedPredictor)
GEMM_TILE_BN = 0    # 32..256: explicit tile width (experiments / tests)
# psam_gemm_out.variant (experiment switches, see include/psam_b200.h); PSAM_GEMM_VARIANT seeds it once at import
GV_2CTA, GV_BK32, GV_SCALAR_EPI, GV_DUAL, GV_NO_DUAL, GV_PERSIST, GV_NO_PERSIST, GV_TWO_ISSUERS = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40, 0x80
GEMM_VARIANT = int(__import__("os").environ.get("PSAM_GEMM_VARIANT", "0"), 0)


def gemm_raw(a: Operand, w: Operand, out: GemmOut, passes: int = 3, split_k: int = 1):
    if out.tile_hint == 0:
        out.tile_hint = GEMM_TILE_BN if GEMM_TILE_BN else GEMM_TILE_HINT
    if out.variant == 0:
        out.variant = GEMM_VARIANT
    nv.check(nv.lib().psam_gemm_bf16x3(byref(a), byref(w), byref(out), passes, split_k, nv.stream()), "gemm_bf16x3")


def gemm(a: Split, w: Split, *, bias=None, out_f32: Optional[torch.Tensor] = None, out_split: Optional[Split] = None,
         resid: Optional[torch.Tensor] = None, act: int = ACT_NONE, alpha: float = 1.0, accumulate: bool = False,
         split_k: int = 1, passes: int = 3, rows: Optional[int] = None, swiglu: bool = False,
         gmax: Optional[torch.Tensor] = None, group_rows: int = 0, rowdot=None, stats_out: Optional[torch.Tensor] = None,
         ln_fold=None):
    """out = act(alpha * a @ w^T + bias (+ resid)); a [M,K], w [N,K] split-bf16."""
    M = rows if rows is not None else a.rows
    o = GemmOut()
    o.out_f32 = nv.ptr(out_f32)
    o.ldo = out_f32.stride(-2) if out_f32 is not None else 0
    o.out_hi = out_split.ptr() if out_split is not None else None
    o.out_plane = out_split.plane if out_split is not None else 0
    o.ldo_s = out_split.pitch if out_split is not None else 0
    o.bias = nv.ptr(bias)
    o.resid = nv.ptr(resid)
    o.alpha = alpha
    o.act = act
    o.accumulate = int(accumulate)
    o.swiglu = int(swiglu)
    if gmax is not None:
        o.gmax, o.ld_gmax, o.group_rows = nv.ptr(gmax), gmax.shape[-1], group_rows
    if rowdot is not None:  # (w [Z,C,N], out [Z,C,rows] zero-filled)
        rw, ro = rowdot
        o.rd_w, o.rd_out, o.rd_rows, o.rd_c = nv.ptr(rw), nv.ptr(ro), ro.shape[-1], ro.shape[-2]
    o.stats_out = nv.ptr(stats_out)
    if ln_fold is not None:  # (stats [M,2], c [N], H, eps): LayerNorm over the K axis folded into this GEMM
        st, c, hh, eps = ln_fold
        o.ln_stats, o.ln_c, o.ln_h, o.ln_eps = nv.ptr(st), nv.ptr(c), int(hh), float(eps)
    gemm_raw(a.operand(rows=M), w.operand(), o, passes, split_k)


def gemm_rowln(a: Split, w: Split, gamma, beta, eps: float, out: Split, *, gbias: Optional[torch.Tensor] = None, group_rows: int = 0,
               act: int = ACT_NONE, passes: int = 3):
    """out = act(LayerNorm(a @ w^T + gbias[row // group_rows])) as split-bf16; K <= 128, N in {256, 512} (psam_gemm_rowln_bf16x3)."""
    ao, wo = a.operand(), w.operand()
    nv.check(nv.lib().psam_gemm_rowln_bf16x3(byref(ao), byref(wo), nv.ptr(gbias), gbias.shape[-1] if gbias is not None else 0, group_rows,
                                             nv.ptr(gamma), nv.ptr(beta), float(eps), act, out.ptr(), out.plane, out.pitch, passes,
                                             nv.stream()), "gemm_rowln_bf16x3")


def gemm_rowln_supported(K: int, N: int) -> bool:
    return K <= 128 and N in (256, 512)


def linear_f32(x, w, b=None, *, x2=None, r=None, act=ACT_NONE, out=None, M=None, K=None, ldx=None, Z=1, x_z=0, x2_z=0,
               w_z=0, b_z=0, r_z=0, y_z=0, ldy=None, x_off=0):
    """fp32 SIMT linear (see psam_linear_f32). x [.., K] flattened to rows unless M/ldx given."""
    N = w.shape[-2]
    Kd = K if K is not None else w.shape[-1]
    if M is None:
        M = x.numel() // x.shape[-1]
    if out is None:
        out = torch.empty((Z * M, N) if Z > 1 else (M, N), dtype=torch.float32, device=x.device)
    a = LinearArgs()
    a.x = nv.ptr(x) + 4 * x_off
    a.ldx = ldx if ldx is not None else x.shape[-1]
    a.x_z = x_z
    a.x2 = nv.ptr(x2)
    a.x2_z = x2_z
    a.w = nv.ptr(w)
    a.ldw = w.shape[-1]
    a.w_z = w_z
    a.b = nv.ptr(b)
    a.b_z = b_z
    a.r = nv.ptr(r)
    a.r_z = r_z
    a.y = nv.ptr(out)
    a.ldy = ldy if ldy is not None else N
    a.y_z = y_z
    a.M, a.N, a.K, a.Z, a.act = M, N, Kd, Z, act
    nv.check(nv.lib().psam_linear_f32(byref(a), nv.stream()), "linear_f32")
    return out


def layernorm(x, gamma, beta, eps, *, rows=None, D=None, r=None, gbias=None, group_rows=0, act=ACT_NONE,
              out_f32: Optional[torch.Tensor] = None, out_split: Optional[Split] = None, ldx=None, padded: bool = False,
              post_add: Optional[torch.Tensor] = None, out_split2: Optional[Split] = None):
    D = D if D is not None else x.shape[-1]
    rows = rows if rows is not None else x.numel() // x.shape[-1]
    a = LnArgs()
    a.x, a.ldx = nv.ptr(x), (ldx if ldx is not None else x.shape[-1])
    a.r, a.ldr = nv.ptr(r), (r.shape[-1] if r is not None else 0)
    a.gbias, a.ld_gbias, a.group_rows = nv.ptr(gbias), (gbias.shape[-1] if gbias is not None else 0), group_rows
    a.gamma, a.beta, a.eps = nv.ptr(gamma), nv.ptr(beta), eps
    a.rows, a.D, a.act = rows, D, act
    a.y, a.ldy = nv.ptr(out_f32), (out_f32.shape[-1] if out_f32 is not None else 0)
    if out_split is not None:
        a.y_hi, a.y_plane, a.ldy_s, a.pitch = out_split.ptr(), out_split.plane, out_split.pitch, out_split.pitch
    a.padded = int(padded)
    if out_split2 is not None:  # second split output = split(y + post_add)
        a.post_add, a.ld_post = nv.ptr(post_add), post_add.shape[-1]
        a.y2_hi, a.y2_plane, a.ldy2_s = out_split2.ptr(), out_split2.plane, out_split2.pitch
    a.policy = GEMM_TILE_HINT  # same switch as the GEMM tile policy: 1 while capturing the pipelined predictor's graphs
    nv.check(nv.lib().psam_layernorm_f32(byref(a), nv.stream()), "layernorm")


def swiglu_ln(gx: torch.Tensor, H: int, x_off: int, gamma, beta, eps, out: Split):
    rows = gx.shape[0]
    nv.check(nv.lib().psam_swiglu_ln(nv.ptr(gx), gx.shape[1], x_off, rows, H, nv.ptr(gamma), nv.ptr(beta), eps,
                                     out.ptr(), out.plane, out.pitch, out.pitch, nv.stream()), "swiglu_ln")


def small_in_linear(x, W, b, gamma, beta, eps, use_ln: bool, act: int, out: Split):
    rows, Cin = x.numel() // x.shape[-1], x.shape[-1]
    nv.check(nv.lib().psam_small_in_linear(nv.ptr(x), rows, Cin, nv.ptr(W), nv.ptr(b), nv.ptr(gamma), nv.ptr(beta), eps,
                                           int(use_ln), act, W.shape[0], out.ptr(), out.plane, out.pitch, nv.stream()),
             "small_in_linear")


def group_max(x: torch.Tensor, groups: int, K: int, out_f32=None, out_split: Optional[Split] = None):
    D = x.shape[-1]
    nv.check(nv.lib().psam_group_max(nv.ptr(x), D, groups, K, D, nv.ptr(out_f32), D,
                                     out_split.ptr() if out_split is not None else None,
                                     out_split.plane if out_split is not None else 0,
                                     out_split.pitch if out_split is not None else 0, nv.stream()), "group_max")


def softmax_split(s: torch.Tensor, L: int, scale: float, out: Split):
    rows = s.numel() // s.shape[-1]
    nv.check(nv.lib().psam_softmax_split(nv.ptr(s), s.shape[-1], rows, L, scale, out.ptr(), out.plane, out.pitch, nv.stream()),
             "softmax_split")


def posenc(coords, gauss, labels=None, emb0=None, emb1=None, bad_flag=None):
    rows = coords.numel() // 3
    F = gauss.shape[1]
    out = torch.empty(coords.shape[:-1] + (2 * F,), dtype=torch.float32, device=coords.device)
    nv.check(nv.lib().psam_posenc_f32(nv.ptr(coords), rows, nv.ptr(gauss), F, nv.ptr(labels), nv.ptr(emb0), nv.ptr(emb1),
                                      nv.ptr(out), nv.ptr(bad_flag), nv.stream()), "posenc")
    return out


def attention_f32(q, k, v, Z, Lq, Lk, H, dh, q_off=0, k_off=0, v_off=0):
    """q / k / v may be column windows of wider row-major tensors: *_off = first column, the row stride is the tensor's width."""
    o = torch.empty((Z * Lq, H * dh), dtype=torch.float32, device=q.device)
    nv.check(nv.lib().psam_attention_f32(nv.ptr(q) + 4 * q_off, nv.ptr(k) + 4 * k_off, nv.ptr(v) + 4 * v_off, nv.ptr(o), Z, Lq, Lk, H,
                                         dh, q.shape[-1], k.shape[-1], v.shape[-1], H * dh, nv.stream()), "attention_f32")
    return o


def add_bcast(a, b, chunk=None, rep=1):
    out = torch.empty_like(a)
    n = a.numel()
    nv.check(nv.lib().psam_add_bcast_f32(nv.ptr(a), nv.ptr(b), n, chunk if chunk else n, rep, b.numel(), nv.ptr(out), nv.stream()),
             "add_bcast")
    return out


def split_f32(x: torch.Tensor, out: Split, add: Optional[torch.Tensor] = None):
    """out = split-bf16(x (+ add))."""
    rows = x.numel() // x.shape[-1]
    if add is None:
        nv.check(nv.lib().psam_split_f32(nv.ptr(x), x.shape[-1], rows, x.shape[-1], out.ptr(), out.plane, out.pitch, out.pitch,
                                         nv.stream()), "split_f32")
    else:
        nv.check(nv.lib().psam_split_add_f32(nv.ptr(x), nv.ptr(add), x.shape[-1], rows, x.shape[-1], out.ptr(), out.plane, out.pitch,
                                             out.pitch, nv.stream()), "split_add_f32")


# ------------------------------------------------------------------------------------------------
# automatic mask generation: bit-packed candidate masks (bit j of word w = point 32 w + j)
def mask_words(N: int) -> int:
    return (N + 31) // 32


def mask_stats(logits: torch.Tensor, iou_pred: torch.Tensor, mask_threshold: float, stability_offset: float,
               pred_iou_thresh: float, stability_thresh: float, out=None, row0: int = 0):
    """logits [R, N] (any leading shape flattened to rows), iou_pred [R] -> (bits [R, W] int32, area [R] int32,
    stability [R] fp32, keep [R] uint8).  out = (bits, area, stability, keep) of a larger candidate table: rows
    row0 .. row0 + R are written (psam_mask_stats_f32)."""
    N = logits.shape[-1]
    R = logits.numel() // N
    if logits.dtype != torch.float32 or iou_pred.dtype != torch.float32 or iou_pred.numel() != R:
        raise ValueError("mask_stats: fp32 logits [R, N] and fp32 iou_pred [R] expected")
    if not logits.is_contiguous() or not iou_pred.is_contiguous():
        raise ValueError("mask_stats: logits and iou_pred must be contiguous")
    W = mask_words(N)
    dev = logits.device
    if out is None:
        out = (torch.empty((R, W), dtype=torch.int32, device=dev), torch.empty(R, dtype=torch.int32, device=dev),
               torch.empty(R, dtype=torch.float32, device=dev), torch.empty(R, dtype=torch.uint8, device=dev))
        row0 = 0
    bits, area, stab, keep = out
    if bits.shape[1] != W or row0 < 0 or row0 + R > bits.shape[0] or any(t.shape[0] != bits.shape[0] for t in (area, stab, keep)):
        raise ValueError("mask_stats: output table too small for rows row0 .. row0 + R")
    nv.check(nv.lib().psam_mask_stats_f32(nv.ptr(logits), nv.ptr(iou_pred), R, N, float(mask_threshold), float(stability_offset),
                                          float(pred_iou_thresh), float(stability_thresh), nv.ptr(bits) + 4 * W * row0,
                                          nv.ptr(area) + 4 * row0, nv.ptr(stab) + 4 * row0, nv.ptr(keep) + row0, nv.stream()),
             "mask_stats_f32")
    return out


def mask_iou(a_bits: torch.Tensor, b_bits: torch.Tensor, want_inter: bool = False):
    """IoU [Ka, Kb] fp32 (and the int32 intersections) of two bit-mask sets [Ka, W], [Kb, W] (psam_mask_iou_u32)."""
    if a_bits.dtype != torch.int32 or b_bits.dtype != torch.int32 or a_bits.shape[1] != b_bits.shape[1]:
        raise ValueError("mask_iou: int32 bit masks with the same number of words expected")
    a, b = a_bits.contiguous(), b_bits.contiguous()
    Ka, W = a.shape
    Kb = b.shape[0]
    iou = torch.empty((Ka, Kb), dtype=torch.float32, device=a.device)
    inter = torch.empty((Ka, Kb), dtype=torch.int32, device=a.device) if want_inter else None
    nv.check(nv.lib().psam_mask_iou_u32(nv.ptr(a), Ka, nv.ptr(b), Kb, W, nv.ptr(iou), nv.ptr(inter), nv.stream()), "mask_iou_u32")
    return (iou, inter) if want_inter else iou


def mask_nms(bits: torch.Tensor, area: torch.Tensor, score: torch.Tensor, keep: torch.Tensor, nms_thresh: float):
    """Greedy NMS of the candidates with keep != 0 (psam_mask_nms): keep_idx [K] int32 (kept candidates in score order,
    -1 after the last) and kept_count [1] int32, both on the device (nothing is read back)."""
    K, W = bits.shape
    if bits.dtype != torch.int32 or area.dtype != torch.int32 or score.dtype != torch.float32 or keep.dtype != torch.uint8:
        raise ValueError("mask_nms: int32 bits / areas, fp32 scores and uint8 keep flags expected")
    dev = bits.device
    keep_idx = torch.empty(K, dtype=torch.int32, device=dev)
    count = torch.empty(1, dtype=torch.int32, device=dev)
    ws = torch.empty(nv.lib().psam_mask_nms_workspace_bytes(K, W), dtype=torch.uint8, device=dev)
    nv.check(nv.lib().psam_mask_nms(nv.ptr(bits), nv.ptr(area), nv.ptr(score), nv.ptr(keep), K, W, float(nms_thresh),
                                    nv.ptr(keep_idx), nv.ptr(count), nv.ptr(ws), nv.stream()), "mask_nms")
    return keep_idx, count


def mask_unpack(bits: torch.Tensor, N: int, rows: Optional[torch.Tensor] = None) -> torch.Tensor:
    """bool [k, N] masks of the bit rows `rows` (int32 [k]; None: all rows) (psam_mask_unpack_u8)."""
    r = rows.to(torch.int32).contiguous() if rows is not None else None
    k = r.numel() if r is not None else bits.shape[0]
    out = torch.empty((k, N), dtype=torch.uint8, device=bits.device)
    if k:
        nv.check(nv.lib().psam_mask_unpack_u8(nv.ptr(bits), bits.shape[1], nv.ptr(r), k, N, nv.ptr(out), nv.stream()), "mask_unpack_u8")
    return out.view(torch.bool)
