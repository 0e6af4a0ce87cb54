"""Execution engine: runs the Point-SAM hot path through the C ABI kernels.

The modules in ``pc_sam.model`` only hold parameters (reference state-dict layout); their ``forward``
methods call the ``run_*`` functions here.  Weights are re-packed (split-bf16, fused qkv, padded SwiGLU)
lazily and cached per module; the cache is keyed on parameter storage/version so ``load_state_dict``,
``safetensors.load_model`` and ``.cuda()`` are picked up automatically.
"""
from __future__ import annotations

import contextlib
import math
import os
import threading
from ctypes import byref
from typing import Optional

import torch

from . import native as nv
from . import ops
from .ops import ACT_GELU, ACT_NONE, ACT_RELU, Split

FUSED_ATTENTION = True
FUSED_ATTENTION_LONG = os.environ.get("PSAM_FUSED_ATTENTION_LONG", "1") != "0"
ATTENTION_TWOPASS = os.environ.get("PSAM_ATTENTION_TWOPASS", "0") == "1"  # A/B: first-generation two-pass kernels
FUSED_INNER_LN = os.environ.get("PSAM_FUSED_INNER_LN", "1") != "0"  # SwiGLU.norm folded into the fc1 / fc2 GEMM epilogues
FUSED_MASK_DOT = os.environ.get("PSAM_FUSED_MASK_DOT", "1") != "0"
# the decoder's projections of the G patch rows (keys of the two-way transformer, 512 rows at c2) on the tcgen05 GEMM instead of
# the fp32 SIMT linear; the token-side (<= 16 rows) projections stay SIMT
DECODER_TC = os.environ.get("PSAM_DECODER_TC", "1") != "0"
# norm1 / norm2 / fc_norm folded into the qkv / fc1 / out_proj GEMMs: the producer of the residual stream (pos_embed, proj and
# fc2 GEMM epilogues) writes x as fp32 + split-bf16 and accumulates the row statistics, so no LayerNorm kernel runs in a block
# EVA-giant heads (dh = 88) on the fused attention kernel (64 + 24 columns, zero padded by TMA).  Full-size parity of the 40-block
# model holds with it (tests/test_gpu_model.py::test_config5_full_size_vs_fp32_oracle_on_gpu, both LayerNorm forms); c5: 213 -> 243
# clouds/s (profiles/r02_bench_c5_fused_dh88.json).  PSAM_FUSED_ATTENTION_DH88=0 selects the unfused tensor-core path (QK^T GEMM,
# softmax, V transpose, PV GEMM) it replaces.
FUSED_ATTENTION_DH88 = os.environ.get("PSAM_FUSED_ATTENTION_DH88", "1") != "0"
FUSED_ROW_LN = os.environ.get("PSAM_FUSED_ROW_LN", "1") != "0"  # mini-PointNet conv2[0] + LayerNorm + GELU in one row-complete GEMM
FUSED_BLOCK_LN = os.environ.get("PSAM_FUSED_BLOCK_LN", "1") != "0"  # capability: pack the LayerNorm-folded weights as well
# When the LayerNorm-free form of the ViT blocks is USED (both weight sets are packed):
#   "auto"   - only inside PipelinedPredictor captures with >= 8 clouds in flight.  MEASURED (c2): at depth 8 the folded form
#              ties with the LayerNorm kernels (642 vs 645 clouds/s) at 49 fewer launches per cloud; at depth 4 it loses
#              (543 vs 574) and single-stream latency is 4.0 vs 3.4 ms, because the fold needs split_k = 1 on proj / fc2.
#   "always" / "never" - forced (tests, experiments; PSAM_BLOCK_LN_POLICY).
BLOCK_LN_POLICY = os.environ.get("PSAM_BLOCK_LN_POLICY", "auto")
_fold_ctx = threading.local()


@contextlib.contextmanager
def block_ln_fold(active: bool):
    """Scope inside which policy "auto" resolves to `active` (set by the pipelined predictor while it captures its graphs)."""
    prev = getattr(_fold_ctx, "active", False)
    _fold_ctx.active = bool(active)
    try:
        yield
    finally:
        _fold_ctx.active = prev


def _use_block_ln_fold() -> bool:
    if BLOCK_LN_POLICY == "always":
        return True
    if BLOCK_LN_POLICY == "never":
        return False
    return bool(getattr(_fold_ctx, "active", False))
PASSES = 3  # split-bf16 (fp32-parity) mode; 1 = plain bf16 (fails the 1e-3 parity bound, see DESIGN.md)


def _fingerprint(module) -> tuple:
    return tuple((p.data_ptr(), p._version) for p in module.parameters()) + tuple(
        (b.data_ptr(), b._version) for b in module.buffers())


def _cached(module, builder):
    fp = _fingerprint(module)
    c = module.__dict__.get("_psam_packed")
    if c is None or c[0] != fp:
        if any(not p.is_cuda for p in module.parameters()):
            raise RuntimeError("psam_b200: model parameters must live on a CUDA device (no CPU path)")
        c = (fp, builder(module))
        module.__dict__["_psam_packed"] = c
    return c[1]


def _f32(t):
    return t.detach().float().contiguous()


def _split_k_for(M: int, N: int, K: int) -> int:
    """Fill the 148 SMs when the output has few tiles (small-batch inference)."""
    tiles = ((M + 127) // 128) * ((N + 127) // 128)
    kb = (K + 63) // 64
    s = 1
    while tiles * s * 2 <= 148 and s * 2 <= max(1, kb // 4):
        s *= 2
    return s


# ------------------------------------------------------------------------------------------------
# PatchEncoder (mini-PointNet), pc_sam/model/common.py:477-506
# ------------------------------------------------------------------------------------------------
class _PackedPatchEncoder:
    def __init__(self, m):
        c1, c2 = m.conv1, m.conv2
        self.h0 = c1[0].out_features
        self.h1 = c2[0].out_features
        self.cout = c2[3].out_features
        self.w10, self.b10 = _f32(c1[0].weight), _f32(c1[0].bias)
        self.w10s = ops.pack_weight(c1[0].weight) if c1[0].in_features > 16 else None
        self.g11, self.be11, self.eps11 = _f32(c1[1].weight), _f32(c1[1].bias), c1[1].eps
        self.w13, self.b13 = ops.pack_weight(c1[3].weight), _f32(c1[3].bias)
        w20 = c2[0].weight.detach().float()
        self.w20a = ops.pack_weight(w20[:, : self.h0])  # acts on the pooled (broadcast) half
        self.w20b = ops.pack_weight(w20[:, self.h0:])   # acts on the per-point half
        self.b20 = _f32(c2[0].bias)
        self.g21, self.be21, self.eps21 = _f32(c2[1].weight), _f32(c2[1].bias), c2[1].eps
        self.w23, self.b23 = ops.pack_weight(c2[3].weight), _f32(c2[3].bias)


def run_patch_encoder(m, patches: torch.Tensor, want_split: bool = False):
    """patches [B,L,K,Cin] fp32 -> [B,L,Cout] fp32 (and optionally the split-bf16 copy)."""
    pk = _cached(m, _PackedPatchEncoder)
    B, L, K, Cin = patches.shape
    dev = patches.device
    R, BG = B * L * K, B * L
    h1 = Split(R, pk.h0, dev)
    if Cin <= 16 and pk.h0 % 32 == 0 and pk.h0 <= 512:
        ops.small_in_linear(patches, pk.w10, pk.b10, pk.g11, pk.be11, pk.eps11, True, ACT_GELU, h1)
    else:
        # wide inputs (second level of PatchEmbedHier: 128 + 3 channels): conv1[0] on the tensor cores, LayerNorm + GELU after it
        ps = Split(R, Cin, dev)
        ops.split_f32(patches.reshape(R, Cin), ps)
        u = torch.empty((R, pk.h0), dtype=torch.float32, device=dev)
        ops.gemm(ps, pk.w10s, bias=pk.b10, out_f32=u, passes=PASSES)
        ops.layernorm(u, pk.g11, pk.be11, pk.eps11, act=ACT_GELU, out_split=h1)
    x1s = Split(R, pk.h0, dev)
    y1s = Split(BG, pk.h0, dev)
    fused_max = K % 32 == 0  # the max-pool over the K rows of a group runs inside the GEMM epilogue
    if fused_max:
        y1 = torch.full((BG, pk.h0), float("-inf"), dtype=torch.float32, device=dev)
        ops.gemm(h1, pk.w13, bias=pk.b13, out_split=x1s, gmax=y1, group_rows=K, passes=PASSES)
        ops.split_f32(y1, y1s)
    else:
        x1 = torch.empty((R, pk.h0), dtype=torch.float32, device=dev)
        ops.gemm(h1, pk.w13, bias=pk.b13, out_f32=x1, out_split=x1s, passes=PASSES)
        ops.group_max(x1, BG, K, out_split=y1s)
    # conv2[0] on cat([max, x]) = W_a max + W_b x + b : the pooled half is computed once per group
    t = torch.empty((BG, pk.h1), dtype=torch.float32, device=dev)
    ops.gemm(y1s, pk.w20a, bias=pk.b20, out_f32=t, passes=PASSES)
    h2 = Split(R, pk.h1, dev)
    if FUSED_ROW_LN and ops.gemm_rowln_supported(pk.h0, pk.h1):
        # conv2[0] on the per-point half + group bias + LayerNorm + GELU in ONE kernel: a CTA owns the full row, the fp32
        # pre-activation (R x h1 floats: 64 MB per cloud at c2) never reaches memory
        ops.gemm_rowln(x1s, pk.w20b, pk.g21, pk.be21, pk.eps21, h2, gbias=t, group_rows=K, act=ACT_GELU, passes=PASSES)
    else:
        x2 = torch.empty((R, pk.h1), dtype=torch.float32, device=dev)
        ops.gemm(x1s, pk.w20b, out_f32=x2, passes=PASSES)
        ops.layernorm(x2, pk.g21, pk.be21, pk.eps21, gbias=t, group_rows=K, act=ACT_GELU, out_split=h2)
    embs = Split(BG, pk.cout, dev) if want_split else None
    if fused_max:
        emb = torch.full((B, L, pk.cout), float("-inf"), dtype=torch.float32, device=dev)
        ops.gemm(h2, pk.w23, bias=pk.b23, gmax=emb.view(BG, pk.cout), group_rows=K, passes=PASSES)
        if want_split:
            ops.split_f32(emb.view(BG, pk.cout), embs)
    else:
        x3 = torch.empty((R, pk.cout), dtype=torch.float32, device=dev)
        ops.gemm(h2, pk.w23, bias=pk.b23, out_f32=x3, passes=PASSES)
        emb = torch.empty((B, L, pk.cout), dtype=torch.float32, device=dev)
        ops.group_max(x3, BG, K, out_f32=emb, out_split=embs)
    return (emb, embs) if want_split else emb


# ------------------------------------------------------------------------------------------------
# KNNGrouper, pc_sam/model/common.py:59-123
# ------------------------------------------------------------------------------------------------
def run_knn_grouper(g, xyz, features, use_fps=True):
    xyz32 = xyz.float().contiguous()
    feats = features.float().contiguous()
    B, N, _ = xyz32.shape
    if N < g.num_groups:
        raise RuntimeError("sample_farthest_points: number of points must be >= num_samples")
    if use_fps:
        fps_idx, centers = ops.fps(xyz32, g.num_groups)
    else:  # `xyz` is already FPS-ordered: the first num_groups points are the centres (common.py:93-96)
        fps_idx = torch.arange(g.num_groups, device=xyz.device).expand(B, -1).contiguous()
        centers = xyz32[:, : g.num_groups].contiguous()
    knn_idx, _ = ops.knn(centers, xyz32, g.group_size)
    groups = ops.group_gather(xyz32, feats, centers, knn_idx, g.radius,
                              center_idx=fps_idx if g.centralize_features else None)  # common.py:116-118
    return dict(features=groups, centers=centers, knn_idx=knn_idx, fps_idx=fps_idx)


# ------------------------------------------------------------------------------------------------
# Voronoi tokenizer: NNGrouper (common.py:190-212), PatchEmbedNN + Block (pc_encoder.py:147-197)
# ------------------------------------------------------------------------------------------------
def run_nn_grouper(g, xyz, features, want_split: bool = False):
    xyz32 = xyz.float().contiguous()
    feats = features.float().contiguous()
    if xyz32.shape[1] < g.num_groups:
        raise RuntimeError("sample_farthest_points: number of points must be >= num_samples")
    _, centers = ops.fps(xyz32, g.num_groups)
    nn_idx = ops.nn_index(xyz32, centers)  # knn_points(xyz, centers, 1): nearest centre of every point
    out = ops.voronoi_features(xyz32, centers, nn_idx, feats, want_split=want_split)
    gf, sp = out if want_split else (out, None)
    d = dict(features=gf, centers=centers, nn_idx=nn_idx)
    if want_split:
        d["_features_split"] = sp
    return d


class _PackedResBlock:
    """Block (pc_encoder.py:147-162): x + Linear(LayerNorm(GELU(Linear(LayerNorm(x)))))."""

    def __init__(self, blk):
        lin1, ln_mid, lin2 = blk.mlp[0], blk.mlp[2], blk.mlp[3]
        self.g0, self.b0, self.eps0 = _f32(blk.norm.weight), _f32(blk.norm.bias), blk.norm.eps
        self.w1, self.bb1 = ops.pack_weight(lin1.weight), _f32(lin1.bias)
        self.g1, self.b1, self.eps1 = _f32(ln_mid.weight), _f32(ln_mid.bias), ln_mid.eps
        self.w2, self.bb2 = ops.pack_weight(lin2.weight), _f32(lin2.bias)
        self.hid = lin1.out_features


class _PackedPatchEmbedNN:
    def __init__(self, m):
        self.hid = m.in_proj.out_features
        self.win, self.bin = ops.pack_weight(m.in_proj.weight), _f32(m.in_proj.bias)
        self.blocks1 = [_PackedResBlock(b) for b in m.blocks1]
        self.blocks2 = [_PackedResBlock(b) for b in m.blocks2]
        self.g, self.b, self.eps = _f32(m.norm.weight), _f32(m.norm.bias), m.norm.eps
        self.wout, self.bout = ops.pack_weight(m.out_proj.weight), _f32(m.out_proj.bias)


def _run_res_blocks(blocks, x: torch.Tensor):
    """x fp32 [rows, D], updated in place."""
    rows, D = x.shape
    dev = x.device
    for pb in blocks:
        xn = Split(rows, D, dev)
        ops.layernorm(x, pb.g0, pb.b0, pb.eps0, out_split=xn)
        u = torch.empty((rows, pb.hid), dtype=torch.float32, device=dev)
        ops.gemm(xn, pb.w1, bias=pb.bb1, out_f32=u, act=ACT_GELU, passes=PASSES)
        un = Split(rows, pb.hid, dev)
        ops.layernorm(u, pb.g1, pb.b1, pb.eps1, out_split=un)
        ops.gemm(un, pb.w2, bias=pb.bb2, out_f32=x, resid=x, passes=PASSES)


def run_patch_embed_hier(m, coords, features):
    """PatchEmbedHier.forward (pc_encoder.py:200-239): PointNet++-style two-level tokenizer; the second level groups the
    first level's centres (already in FPS order: use_fps=False) with the first level's embeddings as features."""
    patches1 = run_knn_grouper(m.grouper1, coords, features)
    x1 = run_patch_encoder(m.patch_encoder1, patches1["features"])
    patches1["embeddings"] = x1
    patches2 = run_knn_grouper(m.grouper2, patches1["centers"], x1, use_fps=False)
    patches2["embeddings"] = run_patch_encoder(m.patch_encoder2, patches2["features"])
    return [patches1, patches2]


def run_patch_embed_nn(m, coords, features):
    """PatchEmbedNN.forward (pc_encoder.py:181-197): per-point residual MLPs, maximum per Voronoi cell, per-cell MLPs."""
    pk = _cached(m, _PackedPatchEmbedNN)
    patches = run_nn_grouper(m.grouper, coords, features, want_split=True)
    fs = patches.pop("_features_split")
    B, N, _ = patches["features"].shape
    G, dev = m.grouper.num_groups, coords.device
    x = torch.empty((B * N, pk.hid), dtype=torch.float32, device=dev)
    ops.gemm(fs, pk.win, bias=pk.bin, out_f32=x, passes=PASSES)
    _run_res_blocks(pk.blocks1, x)
    y = ops.scatter_amax(x.view(B, N, pk.hid), patches["nn_idx"], G).view(B * G, pk.hid)
    _run_res_blocks(pk.blocks2, y)
    yn = Split(B * G, pk.hid, dev)
    ops.layernorm(y, pk.g, pk.b, pk.eps, out_split=yn)
    emb = torch.empty((B, G, m.out_channels), dtype=torch.float32, device=dev)
    ops.gemm(yn, pk.wout, bias=pk.bout, out_f32=emb.view(B * G, -1), passes=PASSES)
    patches["embeddings"] = emb
    return patches


# ------------------------------------------------------------------------------------------------
# timm EVA / EVA02 blocks + PointCloudEncoder, pc_sam/model/pc_encoder.py:84-145
# ------------------------------------------------------------------------------------------------
def _is_noop(m) -> bool:
    """Identity-like sub-module of an inference-only block (None, nn.Identity, Dropout / DropPath with p == 0 or in eval mode)."""
    if m is None or isinstance(m, torch.nn.Identity):
        return True
    p = getattr(m, "p", getattr(m, "drop_prob", None))
    if p is not None and isinstance(m, torch.nn.Module) and not any(True for _ in m.parameters()):
        return float(p) == 0.0 or not m.training
    return False


def _refuse(what: str):
    raise NotImplementedError(
        f"psam_b200: the transformer block carries {what}, which this engine does not execute - results would be silently "
        "wrong.  Modelled: timm EvaBlock as Point-SAM calls it (pre-LN, rope=None, no LayerScale, SwiGLU+inner LN or GELU Mlp).")


_BLOCK_CHILDREN = {"norm1", "attn", "norm2", "mlp", "drop_path1", "drop_path2"}
_ATTN_CHILDREN = {"q_proj", "k_proj", "v_proj", "qkv", "proj", "norm", "q_norm", "k_norm", "attn_drop", "proj_drop"}
_ATTN_PARAMS = {"q_bias", "v_bias", "k_bias"}
_SWIGLU_CHILDREN = {"fc1_g", "fc1_x", "act", "drop1", "norm", "fc2", "drop2"}
_MLP_CHILDREN = {"fc1", "act", "drop1", "norm", "fc2", "drop2"}


def validate_eva_block(blk) -> None:
    """Refuse module trees this engine does not model (timm/models/eva.py EvaBlock / EvaAttention options that
    Point-SAM's released configs leave off): LayerScale (gamma_1/gamma_2), attention inner scale-norm (attn.norm),
    q/k norms, rotary embedding stored on the module, unknown parameterised children, non-GELU / non-SiLU activations,
    GluMlp.  Pure Python (no CUDA), unit-tested on CPU with fake modules."""
    LN = torch.nn.LayerNorm
    for g in ("gamma_1", "gamma_2"):
        if getattr(blk, g, None) is not None:
            _refuse(f"LayerScale ({g})")
    for n in ("norm1", "norm2"):
        m = getattr(blk, n, None)
        if not isinstance(m, LN) or m.weight is None or m.bias is None:
            _refuse(f"{n} = {type(m).__name__} (expected an affine LayerNorm)")
    for n in ("drop_path1", "drop_path2"):
        if not _is_noop(getattr(blk, n, None)):
            _refuse(f"an active {n}")
    for name, child in blk.named_children():
        if name not in _BLOCK_CHILDREN and any(True for _ in child.parameters()):
            _refuse(f"an unknown parameterised sub-module '{name}'")
    for name, _ in blk.named_parameters(recurse=False):
        if name not in ("gamma_1", "gamma_2"):
            _refuse(f"an unknown block parameter '{name}'")
    at = getattr(blk, "attn", None)
    if at is None or not hasattr(at, "num_heads") or getattr(at, "proj", None) is None:
        _refuse("an attention module without num_heads / proj")
    for n in ("norm", "q_norm", "k_norm"):
        if not _is_noop(getattr(at, n, None)):
            _refuse(f"attn.{n} = {type(getattr(at, n)).__name__} (inner scale-norm / qk-norm)")
    if getattr(at, "rope", None) is not None:
        _refuse("a rotary position embedding on attn.rope")
    for n in ("attn_drop", "proj_drop"):
        if not _is_noop(getattr(at, n, None)):
            _refuse(f"an active attn.{n}")
    for name, child in at.named_children():
        if name not in _ATTN_CHILDREN and any(True for _ in child.parameters()):
            _refuse(f"an unknown parameterised sub-module 'attn.{name}'")
    for name, _ in at.named_parameters(recurse=False):
        if name not in _ATTN_PARAMS:
            _refuse(f"an unknown attention parameter 'attn.{name}'")
    fused = getattr(at, "qkv", None) is not None
    if fused:
        if getattr(at.qkv, "bias", None) is not None:
            _refuse("attn.qkv with its own bias (timm keeps the q/v bias in q_bias / v_bias)")
        if (getattr(at, "q_bias", None) is None) != (getattr(at, "v_bias", None) is None):
            _refuse("attn.q_bias without attn.v_bias")
    else:
        for n in ("q_proj", "k_proj", "v_proj"):
            if getattr(at, n, None) is None:
                _refuse(f"neither attn.qkv nor attn.{n}")
    mlp = getattr(blk, "mlp", None)
    if hasattr(mlp, "fc1_g") and hasattr(mlp, "fc1_x"):
        allowed = _SWIGLU_CHILDREN
        nm = getattr(mlp, "norm", None)
        if not isinstance(nm, LN) or nm.weight is None or nm.bias is None:
            _refuse(f"SwiGLU.norm = {type(nm).__name__} (expected the affine inner LayerNorm of scale_mlp=True)")
        act = getattr(mlp, "act", None)
        if act is not None and not isinstance(act, torch.nn.SiLU):
            _refuse(f"SwiGLU activation {type(act).__name__} (expected SiLU)")
    elif hasattr(mlp, "fc1") and hasattr(mlp, "fc2"):
        allowed = _MLP_CHILDREN
        if mlp.fc1.out_features != mlp.fc2.in_features:
            _refuse("a gated GluMlp (fc1 twice as wide as fc2's input)")
        if not _is_noop(getattr(mlp, "norm", None)):
            _refuse(f"Mlp.norm = {type(mlp.norm).__name__}")
        act = getattr(mlp, "act", None)
        if act is not None and not (isinstance(act, torch.nn.GELU) and getattr(act, "approximate", "none") == "none"):
            _refuse(f"Mlp activation {act!r} (expected exact-erf GELU)")
    else:
        _refuse(f"an MLP of type {type(mlp).__name__}")
    for name, child in mlp.named_children():
        if name not in allowed and any(True for _ in child.parameters()):
            _refuse(f"an unknown parameterised sub-module 'mlp.{name}'")
    for n in ("drop1", "drop2"):
        if not _is_noop(getattr(mlp, n, None)):
            _refuse(f"an active mlp.{n}")


def validate_transformer(tr) -> list:
    """pc_encoder.py:136-142 applies pos_drop, blocks, norm, fc_norm.  Returns the LayerNorms to run after the blocks
    (timm: exactly one of norm / fc_norm is a LayerNorm, the other nn.Identity)."""
    if not _is_noop(getattr(tr, "pos_drop", None)):
        _refuse("an active pos_drop")
    tail = []
    for n in ("norm", "fc_norm"):
        m = getattr(tr, n, None)
        if isinstance(m, torch.nn.LayerNorm) and m.weight is not None and m.bias is not None:
            tail.append(m)
        elif not _is_noop(m):
            _refuse(f"transformer.{n} = {type(m).__name__}")
    for blk in tr.blocks:
        validate_eva_block(blk)
    return tail


def _fold_ln(w: torch.Tensor, b: torch.Tensor, norm):
    """(W * gamma packed split-bf16, c = (W * gamma) 1, b' = W beta + b) in fp64 -> fp32."""
    wd = w.detach().double()
    g, be = norm.weight.detach().double(), norm.bias.detach().double()
    wg = wd * g[None, :]
    return ops.pack_weight(wg.float()), wg.sum(dim=1).float().contiguous(), (wd @ be + b.detach().double()).float().contiguous()


class _PackedBlock:
    def __init__(self, blk, D):
        validate_eva_block(blk)
        at = blk.attn
        self.H, self.dh = at.num_heads, D // at.num_heads
        self.g1, self.b1, self.eps1 = _f32(blk.norm1.weight), _f32(blk.norm1.bias), blk.norm1.eps
        self.g2, self.b2, self.eps2 = _f32(blk.norm2.weight), _f32(blk.norm2.bias), blk.norm2.eps
        dev = blk.norm1.weight.device
        zeros = torch.zeros(D, dtype=torch.float32, device=dev)
        if getattr(at, "qkv", None) is not None:
            wqkv = at.qkv.weight.detach().float()
            qb = at.q_bias.detach().float() if getattr(at, "q_bias", None) is not None else zeros
            vb = at.v_bias.detach().float() if getattr(at, "v_bias", None) is not None else zeros
            bqkv = torch.cat([qb, zeros, vb])
        else:
            wqkv = torch.cat([at.q_proj.weight, at.k_proj.weight, at.v_proj.weight]).detach().float()
            bias = lambda lin: lin.bias.detach().float() if lin.bias is not None else zeros
            bqkv = torch.cat([bias(at.q_proj), bias(at.k_proj), bias(at.v_proj)])
        self.wqkv, self.bqkv = ops.pack_weight(wqkv), bqkv.contiguous()
        # the folded forms live in the GEMM's vectorised epilogue (whole 32-column chunks): D and the MLP width must be
        # multiples of 32, otherwise the block keeps its LayerNorm kernels
        mlp_w = blk.mlp.fc1_g.out_features if hasattr(blk.mlp, "fc1_g") else blk.mlp.fc1.out_features
        self.fold_block = FUSED_BLOCK_LN and D % 32 == 0 and (hasattr(blk.mlp, "fc1_g") or mlp_w % 32 == 0)
        if self.fold_block:
            # LN(x) @ W^T + b = rstd * (x @ (W gamma)^T - mean * (W gamma) 1) + (W beta + b)
            self.wqkv_f, self.cqkv, self.bqkv_f = _fold_ln(wqkv, bqkv, blk.norm1)
        self.wproj, self.bproj = ops.pack_weight(at.proj.weight), _f32(at.proj.bias)
        mlp = blk.mlp
        self.swiglu = hasattr(mlp, "fc1_g")
        if self.swiglu:
            Hd = mlp.fc1_g.out_features
            Hp = (Hd + 63) // 64 * 64
            w1 = torch.zeros((2 * Hp, D), dtype=torch.float32, device=dev)
            b1 = torch.zeros(2 * Hp, dtype=torch.float32, device=dev)
            # gate / value rows interleaved (2i, 2i+1): the GEMM epilogue computes silu(g) * x directly
            w1[0:2 * Hd:2], w1[1:2 * Hd:2] = mlp.fc1_g.weight.detach().float(), mlp.fc1_x.weight.detach().float()
            b1[0:2 * Hd:2], b1[1:2 * Hd:2] = mlp.fc1_g.bias.detach().float(), mlp.fc1_x.bias.detach().float()
            self.hid, self.hp = Hd, Hp
            self.w1, self.bb1 = ops.pack_weight(w1), b1
            if self.fold_block:
                self.w1_f, self.c1, self.bb1_f = _fold_ln(w1, b1, blk.norm2)
            gpad = torch.zeros(Hp, dtype=torch.float32, device=dev)
            bpad = torch.zeros(Hp, dtype=torch.float32, device=dev)
            gpad[:Hd], bpad[:Hd] = mlp.norm.weight.detach().float(), mlp.norm.bias.detach().float()
            self.gn, self.bn, self.epsn = gpad, bpad, mlp.norm.eps  # zero-padded to Hp for the float4 LN path
            w2 = torch.zeros((D, Hp), dtype=torch.float32, device=dev)
            w2[:, :Hd] = mlp.fc2.weight.detach().float()
            self.fold_ln = FUSED_INNER_LN
            if self.fold_ln:
                # fc2(LN(h)) = rstd * (h @ (W2 * gamma)^T - mean * (W2 @ gamma)) + (W2 @ beta + b2): the normalisation becomes a
                # per-row scale / per-column offset in the fc2 epilogue, fed by row sums the fc1 epilogue accumulates
                w2d = w2.double()
                self.w2 = ops.pack_weight((w2d * gpad.double()[None, :]).float())
                self.c2 = (w2d @ gpad.double()).float().contiguous()
                self.bb2 = (w2d @ bpad.double() + mlp.fc2.bias.detach().double()).float().contiguous()
            else:
                self.w2, self.bb2 = ops.pack_weight(w2), _f32(mlp.fc2.bias)
        else:
            self.hid = mlp.fc1.out_features
            self.w1, self.bb1 = ops.pack_weight(mlp.fc1.weight), _f32(mlp.fc1.bias)
            if self.fold_block:
                self.w1_f, self.c1, self.bb1_f = _fold_ln(mlp.fc1.weight.detach().float(), mlp.fc1.bias.detach().float(), blk.norm2)
            self.w2, self.bb2 = ops.pack_weight(mlp.fc2.weight), _f32(mlp.fc2.bias)


class _PackedEncoder:
    def __init__(self, enc):
        D = enc.transformer_dim
        self.D = D
        self.wpp, self.bpp = ops.pack_weight(enc.patch_proj.weight), _f32(enc.patch_proj.bias)
        self.wpos0, self.bpos0 = _f32(enc.pos_embed[0].weight), _f32(enc.pos_embed[0].bias)
        self.wpos2, self.bpos2 = ops.pack_weight(enc.pos_embed[2].weight), _f32(enc.pos_embed[2].bias)
        self.tail = [(_f32(m.weight), _f32(m.bias), m.eps) for m in validate_transformer(enc.transformer)]
        self.blocks = [_PackedBlock(b, D) for b in enc.transformer.blocks]
        self.wout, self.bout = ops.pack_weight(enc.out_proj.weight), _f32(enc.out_proj.bias)
        self.fold_block = (FUSED_BLOCK_LN and len(self.tail) == 1 and all(b.fold_block for b in self.blocks)
                           and enc.embed_dim % 32 == 0)
        for b in self.blocks:
            b.fold_block = self.fold_block
        if self.fold_block:
            m = validate_transformer(enc.transformer)[0]
            self.wout_f, self.cout, self.bout_f = _fold_ln(enc.out_proj.weight.detach().float(), enc.out_proj.bias.detach().float(), m)
            self.eps_tail = m.eps


def _attention_unfused(qkv: Split, att: Split, B: int, L: int, H: int, dh: int, D: int, dev):
    """Fallback for head dims the fused kernels do not cover (EVA-giant dh=88)."""
    # V^T per (cloud, head): [B, H, dh, Lp]
    Lp = (L + 63) // 64 * 64
    vt = Split(B * H * dh, L, dev, pitch=Lp, zero=(Lp != L))
    nv.check(nv.lib().psam_transpose_split(qkv.ptr(2 * D), qkv.plane, qkv.pitch, dh, L * qkv.pitch,
                                           vt.ptr(), vt.plane, vt.pitch, dh * Lp, H * dh * Lp,
                                           L, dh, H, B, nv.stream()), "transpose_split")
    # S = Q K^T  (batched over heads and clouds), fp32 [B, H, L, L]
    s = torch.empty((B * H * L, L), dtype=torch.float32, device=dev)
    qa = qkv.operand(rows=L, k=dh, col=0, nb1=H, b1_stride=dh, nb2=B, b2_stride=L * qkv.pitch)
    ka = qkv.operand(rows=L, k=dh, col=D, nb1=H, b1_stride=dh, nb2=B, b2_stride=L * qkv.pitch)
    o = ops.GemmOut()
    o.out_f32, o.ldo, o.out_b1, o.out_b2 = nv.ptr(s), L, L * L, H * L * L
    o.alpha = 1.0
    ops.gemm_raw(qa, ka, o, PASSES, 1)
    p = Split(B * H * L, L, dev, pitch=Lp, zero=(Lp != L))
    ops.softmax_split(s, L, dh ** -0.5, p)
    # O = P V  -> heads recombined into [M, D]
    pa = p.operand(rows=L, k=L, nb1=H, b1_stride=L * Lp, nb2=B, b2_stride=H * L * Lp)
    va = vt.operand(rows=dh, k=L, nb1=H, b1_stride=dh * Lp, nb2=B, b2_stride=H * dh * Lp)
    o2 = ops.GemmOut()
    o2.out_hi, o2.out_plane, o2.ldo_s, o2.outs_b1, o2.outs_b2 = att.ptr(), att.plane, att.pitch, dh, L * att.pitch
    o2.alpha = 1.0
    ops.gemm_raw(pa, va, o2, PASSES, 1)


def _run_block(pb: _PackedBlock, x: torch.Tensor, B: int, L: int, D: int, fold=None):
    """x fp32 [B*L, D], updated in place (pre-LN residual block, rope=None).
    fold = (xs, st_in, st_mid, st_out): LayerNorm-free form - xs is the split-bf16 copy of x and st_in its row statistics
    (both written by the GEMM that last produced x); proj refreshes xs + st_mid, fc2 refreshes xs + st_out."""
    dev = x.device
    M = B * L
    H, dh = pb.H, pb.dh
    qkv = Split(M, 3 * D, dev)
    if fold is not None:
        xs, st_in, st_mid, st_out = fold[:4]
        ops.gemm(xs, pb.wqkv_f, bias=pb.bqkv_f, out_split=qkv, passes=PASSES, ln_fold=(st_in, pb.cqkv, D, pb.eps1))
    else:
        xn = Split(M, D, dev)
        ops.layernorm(x, pb.g1, pb.b1, pb.eps1, out_split=xn)
        ops.gemm(xn, pb.wqkv, bias=pb.bqkv, out_split=qkv, passes=PASSES)
    att = Split(M, D, dev)
    if FUSED_ATTENTION and (dh == 64 or (dh == 88 and not ATTENTION_TWOPASS and FUSED_ATTENTION_DH88)) and (L <= 512 or FUSED_ATTENTION_LONG):
        # fused tcgen05 attention: S stays in tensor memory (L <= 512) or streams through a ring of TMEM slots in two
        # sweeps (longer rows); V^T is read as an MN-major operand
        mk = lambda col: qkv.operand(rows=L, k=dh, col=col, nb1=H, b1_stride=dh, nb2=B, b2_stride=L * qkv.pitch)
        qa, ka, va = mk(0), mk(D), mk(2 * D)
        entry = nv.lib().psam_attention_bf16x3_twopass if ATTENTION_TWOPASS else nv.lib().psam_attention_bf16x3
        nv.check(entry(byref(qa), byref(ka), byref(va), att.ptr(), att.plane, att.pitch, dh, L * att.pitch, dh ** -0.5,
                       nv.stream()), "attention_bf16x3")
    else:
        _attention_unfused(qkv, att, B, L, H, dh, D, dev)
    # x += proj(att)
    if fold is not None:
        # one writer per element (no split-K): the epilogue also emits split-bf16(x) and the row statistics for norm2
        ops.gemm(att, pb.wproj, bias=pb.bproj, out_f32=x, resid=x, out_split=xs, stats_out=st_mid, passes=PASSES)
        _run_mlp_folded(pb, x, xs, st_mid, st_out, M, D, dev, stats=fold[4] if len(fold) > 4 else None)
        return
    sk = _split_k_for(M, D, D)
    if sk > 1:
        ops.gemm(att, pb.wproj, bias=pb.bproj, out_f32=x, accumulate=True, split_k=sk, passes=PASSES)
    else:
        ops.gemm(att, pb.wproj, bias=pb.bproj, out_f32=x, resid=x, passes=PASSES)
    # MLP
    ops.layernorm(x, pb.g2, pb.b2, pb.eps2, out_split=xn)
    fold = None
    if pb.swiglu and pb.fold_ln:
        # h = silu(fc1_g) * fc1_x leaves the fc1 epilogue as split-bf16 together with its row sums; SwiGLU.norm is applied
        # inside the fc2 epilogue (no LayerNorm kernel, no fp32 copy of h)
        stats = torch.zeros((M, 2), dtype=torch.float32, device=dev)
        h = Split(M, pb.hp, dev, pitch=pb.hp)
        ops.gemm(xn, pb.w1, bias=pb.bb1, out_split=h, passes=PASSES, swiglu=True, stats_out=stats)
        fold = (stats, pb.c2, pb.hid, pb.epsn)
    elif pb.swiglu:
        hf = torch.empty((M, pb.hp), dtype=torch.float32, device=dev)
        ops.gemm(xn, pb.w1, bias=pb.bb1, out_f32=hf, passes=PASSES, swiglu=True)  # hf = silu(fc1_g) * fc1_x
        h = Split(M, pb.hp, dev, pitch=pb.hp)  # columns hid..hp are zero-filled by the LayerNorm kernel
        ops.layernorm(hf, pb.gn, pb.bn, pb.epsn, D=pb.hid, out_split=h, padded=True)
    else:
        h = Split(M, pb.hid, dev)
        ops.gemm(xn, pb.w1, bias=pb.bb1, out_split=h, act=ACT_GELU, passes=PASSES)
    sk = _split_k_for(M, D, pb.hid)
    if sk > 1:
        ops.gemm(h, pb.w2, bias=pb.bb2, out_f32=x, accumulate=True, split_k=sk, passes=PASSES, ln_fold=fold)
    else:
        ops.gemm(h, pb.w2, bias=pb.bb2, out_f32=x, resid=x, passes=PASSES, ln_fold=fold)


def _run_mlp_folded(pb: _PackedBlock, x, xs, st_mid, st_out, M, D, dev, stats=None):
    """x += mlp(norm2(x)) with norm2 folded into fc1 (and SwiGLU.norm into fc2); fc2 refreshes xs and st_out."""
    if pb.swiglu:
        if not pb.fold_ln:
            raise RuntimeError("PSAM_FUSED_BLOCK_LN requires PSAM_FUSED_INNER_LN")
        if stats is None:
            stats = torch.zeros((M, 2), dtype=torch.float32, device=dev)
        h = Split(M, pb.hp, dev, pitch=pb.hp)
        ops.gemm(xs, pb.w1_f, bias=pb.bb1_f, out_split=h, passes=PASSES, swiglu=True, stats_out=stats,
                 ln_fold=(st_mid, pb.c1, D, pb.eps2))
        ops.gemm(h, pb.w2, bias=pb.bb2, out_f32=x, resid=x, out_split=xs, stats_out=st_out, passes=PASSES,
                 ln_fold=(stats, pb.c2, pb.hid, pb.epsn))
    else:
        h = Split(M, pb.hid, dev)
        ops.gemm(xs, pb.w1_f, bias=pb.bb1_f, out_split=h, act=ACT_GELU, passes=PASSES, ln_fold=(st_mid, pb.c1, D, pb.eps2))
        ops.gemm(h, pb.w2, bias=pb.bb2, out_f32=x, resid=x, out_split=xs, stats_out=st_out, passes=PASSES)


def run_pc_encoder(enc, coords, features):
    pk = _cached(enc, _PackedEncoder)
    patches = run_knn_grouper(enc.patch_embed.grouper, coords, features)
    emb, embs = run_patch_encoder(enc.patch_embed.patch_encoder, patches["features"], want_split=True)
    patches["embeddings"] = emb
    B, L, _ = emb.shape
    D, dev = pk.D, emb.device
    M = B * L
    x = torch.empty((M, D), dtype=torch.float32, device=dev)
    ops.gemm(embs, pk.wpp, bias=pk.bpp, out_f32=x, passes=PASSES)
    pos = Split(M, pk.wpos0.shape[0], dev)
    ops.small_in_linear(patches["centers"], pk.wpos0, pk.bpos0, None, None, 0.0, False, ACT_GELU, pos)
    if pk.fold_block and _use_block_ln_fold():
        # LayerNorm-free encoder: every GEMM that writes the residual stream also writes its split-bf16 copy and row
        # statistics; norm1 / norm2 / fc_norm are applied inside the consuming GEMMs' epilogues
        nb = len(pk.blocks)
        # one memset for all row statistics of the step: residual stream (2 nb + 1) and SwiGLU hidden rows (nb)
        st = torch.zeros((3 * nb + 1, M, 2), dtype=torch.float32, device=dev)
        xs = Split(M, D, dev)
        ops.gemm(pos, pk.wpos2, bias=pk.bpos2, out_f32=x, resid=x, out_split=xs, stats_out=st[0], passes=PASSES)
        for i, pb in enumerate(pk.blocks):
            _run_block(pb, x, B, L, D, fold=(xs, st[2 * i], st[2 * i + 1], st[2 * i + 2], st[2 * nb + 1 + i]))
        out = torch.empty((B, L, enc.embed_dim), dtype=torch.float32, device=dev)
        ops.gemm(xs, pk.wout_f, bias=pk.bout_f, out_f32=out.view(M, -1), passes=PASSES,
                 ln_fold=(st[2 * nb], pk.cout, D, pk.eps_tail))
        return out, patches
    ops.gemm(pos, pk.wpos2, bias=pk.bpos2, out_f32=x, resid=x, passes=PASSES)
    for pb in pk.blocks:
        _run_block(pb, x, B, L, D)
    xn = Split(M, D, dev)
    for i, (g_, b_, e_) in enumerate(pk.tail):  # transformer.norm / transformer.fc_norm (pc_encoder.py:141-142)
        if i + 1 < len(pk.tail):
            ops.layernorm(x, g_, b_, e_, out_f32=x)
        else:
            ops.layernorm(x, g_, b_, e_, out_split=xn)
    if not pk.tail:
        ops.split_f32(x, xn)
    out = torch.empty((B, L, enc.embed_dim), dtype=torch.float32, device=dev)
    ops.gemm(xn, pk.wout, bias=pk.bout, out_f32=out.view(M, -1), passes=PASSES)
    return out, patches


# ------------------------------------------------------------------------------------------------
# prompt encoders, pc_sam/model/prompt_encoder.py:13-133
# ------------------------------------------------------------------------------------------------
_bad_flags = {}
_flag_ctx = threading.local()


@contextlib.contextmanager
def flag_scope(range_flag: Optional[torch.Tensor] = None, sampler: Optional[torch.Tensor] = None):
    """Route the device-side error flags of everything run inside the scope to caller-owned tensors.  The graph
    predictors give every lane its own flags (captured into its CUDA graph), so a bad request is reported for that
    ticket only and never leaks into an unrelated eager call on the same GPU."""
    prev = (getattr(_flag_ctx, "range", None), getattr(_flag_ctx, "sampler", None))
    _flag_ctx.range, _flag_ctx.sampler = range_flag, sampler
    try:
        yield
    finally:
        _flag_ctx.range, _flag_ctx.sampler = prev


def bad_flag(device) -> torch.Tensor:
    o = getattr(_flag_ctx, "range", None)
    if o is not None:
        return o
    f = _bad_flags.get(device)
    if f is None:
        f = torch.zeros(1, dtype=torch.int32, device=device)
        _bad_flags[device] = f
    return f


def raise_if_out_of_range(device):
    """The reference raises inside PositionEmbeddingRandom.forward (host sync, prompt_encoder.py:44-46)."""
    if torch.cuda.is_current_stream_capturing():
        return
    f = bad_flag(device)
    if int(f.item()) != 0:
        f.zero_()
        raise ValueError("Input coordinates must be normalized to [-1, 1].")


_sampler_flags = {}


def sampler_flag(device) -> torch.Tensor:
    """Sticky device flag set by psam_border_prompt_f32 when a mask has no border to sample from."""
    o = getattr(_flag_ctx, "sampler", None)
    if o is not None:
        return o
    f = _sampler_flags.get(device)
    if f is None:
        f = torch.zeros(1, dtype=torch.int32, device=device)
        _sampler_flags[device] = f
    return f


def raise_if_sampler_failed(device):
    """The reference fails in torch.stack([... None ...]) (common.py:433); checked once per prompt iteration, or once
    per replay when the loop runs as a CUDA graph."""
    if torch.cuda.is_current_stream_capturing():
        return
    f = sampler_flag(device)
    if int(f.item()) != 0:
        f.zero_()
        raise RuntimeError("prompt sampling: a ground-truth mask is empty or covers the whole cloud (no border to sample from)")


def run_pos_embedding(pe_layer, coords, labels=None, emb0=None, emb1=None, check=True):
    c = coords.float().contiguous()
    lab = labels.to(torch.int32).contiguous() if labels is not None else None
    out = ops.posenc(c, _f32(pe_layer.positional_encoding_gaussian_matrix), lab, emb0, emb1, bad_flag(c.device))
    if check:
        raise_if_out_of_range(c.device)
    return out


def run_point_encoder(pe, points, labels, check=True):
    assert points.shape[:-1] == labels.shape
    return run_pos_embedding(pe.pe_layer, points, labels, _f32(pe.point_embeddings[0].weight),
                             _f32(pe.point_embeddings[1].weight), check=check)


def run_mask_encoder(me, masks, coords, centers, knn_idx, center_idx=None):
    if masks is None:
        return me.no_mask_embed.weight.reshape(1, 1, -1).expand(centers.shape[0], centers.shape[1], -1)
    if me.centralize_features and center_idx is None:
        raise RuntimeError("MaskEncoder(centralize_features=True) needs center_idx (the FPS indices of the centres)")
    m = masks.detach().float().contiguous().unsqueeze(-1)
    # centralize_features (prompt_encoder.py:121-130 -> common.py:181-185): one more channel, logit - logit at the group's centre
    groups = ops.group_gather(coords.float().contiguous(), m, centers, knn_idx, me.radius,
                              center_idx=center_idx.contiguous() if me.centralize_features else None)
    return run_patch_encoder(me.patch_encoder, groups)


# ------------------------------------------------------------------------------------------------
# two-way transformer + mask decoder, pc_sam/model/transformer.py, mask_decoder.py
# ------------------------------------------------------------------------------------------------
class _PackedAttn:
    def __init__(self, a):
        self.H = a.num_heads
        self.inner = a.internal_dim
        self.wq, self.bq = _f32(a.q_proj.weight), _f32(a.q_proj.bias)
        self.wk, self.bk = _f32(a.k_proj.weight), _f32(a.k_proj.bias)
        self.wv, self.bv = _f32(a.v_proj.weight), _f32(a.v_proj.bias)
        self.wo, self.bo = _f32(a.out_proj.weight), _f32(a.out_proj.bias)


def _ln(n):
    return _f32(n.weight), _f32(n.bias), n.eps


class _PackedDecoder:
    def __init__(self, md):
        tr = md.transformer
        self.D = md.transformer_dim
        self.layers = []
        for l in tr.layers:
            act = l.mlp.act
            if isinstance(act, torch.nn.ReLU):
                a = ACT_RELU
            elif isinstance(act, torch.nn.GELU):
                a = ACT_GELU
            else:
                raise NotImplementedError(f"MLPBlock activation {type(act)}")
            self.layers.append(dict(
                sa=_PackedAttn(l.self_attn), n1=_ln(l.norm1), t2i=_PackedAttn(l.cross_attn_token_to_image), n2=_ln(l.norm2),
                w1=_f32(l.mlp.lin1.weight), b1=_f32(l.mlp.lin1.bias), w2=_f32(l.mlp.lin2.weight), b2=_f32(l.mlp.lin2.bias),
                act=a, n3=_ln(l.norm3), n4=_ln(l.norm4), i2t=_PackedAttn(l.cross_attn_image_to_token), skip=l.skip_first_layer_pe))
        self.final = _PackedAttn(tr.final_attn_token_to_image)
        self.nf = _ln(tr.norm_final_attn)
        self.tc = DECODER_TC
        if self.tc:
            # patch-row projections as split-bf16 GEMM operands: per layer [k_proj of token->patch ; q_proj of patch->token] act
            # on (keys + pe), v_proj of token->patch on keys
            for l in self.layers:
                t2i, i2t = l["t2i"], l["i2t"]
                l["wkq"] = ops.pack_weight(torch.cat([t2i.wk, i2t.wq]))
                l["bkq"] = torch.cat([t2i.bk, i2t.bq]).contiguous()
                l["wv"] = ops.pack_weight(t2i.wv)
                l["n_k"] = t2i.wk.shape[0]
            self.wk_f, self.wv_f = ops.pack_weight(self.final.wk), ops.pack_weight(self.final.wv)
        self.iou_token, self.mask_tokens = _f32(md.iou_token.weight), _f32(md.mask_tokens.weight)
        self.nmt = md.num_mask_tokens
        self.hyper = []
        for li in range(3):
            self.hyper.append((torch.stack([_f32(m.layers[li].weight) for m in md.output_hypernetworks_mlps]).contiguous(),
                               torch.stack([_f32(m.layers[li].bias) for m in md.output_hypernetworks_mlps]).contiguous()))
        up = md.output_upscaling
        self.up0w, self.up0b = _f32(up[0].weight), _f32(up[0].bias)
        if DECODER_TC:
            self.up0w_s = ops.pack_weight(up[0].weight)
        self.up1 = _ln(up[1])
        self.up3w, self.up3b = ops.pack_weight(up[3].weight), _f32(up[3].bias)
        self.iou = [(_f32(l.weight), _f32(l.bias)) for l in md.iou_prediction_head.layers]
        self.iou_sigmoid = md.iou_prediction_head.sigmoid_output


def _attend(pa: _PackedAttn, q_in, q_pe, k_in, k_pe, v_in, Z, Lq, Lk):
    """Attention.forward (transformer.py:214-236); *_pe are optional addends fused into the projections."""
    q = ops.linear_f32(q_in, pa.wq, pa.bq, x2=q_pe)
    k = ops.linear_f32(k_in, pa.wk, pa.bk, x2=k_pe)
    v = ops.linear_f32(v_in, pa.wv, pa.bv)
    o = ops.attention_f32(q, k, v, Z, Lq, Lk, pa.H, pa.inner // pa.H)
    return ops.linear_f32(o, pa.wo, pa.bo)


def _add_ln(x, r, n):
    out = torch.empty_like(x)
    ops.layernorm(x, n[0], n[1], n[2], r=r, out_f32=out)
    return out


def run_mask_decoder(md, pc_embeddings, pc_pe, sparse, dense, aux, multimask_output: bool):
    pk = _cached(md, _PackedDecoder)
    dev = pc_embeddings.device
    D = pk.D
    Z, P, _ = sparse.shape
    B, G, _ = pc_embeddings.shape
    rep = Z // B
    T = 1 + pk.nmt + P
    mask_slice = slice(1, None) if multimask_output else slice(0, 1)
    ids = list(range(pk.nmt))[mask_slice]
    C = len(ids)

    # tokens / src (mask_decoder.py:126-139)
    sparse = sparse.float().contiguous()
    pc_embeddings = pc_embeddings.float().contiguous()
    if dense.stride(0) == 0 and dense.stride(1) == 0:  # no-mask embedding broadcast
        dense_t, dz, dg = dense[0, 0].contiguous(), 0, 0
    else:
        dense_t = dense.float().contiguous()
        dz, dg = (G * D if dense_t.shape[0] == Z else 0), D
        if dense_t.shape[0] not in (Z, 1):
            raise RuntimeError("dense prompt embeddings must have batch B*M (or 1)")
    tokens = torch.empty((Z * T, D), dtype=torch.float32, device=dev)
    src = torch.empty((Z * G, D), dtype=torch.float32, device=dev)
    nv.check(nv.lib().psam_decoder_prepare(nv.ptr(pk.iou_token), nv.ptr(pk.mask_tokens), pk.nmt, nv.ptr(sparse), P,
                                           nv.ptr(pc_embeddings), nv.ptr(dense_t), dz, dg, Z, rep, G, D,
                                           nv.ptr(tokens), nv.ptr(src), nv.stream()), "decoder_prepare")
    pe_z = ops.add_bcast(torch.zeros_like(src), pc_pe.float().contiguous(), chunk=G * D, rep=rep)  # repeat_interleave(pc_pe)

    queries, keys, qpe = tokens, src, tokens
    if pk.tc:
        return _run_decoder_tc(pk, queries, keys, qpe, pe_z, aux, Z, T, G, D, rep, ids, mask_slice, dev)
    for l in pk.layers:
        if l["skip"]:
            queries = _add_ln(_attend(l["sa"], queries, None, queries, None, queries, Z, T, T), None, l["n1"])
        else:
            queries = _add_ln(queries, _attend(l["sa"], queries, qpe, queries, qpe, queries, Z, T, T), l["n1"])
        queries = _add_ln(queries, _attend(l["t2i"], queries, qpe, keys, pe_z, keys, Z, T, G), l["n2"])
        h = ops.linear_f32(queries, l["w1"], l["b1"], act=l["act"])
        queries = _add_ln(queries, ops.linear_f32(h, l["w2"], l["b2"]), l["n3"])
        keys = _add_ln(keys, _attend(l["i2t"], keys, pe_z, queries, qpe, queries, Z, G, T), l["n4"])
    queries = _add_ln(queries, _attend(pk.final, queries, qpe, keys, pe_z, keys, Z, T, G), pk.nf)
    f0 = ops.linear_f32(keys, pk.up0w, pk.up0b)  # [Z*G, D]
    return _decoder_heads(pk, queries, f0, aux, Z, T, G, D, rep, ids, mask_slice, dev)


def _run_decoder_tc(pk, queries, keys, qpe, pe_z, aux, Z, T, G, D, rep, ids, mask_slice, dev):
    """Two-way transformer (transformer.py:55-180) with the patch-row projections on tensor cores.  keys_s / keyspe_s are the
    split-bf16 copies of keys and keys + pe; the LayerNorm that updates keys refreshes both."""
    ZG = Z * G
    keys_s, keyspe_s = Split(ZG, D, dev), Split(ZG, D, dev)
    ops.split_f32(keys, keys_s)
    ops.split_f32(keys, keyspe_s, add=pe_z)
    for l in pk.layers:
        sa, t2i, i2t = l["sa"], l["t2i"], l["i2t"]
        if l["skip"]:
            queries = _add_ln(_attend(sa, queries, None, queries, None, queries, Z, T, T), None, l["n1"])
        else:
            queries = _add_ln(queries, _attend(sa, queries, qpe, queries, qpe, queries, Z, T, T), l["n1"])
        nk = l["n_k"]
        kq = torch.empty((ZG, l["bkq"].shape[0]), dtype=torch.float32, device=dev)  # [:, :nk] = k of t2i, [:, nk:] = q of i2t
        ops.gemm(keyspe_s, l["wkq"], bias=l["bkq"], out_f32=kq, passes=PASSES)
        vv = torch.empty((ZG, t2i.wv.shape[0]), dtype=torch.float32, device=dev)
        ops.gemm(keys_s, l["wv"], bias=t2i.bv, out_f32=vv, passes=PASSES)
        # tokens -> patches
        q = ops.linear_f32(queries, t2i.wq, t2i.bq, x2=qpe)
        o = ops.attention_f32(q, kq, vv, Z, T, G, t2i.H, t2i.inner // t2i.H)
        queries = _add_ln(queries, ops.linear_f32(o, t2i.wo, t2i.bo), l["n2"])
        h = ops.linear_f32(queries, l["w1"], l["b1"], act=l["act"])
        queries = _add_ln(queries, ops.linear_f32(h, l["w2"], l["b2"]), l["n3"])
        # patches -> tokens
        k2 = ops.linear_f32(queries, i2t.wk, i2t.bk, x2=qpe)
        v2 = ops.linear_f32(queries, i2t.wv, i2t.bv)
        o2 = ops.attention_f32(kq, k2, v2, Z, G, T, i2t.H, i2t.inner // i2t.H, q_off=nk)
        upd = ops.linear_f32(o2, i2t.wo, i2t.bo)
        new_keys = torch.empty_like(keys)
        n4 = l["n4"]
        ops.layernorm(keys, n4[0], n4[1], n4[2], r=upd, out_f32=new_keys, out_split=keys_s, post_add=pe_z, out_split2=keyspe_s)
        keys = new_keys
    kf = torch.empty((ZG, pk.final.wk.shape[0]), dtype=torch.float32, device=dev)
    ops.gemm(keyspe_s, pk.wk_f, bias=pk.final.bk, out_f32=kf, passes=PASSES)
    vf = torch.empty((ZG, pk.final.wv.shape[0]), dtype=torch.float32, device=dev)
    ops.gemm(keys_s, pk.wv_f, bias=pk.final.bv, out_f32=vf, passes=PASSES)
    q = ops.linear_f32(queries, pk.final.wq, pk.final.bq, x2=qpe)
    o = ops.attention_f32(q, kf, vf, Z, T, G, pk.final.H, pk.final.inner // pk.final.H)
    queries = _add_ln(queries, ops.linear_f32(o, pk.final.wo, pk.final.bo), pk.nf)
    f0 = torch.empty((ZG, D), dtype=torch.float32, device=dev)
    ops.gemm(keys_s, pk.up0w_s, bias=pk.up0b, out_f32=f0, passes=PASSES)
    return _decoder_heads(pk, queries, f0, aux, Z, T, G, D, rep, ids, mask_slice, dev)


def _decoder_heads(pk, queries, f0, aux, Z, T, G, D, rep, ids, mask_slice, dev):
    """mask_decoder.py:146-184: upsampling, hyper-network product, IoU head.  f0 = output_upscaling[0](keys) [Z*G, D]."""
    hs = queries  # [Z*T, D]
    C = len(ids)
    # upscaling (mask_decoder.py:146-164): Linear0 commutes with the (affine, weights sum to 1) interpolation
    if aux.interp_index is None or aux.interp_weight is None:
        aux.interp_index, aux.interp_weight = ops.knn3_interp(aux.coords.float().contiguous(), aux.centers)
    N = aux.coords.shape[1]
    u1 = Split(Z * N, D, dev)
    nv.check(nv.lib().psam_interp_ln_gelu(nv.ptr(f0), Z, rep, G, D, nv.ptr(aux.interp_index), nv.ptr(aux.interp_weight), N,
                                          nv.ptr(pk.up1[0]), nv.ptr(pk.up1[1]), pk.up1[2], u1.ptr(), u1.plane, u1.pitch,
                                          nv.stream()), "interp_ln_gelu")
    # hyper-network MLPs on the selected mask tokens (mask_decoder.py:167-175), batched over tokens
    i0 = ids[0]
    x = hs
    ld = T * D
    xoff = (1 + i0) * D
    hyper = None
    for li, (w, b) in enumerate(pk.hyper):
        y = torch.empty((Z, C, D), dtype=torch.float32, device=dev)
        ops.linear_f32(x, w[i0:i0 + C], b[i0:i0 + C], act=ACT_RELU if li < 2 else ACT_NONE, out=y, M=Z, K=D, ldx=ld, Z=C,
                       x_z=D, w_z=D * D, b_z=D, y_z=D, ldy=C * D, x_off=xoff)
        x, ld, xoff, hyper = y, C * D, 0, y
    if FUSED_MASK_DOT and N % 32 == 0 and C <= 8:
        # output_upscaling[3..4] (Linear + GELU) and the hyper-network product fused into one GEMM epilogue
        masks = torch.zeros((Z, C, N), dtype=torch.float32, device=dev)
        ops.gemm(u1, pk.up3w, bias=pk.up3b, act=ACT_GELU, passes=PASSES, rowdot=(hyper, masks))
    else:
        u2 = torch.empty((Z * N, D), dtype=torch.float32, device=dev)
        ops.gemm(u1, pk.up3w, bias=pk.up3b, out_f32=u2, act=ACT_GELU, passes=PASSES)
        masks = torch.empty((Z, C, N), dtype=torch.float32, device=dev)
        nv.check(nv.lib().psam_mask_dot(nv.ptr(u2), D, nv.ptr(hyper), Z, C, N, D, nv.ptr(masks), nv.stream()), "mask_dot")

    # IoU head on the iou token (mask_decoder.py:180-182)
    y = hs
    ld = T * D
    for li, (w, b) in enumerate(pk.iou):
        y = ops.linear_f32(y, w, b, act=ACT_RELU if li < len(pk.iou) - 1 else ACT_NONE, M=Z, K=w.shape[1], ldx=ld)
        ld = y.shape[-1]
    if pk.iou_sigmoid:
        y = torch.sigmoid(y)
    return masks, y[:, mask_slice].contiguous()


# ------------------------------------------------------------------------------------------------
# automatic mask generation (SAM's SamAutomaticMaskGenerator restated for point clouds: DESIGN.md)
# ------------------------------------------------------------------------------------------------
AMG_MAX_CANDIDATES = 16384  # psam_mask_nms sorts the candidates in one CTA's shared memory


def run_amg_prompts(cloud, P: int) -> torch.Tensor:
    """The P prompt points [1, P, 3] = the points ops.fps(coords, P) selects.  FPS is prefix-stable, so for P <= G they are
    the first P centres the encoder's grouper already selected."""
    patches = cloud["patches"]
    if "fps_idx" in patches and P <= patches["centers"].shape[1]:
        return patches["centers"][:, :P]
    return ops.fps(cloud["coords"], P)[1]


def run_automatic_masks(model, cloud, prompts: torch.Tensor, params) -> dict:
    """Segment everything: every prompt point [1, P, 3] is decoded with multimask output (candidate 3 p + m), each chunk of
    `points_per_batch` prompts is reduced to bit-packed masks + area / stability / filter flag right after its decode (its
    fp32 logits do not outlive the chunk), then one NMS over all candidates and ONE host read (kept count and the prompt
    range flag).  cloud: the dict PointCloudSAM._encode returns (the set_pointcloud cache).  params: a mapping with
    points_per_batch, pred_iou_thresh, stability_score_thresh, stability_score_offset, mask_threshold, nms_thresh."""
    coords, patches = cloud["coords"], cloud["patches"]
    dev = coords.device
    N, P = coords.shape[1], prompts.shape[1]
    K = 3 * P
    W = ops.mask_words(N)
    table = (torch.empty((K, W), dtype=torch.int32, device=dev), torch.empty(K, dtype=torch.int32, device=dev),
             torch.empty(K, dtype=torch.float32, device=dev), torch.empty(K, dtype=torch.uint8, device=dev))
    scores = torch.empty(K, dtype=torch.float32, device=dev)
    dense = run_mask_encoder(model.mask_encoder, None, coords, patches["centers"], patches["knn_idx"])
    step = int(params["points_per_batch"])
    for s in range(0, P, step):
        pts = prompts[0, s:s + step].unsqueeze(1)  # [Z, 1, 3]: one positive point per prompt
        Z = pts.shape[0]
        sparse = run_point_encoder(model.point_encoder, pts, torch.ones((Z, 1), dtype=torch.int32, device=dev), check=False)
        masks, iou = run_mask_decoder(model.mask_decoder, cloud["pc_embeddings"], cloud["pc_pe"], sparse, dense, cloud["aux"], True)
        iou = iou.reshape(-1)
        ops.mask_stats(masks, iou, params["mask_threshold"], params["stability_score_offset"], params["pred_iou_thresh"],
                       params["stability_score_thresh"], out=table, row0=3 * s)
        scores[3 * s:3 * (s + Z)].copy_(iou)
    bits, area, stability, keep = table
    keep_idx, count = ops.mask_nms(bits, area, scores, keep, params["nms_thresh"])
    flag = bad_flag(dev)
    n, bad = torch.cat([count, flag]).tolist()
    if bad:
        flag.zero_()
        raise ValueError("Input coordinates must be normalized to [-1, 1].")
    rows = keep_idx[:n]
    idx = rows.long()
    prompt_index = idx // 3
    return dict(masks=ops.mask_unpack(bits, N, rows), iou_preds=scores[idx], stability_scores=stability[idx],
                areas=area[idx].long(), prompt_coords=prompts[0, prompt_index], prompt_index=prompt_index, mask_index=idx % 3)
