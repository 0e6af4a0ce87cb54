"""GPU parity tests, kernel by kernel, through the C ABI (ctypes) against the oracle / plain torch fp32."""
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import synth, tokenizer_ref, torch_ref  # noqa: E402
from oracle.make_golden import REF_FPS_CASES, REF_FPS_STREAMING_CASES, REF_FPS_STREAMING_SEED, REF_NN  # noqa: E402


def _ops():
    from psam_b200 import ops

    return ops


def _dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------
# FPS
# ------------------------------------------------------------------------------------------------
def test_fps_golden_fixtures(golden_dir):
    ops = _ops()
    g = np.load(os.path.join(golden_dir, "fps_cases.npz"))
    for i in range(int(g["n"])):
        B, N, G, seed = [int(v) for v in g[f"case{i}"]]
        xyz, _ = synth.make_batch(B, N, seed, str(g[f"kind{i}"]))
        idx, centers = ops.fps(xyz.to(_dev()), G)
        want = torch.from_numpy(g[f"idx{i}"].astype(np.int64))
        got = idx.cpu()
        nbad = int((got != want).sum())
        assert nbad == 0, f"case {i} {(B, N, G)}: {nbad} mismatches, first at {(got != want).nonzero()[:3].tolist()}"
        ref_c = torch.gather(xyz, 1, want[..., None].expand(-1, -1, 3))
        assert torch.equal(centers.cpu(), ref_c)


@pytest.mark.parametrize("B,N,G,kind", [(1, 32768, 512, "ball"), (3, 5000, 256, "grid"), (2, 70000, 64, "ball"),
                                        (1, 131072, 96, "kitti"), (2, 100, 100, "ball"), (1, 33, 7, "grid")])
def test_fps_vs_oracle(B, N, G, kind):
    ops = _ops()
    xyz, _ = synth.make_batch(B, N, 7, kind)
    idx, _ = ops.fps(xyz.to(_dev()), G)
    want = tokenizer_ref.fps(xyz.numpy(), G)
    assert (idx.cpu().numpy() == want).all()


def test_fps_degenerate_and_errors():
    ops = _ops()
    same = torch.ones(1, 40, 3, device=_dev())
    idx, _ = ops.fps(same, 5)
    assert (idx == 0).all()
    with pytest.raises(RuntimeError):
        ops.fps(torch.zeros(1, 4, 3, device=_dev()), 5)
    from pc_sam.model.common import sample_farthest_points

    with pytest.raises(RuntimeError):
        sample_farthest_points(torch.zeros(1, 4, 3), 2)  # CPU tensor: no fallback


def test_fps_against_reference_cuda_kernel(golden_dir):
    """Against the outputs of the reference's own kernel compiled for sm_100a (tests/golden/ref_kernels.npz, written by
    oracle/make_golden.py --ref-kernels)."""
    ops = _ops()
    z = np.load(os.path.join(golden_dir, "ref_kernels.npz"))
    for i, (B, N, G, kind, seed) in enumerate(REF_FPS_CASES):
        xyz, _ = synth.make_batch(B, N, seed, kind)
        want = torch.from_numpy(z[f"fps{i}"])
        got, _ = ops.fps(xyz.to(_dev()), G)
        assert torch.equal(got.cpu(), want), (B, N, G, kind)
        assert (tokenizer_ref.fps(xyz.numpy(), G) == want.numpy()).all(), "oracle vs reference kernel"


@pytest.mark.parametrize("N,G,kind", REF_FPS_STREAMING_CASES)
def test_fps_streaming_plan_beyond_cluster_registers(N, G, kind, golden_dir):
    """N > 131072 no longer fits the 16-CTA register plan: the multi-cluster / streaming plan must reproduce the reference
    kernel (sample_farthest_points_kernel.cu:8-104: fmaf chain + bit-reversed tie-break) bit for bit, against the C
    oracle and against the outputs of the reference's own kernel compiled for sm_100a (tests/golden/ref_kernels.npz)."""
    ops = _ops()
    xyz, _ = synth.make_batch(1, N, REF_FPS_STREAMING_SEED, kind)
    x = xyz.to(_dev())
    got, centers = ops.fps(x, G)
    want = tokenizer_ref.fps(xyz.numpy(), G)
    assert np.array_equal(got.cpu().numpy(), want), f"first mismatch at {np.nonzero(got.cpu().numpy() != want)[1][:3]}"
    assert torch.equal(centers.cpu(), torch.gather(xyz, 1, torch.from_numpy(want)[..., None].expand(-1, -1, 3)))
    ref = np.load(os.path.join(golden_dir, "ref_kernels.npz"))[f"fps_streaming_{N}_{G}_{kind}"]
    assert np.array_equal(ref, got.cpu().numpy())


# ------------------------------------------------------------------------------------------------
# kNN / grouping / interpolation
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,Q,K,kind", [(2, 4096, 128, 32, "ball"), (1, 32768, 512, 64, "ball"), (1, 777, 24, 8, "ball"),
                                          (1, 2048, 64, 32, "grid"), (1, 20000, 64, 256, "kitti"), (2, 300, 40, 3, "ball"),
                                          (1, 64, 64, 64, "ball"), (1, 5000, 16, 1, "ball")])
def test_knn_vs_oracle(B, N, Q, K, kind):
    ops = _ops()
    xyz, _ = synth.make_batch(B, N, 11, kind)
    centers = xyz[:, torch.randperm(N, generator=torch.Generator().manual_seed(0))[:Q]].contiguous()
    idx, d2 = ops.knn(centers.to(_dev()), xyz.to(_dev()), K, want_d2=True)
    widx, wd2 = tokenizer_ref.knn(centers.numpy(), xyz.numpy(), K)
    # distances are a multiset property (independent of tie resolution): must agree bit for bit
    assert np.array_equal(d2.cpu().numpy(), wd2), f"max diff {np.abs(d2.cpu().numpy() - wd2).max()}"
    # both sides resolve ties towards the lower index and sort by (d2, index): indices agree exactly
    assert np.array_equal(idx.cpu().numpy(), widx)
    # and the reference semantics (cdist + topk) select the same sets where no tie exists
    if kind != "grid":
        _, ref = torch_ref.knn_points(centers, xyz, K, sorted=True)
        assert np.array_equal(np.sort(ref.numpy(), -1), np.sort(widx, -1))


def test_group_gather_and_interp():
    ops = _ops()
    xyz, feats = synth.make_batch(2, 3000, 3)
    g = torch_ref.KNNGrouper(64, 16)
    want = g(xyz, feats)
    d = _dev()
    idx, centers = ops.fps(xyz.to(d), 64)
    knn, _ = ops.knn(centers, xyz.to(d), 16)
    groups = ops.group_gather(xyz.to(d), feats.to(d), centers, knn)
    # same neighbour sets -> compare after sorting rows of each group by neighbour index
    o1 = torch.argsort(knn.cpu(), -1)
    o2 = torch.argsort(want["knn_idx"], -1)
    a = torch.gather(groups.cpu(), 2, o1[..., None].expand(-1, -1, -1, 6))
    b = torch.gather(want["features"], 2, o2[..., None].expand(-1, -1, -1, 6))
    assert torch.equal(torch.sort(knn.cpu(), -1).values, torch.sort(want["knn_idx"], -1).values)
    torch.testing.assert_close(a, b, atol=0, rtol=0)
    # mask-encoder form: M=2 masks per cloud, 1 channel, radius
    m = torch.randn(4, 3000, 1)
    want2 = torch_ref.group_with_centers_and_knn(xyz, m, want["centers"], knn.cpu(), radius=0.5)
    got2 = ops.group_gather(xyz.to(d), m.to(d), centers, knn, 0.5)
    torch.testing.assert_close(got2.cpu(), want2, atol=1e-7, rtol=1e-6)
    # 3-NN interpolation weights
    ii, ww = ops.knn3_interp(xyz.to(d), centers)
    wi, wwt = torch_ref.compute_interp_weights(xyz, want["centers"])
    assert torch.equal(torch.sort(ii.cpu(), -1).values, torch.sort(wi, -1).values)
    torch.testing.assert_close(torch.sort(ww.cpu(), -1).values, torch.sort(wwt, -1).values, atol=2e-6, rtol=1e-5)


def test_nn_distance_vs_reference_and_bruteforce(golden_dir):
    ops = _ops()
    xyz, _ = synth.make_batch(1, REF_NN["N"], REF_NN["seed"])
    a, b = xyz[0, :REF_NN["split"]].to(_dev()), xyz[0, REF_NN["split"]:].to(_dev())
    got = ops.nn_distance(a, b)
    want = (torch.cdist(a.cpu().double(), b.cpu().double()) ** 2).min(dim=1).values.float()
    torch.testing.assert_close(got.cpu(), want, atol=1e-7, rtol=1e-5)
    # the reference's chamfer kernel compiled for sm_100a (tests/golden/ref_kernels.npz)
    d1 = torch.from_numpy(np.load(os.path.join(golden_dir, "ref_kernels.npz"))["nn_dist"])
    torch.testing.assert_close(got.cpu(), d1, atol=1e-7, rtol=1e-6)


# ------------------------------------------------------------------------------------------------
# tcgen05 GEMM
# ------------------------------------------------------------------------------------------------
def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(_dev())


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (128, 128, 256), (512, 1024, 1024), (300, 200, 2730), (4096, 128, 128),
                                   (256, 64, 64), (77, 344, 128), (512, 5504, 1024), (1, 256, 512)])
def test_gemm_tc_plain(M, N, K):
    ops = _ops()
    a, w, b = _rand(M, K, seed=1), _rand(N, K, seed=2, scale=K ** -0.5), _rand(N, seed=3)
    A, W = ops.pack_weight(a), ops.pack_weight(w)
    # the packed operands reproduce fp32 to 2^-17
    assert float((A.float() - a).abs().max() / a.abs().max()) < 2 ** -16
    out = torch.empty(M, N, device=_dev())
    ops.gemm(A, W, bias=b, out_f32=out)
    want = (a.double() @ w.double().t() + b.double()).float()
    err = float((out - want).abs().max())
    scale = float(want.abs().max())
    assert err < 3e-5 * max(scale, 1.0), f"err {err} scale {scale}"
    # single-pass bf16 mode exists and is (much) less accurate
    out1 = torch.empty(M, N, device=_dev())
    ops.gemm(A, W, bias=b, out_f32=out1, passes=1)
    err1 = float((out1 - want).abs().max())
    assert err1 < 3e-2 * max(scale, 1.0)


def test_gemm_tc_epilogues_and_splitk():
    ops = _ops()
    M, N, K = 512, 1024, 2730
    a, w, b = _rand(M, K, seed=4), _rand(N, K, seed=5, scale=K ** -0.5), _rand(N, seed=6)
    A, W = ops.pack_weight(a), ops.pack_weight(w)
    base = (a.double() @ w.double().t() + b.double())
    r = _rand(M, N, seed=7)
    # residual in place
    x = r.clone()
    ops.gemm(A, W, bias=b, out_f32=x, resid=x)
    assert float((x - (base + r.double()).float()).abs().max()) < 1e-4
    # split-K accumulate (red.add) into the residual stream
    for sk in (2, 4, 7):
        x = r.clone()
        ops.gemm(A, W, bias=b, out_f32=x, accumulate=True, split_k=sk)
        assert float((x - (base + r.double()).float()).abs().max()) < 1e-4, sk
    # GELU + split output + fp32 output together
    o32 = torch.empty(M, N, device=_dev())
    osp = ops.Split(M, N, _dev())
    ops.gemm(A, W, bias=b, out_f32=o32, out_split=osp, act=ops.ACT_GELU)
    want = torch.nn.functional.gelu(base.float())
    assert float((o32 - want).abs().max()) < 1e-4
    assert float((osp.float() - o32).abs().max()) < 2e-5 * float(want.abs().max())
    # alpha
    o = torch.empty(M, N, device=_dev())
    ops.gemm(A, W, out_f32=o, alpha=0.125)
    assert float((o - (0.125 * (base - b.double())).float()).abs().max()) < 1e-4


def test_gemm_tc_fused_group_max_and_row_dot():
    """Epilogue fusions of the tokenizer / decoder: max over the rows of a group (common.py:497 torch.max(x, dim=-2))
    and the hyper-network product masks = hyper @ gelu(linear(u))^T (mask_decoder.py:176)."""
    ops = _ops()
    # --- group max, with and without the split copy of the un-pooled rows ---
    for (G, Kg, N, K) in [(24, 64, 128, 128), (7, 32, 512, 256), (5, 96, 200, 64)]:
        M = G * Kg
        a, w, b = _rand(M, K, seed=11), _rand(N, K, seed=12, scale=K ** -0.5), _rand(N, seed=13)
        A, W = ops.pack_weight(a), ops.pack_weight(w)
        full = (a.double() @ w.double().t() + b.double()).float()
        want = full.view(G, Kg, N).max(dim=1).values
        y = torch.full((G, N), float("-inf"), device=_dev())
        ops.gemm(A, W, bias=b, gmax=y, group_rows=Kg)
        assert float((y - want).abs().max()) < 1e-4
        y2 = torch.full((G, N), float("-inf"), device=_dev())
        xs = ops.Split(M, N, _dev())
        ops.gemm(A, W, bias=b, out_split=xs, gmax=y2, group_rows=Kg)
        assert torch.equal(y, y2)
        assert float((xs.float() - full).abs().max()) < 1e-4
    # --- row dot: Z batches of rd_rows rows, C hyper vectors each ---
    for (Z, R, C, N, K) in [(2, 4096, 4, 256, 256), (3, 160, 1, 256, 256), (1, 2048, 3, 96, 128)]:
        M = Z * R
        a, w, b = _rand(M, K, seed=21), _rand(N, K, seed=22, scale=K ** -0.5), _rand(N, seed=23)
        hyper = _rand(Z, C, N, seed=24)
        A, W = ops.pack_weight(a), ops.pack_weight(w)
        u = torch.nn.functional.gelu((a.double() @ w.double().t() + b.double())).view(Z, R, N)
        want = (hyper.double() @ u.transpose(1, 2)).float()
        masks = torch.zeros(Z, C, R, device=_dev())
        ops.gemm(A, W, bias=b, act=ops.ACT_GELU, rowdot=(hyper, masks))
        assert float((masks - want).abs().max()) < 2e-4 * max(1.0, float(want.abs().max()))
    # invalid combinations are refused, not silently mis-computed
    with pytest.raises(RuntimeError):
        ops.gemm(A, W, bias=b, rowdot=(hyper, torch.zeros(Z, C, R + 1, device=_dev())))  # rows not a multiple of 32


def test_gemm_tc_swiglu_stats_and_folded_layernorm():
    """fc2(LayerNorm(silu(g) * x)) with the normalisation folded into the two GEMM epilogues (timm SwiGLU with scale_mlp,
    as in EVA02) against the unfused fp64 computation."""
    ops = _ops()
    M, D, Hd = 300, 256, 683
    Hp = (Hd + 63) // 64 * 64
    xin = _rand(M, D, seed=31)
    wg, wx = _rand(Hd, D, seed=32, scale=D ** -0.5), _rand(Hd, D, seed=33, scale=D ** -0.5)
    bg, bx = _rand(Hd, seed=34, scale=0.1), _rand(Hd, seed=35, scale=0.1)
    gamma, beta = 1.0 + 0.2 * _rand(Hd, seed=36), 0.1 * _rand(Hd, seed=37)
    w2, b2 = _rand(D, Hd, seed=38, scale=Hd ** -0.5), _rand(D, seed=39, scale=0.1)
    resid = _rand(M, D, seed=40)
    eps = 1e-6
    h = torch.nn.functional.silu(xin.double() @ wg.double().t() + bg.double()) * (xin.double() @ wx.double().t() + bx.double())
    want = resid.double() + torch.nn.functional.layer_norm(h, (Hd,), gamma.double(), beta.double(), eps) @ w2.double().t() + b2.double()
    # pack as the engine does
    w1 = torch.zeros(2 * Hp, D, device=_dev())
    b1 = torch.zeros(2 * Hp, device=_dev())
    w1[0:2 * Hd:2], w1[1:2 * Hd:2] = wg, wx
    b1[0:2 * Hd:2], b1[1:2 * Hd:2] = bg, bx
    gpad, bpad = torch.zeros(Hp, device=_dev()), torch.zeros(Hp, device=_dev())
    gpad[:Hd], bpad[:Hd] = gamma, beta
    w2p = torch.zeros(D, Hp, device=_dev())
    w2p[:, :Hd] = w2
    W1, W2g = ops.pack_weight(w1), ops.pack_weight((w2p.double() * gpad.double()[None]).float())
    c2 = (w2p.double() @ gpad.double()).float().contiguous()
    d2 = (w2p.double() @ bpad.double() + b2.double()).float().contiguous()
    X = ops.pack_weight(xin)
    for sk in (1, 3):
        stats = torch.zeros(M, 2, device=_dev())
        hs = ops.Split(M, Hp, _dev(), pitch=Hp)
        ops.gemm(X, W1, bias=b1, out_split=hs, swiglu=True, stats_out=stats)
        assert float((hs.float()[:, :Hd] - h.float()).abs().max()) < 1e-4
        assert float(hs.float()[:, Hd:].abs().max()) == 0.0
        torch.testing.assert_close(stats[:, 0], h.sum(-1).float(), atol=2e-3, rtol=1e-5)
        torch.testing.assert_close(stats[:, 1], (h * h).sum(-1).float(), atol=2e-3, rtol=1e-5)
        out = resid.clone()
        if sk > 1:
            ops.gemm(hs, W2g, bias=d2, out_f32=out, accumulate=True, split_k=sk, ln_fold=(stats, c2, Hd, eps))
        else:
            ops.gemm(hs, W2g, bias=d2, out_f32=out, resid=out, ln_fold=(stats, c2, Hd, eps))
        err = float((out - want.float()).abs().max())
        assert err < 1e-4 * max(1.0, float(want.abs().max())), (sk, err)


def test_gemm_tc_layernorm_free_block_chain():
    """The LayerNorm-free transformer block: a producer GEMM writes x (fp32 + split-bf16) and its row statistics; the
    consumers apply norm1 / norm2 inside their epilogues with split-bf16, SwiGLU(+statistics) and GELU outputs.  Against
    the unfused fp64 computation, with a row mean that is large against the spread (cancellation stress)."""
    ops = _ops()
    M, D, N1, Hd = 300, 256, 384, 344
    Hp = (Hd + 63) // 64 * 64
    eps = 1e-6
    a0, w0, b0 = _rand(M, 128, seed=51), _rand(D, 128, seed=52, scale=128 ** -0.5), _rand(D, seed=53) + 3.0  # mean >> spread
    r0 = _rand(M, D, seed=54)
    g1, be1 = 1.0 + 0.2 * _rand(D, seed=55), 0.1 * _rand(D, seed=56)
    x_want = r0.double() + a0.double() @ w0.double().t() + b0.double()
    xn = torch.nn.functional.layer_norm(x_want, (D,), g1.double(), be1.double(), eps)

    def fold(w, b):
        wg = w.double() * g1.double()[None]
        return ops.pack_weight(wg.float()), wg.sum(1).float().contiguous(), (w.double() @ be1.double() + b.double()).float().contiguous()

    # producer: x = r0 + a0 @ w0^T + b0 -> fp32, split-bf16 and (sum, sum sq) per row
    x = r0.clone()
    xs = ops.Split(M, D, _dev())
    st = torch.zeros(M, 2, device=_dev())
    ops.gemm(ops.pack_weight(a0), ops.pack_weight(w0), bias=b0, out_f32=x, resid=x, out_split=xs, stats_out=st)
    assert float((x - x_want.float()).abs().max()) < 5e-5 * float(x_want.abs().max())
    assert float((xs.float() - x).abs().max()) < 3e-5 * float(x_want.abs().max())
    torch.testing.assert_close(st[:, 0], x_want.sum(-1).float(), atol=2e-3, rtol=1e-5)
    torch.testing.assert_close(st[:, 1], (x_want * x_want).sum(-1).float(), atol=2e-3, rtol=2e-5)
    tol = lambda want: 2e-4 * max(1.0, float(want.abs().max()))
    # consumer 1 (qkv form): split-bf16 output
    w1, b1 = _rand(N1, D, seed=57, scale=D ** -0.5), _rand(N1, seed=58, scale=0.1)
    W1f, c1, d1 = fold(w1, b1)
    y = ops.Split(M, N1, _dev())
    ops.gemm(xs, W1f, bias=d1, out_split=y, ln_fold=(st, c1, D, eps))
    want = xn @ w1.double().t() + b1.double()
    assert float((y.float() - want.float()).abs().max()) < tol(want)
    # consumer 2 (EVA02 fc1 form): SwiGLU pairs + statistics of the products
    wg_, wx_ = _rand(Hd, D, seed=59, scale=D ** -0.5), _rand(Hd, D, seed=60, scale=D ** -0.5)
    bg_, bx_ = _rand(Hd, seed=61, scale=0.1), _rand(Hd, seed=62, scale=0.1)
    wi, bi = torch.zeros(2 * Hp, D, device=_dev()), torch.zeros(2 * Hp, device=_dev())
    wi[0:2 * Hd:2], wi[1:2 * Hd:2], bi[0:2 * Hd:2], bi[1:2 * Hd:2] = wg_, wx_, bg_, bx_
    Wif, ci, di = fold(wi, bi)
    hs = ops.Split(M, Hp, _dev(), pitch=Hp)
    hst = torch.zeros(M, 2, device=_dev())
    ops.gemm(xs, Wif, bias=di, out_split=hs, swiglu=True, stats_out=hst, ln_fold=(st, ci, D, eps))
    h = torch.nn.functional.silu(xn @ wg_.double().t() + bg_.double()) * (xn @ wx_.double().t() + bx_.double())
    assert float((hs.float()[:, :Hd] - h.float()).abs().max()) < tol(h)
    assert float(hs.float()[:, Hd:].abs().max()) == 0.0
    torch.testing.assert_close(hst[:, 0], h.sum(-1).float(), atol=5e-3, rtol=1e-4)
    # consumer 3 (EVA-giant fc1 form): GELU + split-bf16 output; consumer 4 (out_proj form): fp32 output
    y3 = ops.Split(M, N1, _dev())
    ops.gemm(xs, W1f, bias=d1, out_split=y3, act=ops.ACT_GELU, ln_fold=(st, c1, D, eps))
    want3 = torch.nn.functional.gelu(want)
    assert float((y3.float() - want3.float()).abs().max()) < tol(want3)
    y4 = torch.empty(M, N1, device=_dev())
    ops.gemm(xs, W1f, bias=d1, out_f32=y4, ln_fold=(st, c1, D, eps))
    assert float((y4 - want.float()).abs().max()) < tol(want)
    # statistics of the output are refused where an element has more than one writer
    with pytest.raises(RuntimeError):
        ops.gemm(xs, W1f, bias=d1, out_f32=torch.zeros(M, N1, device=_dev()), accumulate=True, split_k=2, stats_out=st)


def test_gemm_tc_batched_attention_shapes():
    """The batched operand views used by the ViT attention (heads = b1, clouds = b2)."""
    from psam_b200 import native as nv

    ops = _ops()
    B, H, L, dh = 2, 3, 200, 88
    D = H * dh
    qkv = _rand(B * L, 3 * D, seed=8)
    QKV = ops.Split(B * L, 3 * D, _dev())
    ops.split_f32(qkv, QKV)
    s = torch.empty(B * H * L, L, device=_dev())
    qa = QKV.operand(rows=L, k=dh, col=0, nb1=H, b1_stride=dh, nb2=B, b2_stride=L * QKV.pitch)
    ka = QKV.operand(rows=L, k=dh, col=D, nb1=H, b1_stride=dh, nb2=B, b2_stride=L * QKV.pitch)
    o = ops.GemmOut()
    o.out_f32, o.ldo, o.out_b1, o.out_b2, o.alpha = nv.ptr(s), L, L * L, H * L * L, 1.0
    ops.gemm_raw(qa, ka, o, 3, 1)
    q = qkv[:, :D].reshape(B, L, H, dh).permute(0, 2, 1, 3).double()
    k = qkv[:, D:2 * D].reshape(B, L, H, dh).permute(0, 2, 1, 3).double()
    want = (q @ k.transpose(-1, -2)).float().reshape(B * H * L, L)
    assert float((s - want).abs().max()) < 3e-4, float((s - want).abs().max())


# ------------------------------------------------------------------------------------------------
# glue kernels
# ------------------------------------------------------------------------------------------------
def test_layernorm_variants():
    ops = _ops()
    x, r = _rand(1000, 2730, seed=1), _rand(1000, 2730, seed=2)
    g, b = _rand(2730, seed=3), _rand(2730, seed=4)
    out = torch.empty_like(x)
    sp = ops.Split(1000, 2730, _dev(), pitch=2752)
    ops.layernorm(x, g, b, 1e-6, r=r, out_f32=out, out_split=sp)
    want = torch.nn.functional.layer_norm(x + r, (2730,), g, b, 1e-6)
    torch.testing.assert_close(out, want, atol=2e-5, rtol=1e-5)
    assert float((sp.float() - want).abs().max()) < 1e-4
    assert float(sp.t[:, :, 2730:].float().abs().max()) == 0.0
    # group bias + GELU (PatchEncoder conv2[1..2])
    t = _rand(10, 2730, seed=5)
    ops.layernorm(x, g, b, 1e-5, gbias=t, group_rows=100, act=ops.ACT_GELU, out_f32=out)
    want = torch.nn.functional.gelu(torch.nn.functional.layer_norm(x + t.repeat_interleave(100, 0), (2730,), g, b, 1e-5))
    torch.testing.assert_close(out, want, atol=2e-5, rtol=1e-5)
    # the ViT token stream (512 x 1024 / 768) under both launch policies: CTA per row (latency) / warp per row (SM-time)
    for D in (1024, 768, 256):
        x1, r1, g1, b1 = _rand(512, D, seed=6), _rand(512, D, seed=7), _rand(D, seed=8), _rand(D, seed=9)
        want = torch.nn.functional.layer_norm(x1 + r1, (D,), g1, b1, 1e-6)
        for policy in (0, 1):
            prev, ops.GEMM_TILE_HINT = ops.GEMM_TILE_HINT, policy
            try:
                o1, s1 = torch.empty_like(x1), ops.Split(512, D, _dev())
                ops.layernorm(x1, g1, b1, 1e-6, r=r1, out_f32=o1, out_split=s1)
            finally:
                ops.GEMM_TILE_HINT = prev
            torch.testing.assert_close(o1, want, atol=2e-5, rtol=1e-5)
            assert float((s1.float() - want).abs().max()) < 1e-4


def test_swiglu_small_in_groupmax_softmax_transpose():
    ops = _ops()
    d = _dev()
    H, Hp, M = 344, 384, 77
    gx = _rand(M, 2 * Hp, seed=1)
    g, b = _rand(H, seed=2), _rand(H, seed=3)
    out = ops.Split(M, H, d, pitch=Hp)
    ops.swiglu_ln(gx, H, Hp, g, b, 1e-6, out)
    want = torch.nn.functional.layer_norm(torch.nn.functional.silu(gx[:, :H]) * gx[:, Hp:Hp + H], (H,), g, b, 1e-6)
    assert float((out.float() - want).abs().max()) < 2e-5 * float(want.abs().max()) + 1e-6
    assert float(out.t[:, :, H:].float().abs().max()) == 0.0
    # small-input linear (+LN+GELU)
    x = _rand(500, 6, seed=4)
    W, bb, gg, be = _rand(128, 6, seed=5), _rand(128, seed=6), _rand(128, seed=7), _rand(128, seed=8)
    o = ops.Split(500, 128, d)
    ops.small_in_linear(x, W, bb, gg, be, 1e-5, True, ops.ACT_GELU, o)
    want = torch.nn.functional.gelu(torch.nn.functional.layer_norm(x @ W.t() + bb, (128,), gg, be, 1e-5))
    assert float((o.float() - want).abs().max()) < 5e-5
    o = ops.Split(500, 128, d)
    ops.small_in_linear(x[:, :3].contiguous(), W[:, :3].contiguous(), bb, None, None, 0.0, False, ops.ACT_GELU, o)
    want = torch.nn.functional.gelu(x[:, :3] @ W[:, :3].t() + bb)
    assert float((o.float() - want).abs().max()) < 5e-5
    # group max
    x = _rand(30 * 16, 200, seed=9)
    y = torch.empty(30, 200, device=d)
    ys = ops.Split(30, 200, d)
    ops.group_max(x, 30, 16, out_f32=y, out_split=ys)
    want = x.reshape(30, 16, 200).max(1).values
    assert torch.equal(y, want)
    assert float((ys.float() - want).abs().max()) < 1e-4
    # softmax
    s = _rand(300, 200, seed=10, scale=3.0)
    p = ops.Split(300, 200, d, pitch=256, zero=True)
    ops.softmax_split(s, 200, 0.125, p)
    assert float((p.float() - torch.softmax(s * 0.125, -1)).abs().max()) < 2e-6
    # transpose of split planes per (head, cloud)
    B, Hh, L, dh = 2, 3, 50, 16
    src = ops.Split(B * L, 3 * Hh * dh, d)
    ops.split_f32(_rand(B * L, 3 * Hh * dh, seed=11), src)
    Lp = 64
    dst = ops.Split(B * Hh * dh, L, d, pitch=Lp, zero=True)
    from psam_b200 import native as nv

    nv.check(nv.lib().psam_transpose_split(src.ptr(2 * Hh * dh), src.plane, src.pitch, dh, L * src.pitch, dst.ptr(), dst.plane,
                                           dst.pitch, dh * Lp, Hh * dh * Lp, L, dh, Hh, B, nv.stream()), "transpose")
    v = src.float()[:, 2 * Hh * dh:].reshape(B, L, Hh, dh).permute(0, 2, 3, 1).reshape(B * Hh * dh, L)
    assert torch.equal(dst.float(), v)


def test_linear_attention_posenc_misc():
    ops = _ops()
    d = _dev()
    x, x2, w, b, r = _rand(70, 256, seed=1), _rand(70, 256, seed=2), _rand(130, 256, seed=3, scale=0.06), _rand(130, seed=4), _rand(70, 130, seed=5)
    y = ops.linear_f32(x, w, b, x2=x2, r=r, act=ops.ACT_RELU)
    want = torch.relu((x + x2) @ w.t() + b) + r
    torch.testing.assert_close(y, want, atol=2e-5, rtol=1e-5)
    # attention
    Z, Lq, Lk, H, dh = 3, 7, 100, 8, 16
    q, k, v = _rand(Z * Lq, H * dh, seed=6), _rand(Z * Lk, H * dh, seed=7), _rand(Z * Lk, H * dh, seed=8)
    o = ops.attention_f32(q, k, v, Z, Lq, Lk, H, dh)
    qq = q.reshape(Z, Lq, H, dh).transpose(1, 2)
    kk = k.reshape(Z, Lk, H, dh).transpose(1, 2)
    vv = v.reshape(Z, Lk, H, dh).transpose(1, 2)
    want = (torch.softmax(qq @ kk.transpose(-1, -2) / math.sqrt(dh), -1) @ vv).transpose(1, 2).reshape(Z * Lq, H * dh)
    torch.testing.assert_close(o, want, atol=2e-5, rtol=1e-4)
    # positional encoding + labels + range flag
    pe = torch_ref.PointEncoder(256)
    c = (torch.rand(4, 5, 3) * 2 - 1)
    lab = torch.tensor([[1, 0, 1, 0, 1]] * 4)
    want = pe(c, lab)
    from psam_b200 import engine

    got = ops.posenc(c.to(d), pe.pe_layer.positional_encoding_gaussian_matrix.to(d), lab.to(d).int(),
                     pe.point_embeddings[0].weight.detach().to(d), pe.point_embeddings[1].weight.detach().to(d),
                     engine.bad_flag(d))
    torch.testing.assert_close(got.cpu(), want.detach(), atol=3e-5, rtol=1e-5)
    engine.raise_if_out_of_range(d)
    ops.posenc((c * 3).to(d), pe.pe_layer.positional_encoding_gaussian_matrix.to(d), None, None, None, engine.bad_flag(d))
    with pytest.raises(ValueError):
        engine.raise_if_out_of_range(d)
    # broadcast add
    a, bb = _rand(4 * 6 * 8, seed=9), _rand(2 * 6 * 8, seed=10)
    got = ops.add_bcast(a, bb, chunk=6 * 8, rep=2)
    want = a.reshape(4, 48) + bb.reshape(2, 48).repeat_interleave(2, 0)
    torch.testing.assert_close(got.reshape(4, 48), want, atol=0, rtol=0)


def _attention_case(qkv, B, H, L, entry, dh=64):
    from ctypes import byref

    from psam_b200 import native as nv

    ops = _ops()
    D = H * dh
    QKV = ops.Split(B * L, 3 * D, _dev())
    ops.split_f32(qkv, QKV)
    att = ops.Split(B * L, D, _dev())
    att.t.fill_(float("nan"))
    mk = lambda col: QKV.operand(rows=L, k=dh, col=col, nb1=H, b1_stride=dh, nb2=B, b2_stride=L * QKV.pitch)
    qa, ka, va = mk(0), mk(D), mk(2 * D)
    nv.check(getattr(nv.lib(), entry)(byref(qa), byref(ka), byref(va), att.ptr(), att.plane, att.pitch, dh,
                                      L * att.pitch, dh ** -0.5, nv.stream()), entry)
    x = qkv.double().reshape(B, L, 3, H, dh).permute(2, 0, 3, 1, 4)
    want = (torch.softmax(x[0] @ x[1].transpose(-1, -2) * dh ** -0.5, -1) @ x[2]).transpose(1, 2).reshape(B * L, D).float()
    return att.float(), want


@pytest.mark.parametrize("entry", ["psam_attention_bf16x3", "psam_attention_bf16x3_twopass"])
@pytest.mark.parametrize("B,H,L", [(1, 16, 512), (2, 3, 128), (2, 2, 200), (1, 4, 333), (1, 2, 64), (1, 3, 7),
                                   (1, 2, 640), (2, 3, 1000), (1, 16, 2048), (1, 1, 513), (1, 2, 3000)])
def test_fused_attention_tc(B, H, L, entry):
    """psam_attention_bf16x3 (streaming kernel: S ring in TMEM, P written back into TMEM as the A operand of the PV MMA,
    lazily moved reference maximum) and the first-generation two-pass kernels vs fp64 attention."""
    got, want = _attention_case(_rand(B * L, 3 * 64 * H, seed=21), B, H, L, entry)
    err = float((got - want).abs().max())
    assert err < 5e-5 * max(1.0, float(want.abs().max())), err


@pytest.mark.parametrize("B,H,L", [(1, 16, 512), (2, 3, 128), (1, 2, 200), (1, 2, 7), (1, 3, 640), (1, 2, 1100)])
def test_fused_attention_tc_head_dim_88(B, H, L):
    """EVA-giant heads (dh = 88) on the fused kernel: the head is loaded as 64 + 24 columns (TMA zero-fills up to 128), S uses
    4 + 2 k-steps, the PV operand is 256 wide; vs fp64 attention."""
    got, want = _attention_case(_rand(B * L, 3 * 88 * H, seed=23), B, H, L, "psam_attention_bf16x3", dh=88)
    err = float((got - want).abs().max())
    assert err < 5e-5 * max(1.0, float(want.abs().max())), err


@pytest.mark.parametrize("L,step,gain", [(512, 128, 2.0), (1100, 128, 2.0), (512, 32, 4.5), (700, 32, 4.5), (300, 32, 4.5)])
def test_fused_attention_tc_reference_maximum_moves(L, step, gain):
    """Logits that grow along the keys (by far more than the 2^40 slack of the lazy reference maximum) force the rare slow
    path of the streaming kernel: the reference moves and the owning thread rescales O in tensor memory, its running sum
    and - when the jump happens between two 32-key chunks of one block (step = 32) - the P chunks of the current block it
    has already written.  Only a subset of rows is affected (rows whose query is negated see DEcreasing logits)."""
    B, H, dh = 1, 2, 64
    D = H * dh
    g = torch.Generator(device="cpu").manual_seed(5)
    qkv = torch.randn(B * L, 3 * D, generator=g)
    ramp = (torch.arange(L) // step).float()[:, None]           # key block (or 32-key chunk) index
    if step == 32:  # three jumps in a row, at chunks 6, 7, 8: inside block 1 and at the start of block 2 (logits stay moderate)
        ramp = (ramp - 5.0).clamp(0.0, 3.0)
    qkv[:, :D] = torch.randn(L, D, generator=g) * 0.2 + 1.0     # queries: common positive direction ...
    qkv[::3, :D] *= -1.0                                         # ... every third row negated
    qkv[:, D:2 * D] = torch.randn(L, D, generator=g) * 0.2 + gain * ramp  # keys grow with the block / chunk index
    qkv = qkv.to(_dev())
    got, want = _attention_case(qkv, B, H, L, "psam_attention_bf16x3")
    err = float((got - want).abs().max())
    assert err < 5e-5 * max(1.0, float(want.abs().max())), err
    got2, _ = _attention_case(qkv, B, H, L, "psam_attention_bf16x3_twopass")
    assert float((got - got2).abs().max()) < 5e-5 * max(1.0, float(want.abs().max()))


@pytest.mark.parametrize("variant", ["bn256_bk32", "bn256_bk64", "two_cta", "cluster4", "dual_resident", "throughput_policy",
                                     "persistent_bn256", "persistent_bn128", "persistent_bn64", "persistent_3_tiles_per_cta",
                                     "never_persistent", "two_issuers"])
def test_gemm_tc_variants(variant, monkeypatch):
    """Opt-in / policy-selected GEMM variants (psam_gemm_out.variant / tile_hint; the library reads no environment):
    wide tiles with 64-byte-swizzled half-depth stages, the same with 128-byte swizzle, the 2-CTA cta_group::2 kernel,
    W-tile multicast over a 4-CTA cluster, the dual-resident wide-tile kernel (two CTAs per SM) forced, and whatever the
    throughput policy (tile_hint = 1, as baked into the pipelined predictor's graphs) selects."""
    ops = _ops()
    bn, var, hint = {"bn256_bk32": (256, ops.GV_BK32, 0), "bn256_bk64": (256, ops.GV_NO_DUAL, 0), "two_cta": (0, ops.GV_2CTA, 0),
                     "cluster4": (128, 4 << 8, 0), "dual_resident": (256, ops.GV_DUAL, 0), "throughput_policy": (0, 0, 1),
                     # persistent kernel (double-buffered TMEM accumulator, tile loop inside the CTA) at its three tile widths,
                     # with several tiles per CTA forced, and switched off (the one-shot kernels on the many-row shape)
                     "persistent_bn256": (256, ops.GV_PERSIST, 0), "persistent_bn128": (128, ops.GV_PERSIST, 0),
                     "persistent_bn64": (64, ops.GV_PERSIST, 0), "persistent_3_tiles_per_cta": (0, ops.GV_PERSIST | (3 << 16), 1),
                     "never_persistent": (0, ops.GV_NO_PERSIST, 1),
                     # two MMA-issuing warps accumulating into one zero-initialised TMEM accumulator (opt-in experiment)
                     "two_issuers": (256, ops.GV_TWO_ISSUERS | ops.GV_NO_PERSIST, 0)}[variant]
    monkeypatch.setattr(ops, "GEMM_TILE_BN", bn)
    monkeypatch.setattr(ops, "GEMM_VARIANT", var)
    monkeypatch.setattr(ops, "GEMM_TILE_HINT", hint)
    for (M, N, K, sk) in [(512, 3072, 1024, 1), (512, 1024, 2752, 4), (640, 520, 200, 1), (32768, 512, 128, 1)]:
        a, w, b = _rand(M, K, seed=31), _rand(N, K, seed=32, scale=K ** -0.5), _rand(N, seed=33)
        A, W = ops.pack_weight(a), ops.pack_weight(w)
        want = (a.double() @ w.double().t() + b.double())
        if sk > 1:
            r = _rand(M, N, seed=34)
            out = r.clone()
            ops.gemm(A, W, bias=b, out_f32=out, accumulate=True, split_k=sk)
            want = (want + r.double())
        else:
            out = torch.empty(M, N, device=_dev())
            osp = ops.Split(M, N, _dev())
            ops.gemm(A, W, bias=b, out_f32=out, out_split=osp)
            assert float((osp.float() - out).abs().max()) < 3e-5 * max(1.0, float(want.abs().max()))
        err = float((out - want.float()).abs().max())
        assert err < 5e-5 * max(1.0, float(want.abs().max())), (variant, M, N, K, err)


@pytest.mark.parametrize("M,N,K,group_rows", [(32768, 512, 128, 64), (1000, 512, 128, 8), (640, 256, 64, 32), (300, 512, 100, 0),
                                              (128 * 149 * 2 + 5, 256, 128, 1)])
def test_gemm_rowln_fused_layernorm_gelu(M, N, K, group_rows):
    """psam_gemm_rowln_bf16x3: GELU(LayerNorm(A W^T + group bias)) with the full output row inside one CTA (mini-PointNet
    conv2[0..2]) against fp64, including a mean much larger than the spread (the shifted sums must not cancel), ragged last
    tiles, K tails and more tiles than SMs."""
    ops = _ops()
    a, w = _rand(M, K, seed=71), _rand(N, K, seed=72, scale=K ** -0.5)
    gamma, beta = 1.0 + 0.1 * _rand(N, seed=73), 0.1 * _rand(N, seed=74)
    gb = None
    if group_rows:
        gb = _rand((M + group_rows - 1) // group_rows, N, seed=75) + 30.0  # |mean| >> std
    A, W = ops.pack_weight(a), ops.pack_weight(w)
    out = ops.Split(M, N, _dev())
    out.t.fill_(float("nan"))
    ops.gemm_rowln(A, W, gamma, beta, 1e-5, out, gbias=gb, group_rows=group_rows, act=1)
    x = a.double() @ w.double().t()
    if gb is not None:
        x = x + gb.double().repeat_interleave(group_rows, 0)[:M]
    want = torch.nn.functional.gelu(torch.nn.functional.layer_norm(x, (N,), gamma.double(), beta.double(), 1e-5))
    err = float((out.float().double() - want).abs().max())
    assert err < 3e-4 if group_rows else err < 5e-5, (M, N, K, err)
