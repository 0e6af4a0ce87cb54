"""Automatic mask generation: the numpy restatement (oracle/amg_ref.py) on hand-built cases, argument validation of the
C ABI and of the generator without a GPU; on the GPU every kernel exactly against amg_ref, and the generator end to end
(decoder parity at 64+ prompts per cloud, and its output exactly equal to amg_ref applied to the decoder outputs it used)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import amg_ref

gpu = pytest.mark.gpu
F32 = np.float32


# ------------------------------------------------------------------------------------------------ CPU: amg_ref
def _logits(masks):
    return np.where(np.asarray(masks, dtype=bool), F32(5.0), F32(-5.0))


def test_ref_chain_keeps_a_and_c():
    """A > B > C nested; IoU(A,B) = 0.8, IoU(B,C) = 0.75, IoU(A,C) = 0.6 with nms 0.7: B is suppressed by A, so C (which
    only B would suppress) is kept."""
    N = 100
    A = np.arange(N) < 100
    B = np.arange(N) < 80
    C = np.arange(N) < 60
    logits = _logits(np.stack([A, B, C]))
    out = amg_ref.generate(logits, np.array([0.99, 0.98, 0.97], F32), pred_iou_thresh=0.5, stability_score_thresh=0.5,
                           nms_thresh=0.7)
    assert out["candidates"].tolist() == [0, 2]
    assert out["areas"].tolist() == [100, 60]


def test_ref_score_tie_goes_to_lower_index():
    m = np.zeros((4, 64), dtype=bool)
    m[:, :32] = True  # all identical: only the first in score order survives
    out = amg_ref.generate(_logits(m), np.array([0.9, 0.95, 0.95, 0.9], F32), pred_iou_thresh=0.5, stability_score_thresh=0.5)
    assert out["candidates"].tolist() == [1]
    assert amg_ref.score_order(np.array([0.9, 0.95, 0.95, 0.9], F32), np.ones(4, bool)).tolist() == [1, 2, 0, 3]


def test_ref_iou_exactly_at_threshold_is_not_suppressed():
    N = 40
    a = np.arange(N) < 20
    b = (np.arange(N) >= 10) & (np.arange(N) < 30)  # inter 10, union 30 -> 1/3;  c: inter 20 / union 40 = 0.5
    c = np.arange(N) < 40
    logits = _logits(np.stack([a, c]))
    out = amg_ref.generate(logits, np.array([0.99, 0.98], F32), pred_iou_thresh=0.5, stability_score_thresh=0.5, nms_thresh=0.5)
    assert out["candidates"].tolist() == [0, 1]
    out = amg_ref.generate(logits, np.array([0.99, 0.98], F32), pred_iou_thresh=0.5, stability_score_thresh=0.5, nms_thresh=0.49)
    assert out["candidates"].tolist() == [0]
    _, iou = amg_ref.pairwise_iou(np.stack([a, b]), np.stack([a, b]))
    assert iou[0, 1] == F32(10) / F32(30)


def test_ref_all_negative_row_has_stability_zero():
    x = np.full((2, 50), -3.0, F32)
    x[1, :10] = 0.5  # above t, below t + off: stability 0 / 10
    masks, area, stab, keep = amg_ref.mask_stats(x, np.array([0.99, 0.99], F32), 0.0, 1.0, 0.5, 0.0)
    assert area.tolist() == [0, 10] and stab.tolist() == [0.0, 0.0]
    assert keep.tolist() == [False, True]  # area 0 never passes, even with stability_score_thresh = 0


def test_ref_pack_bits_layout():
    m = np.zeros((1, 40), dtype=bool)
    m[0, [0, 5, 31, 32, 39]] = True
    assert amg_ref.pack_bits(m).tolist() == [[(1 << 0) | (1 << 5) | (1 << 31), (1 << 0) | (1 << 7)]]


# ------------------------------------------------------------------------------------------------ CPU: argument validation
@pytest.fixture(scope="module")
def lib():
    from psam_b200 import build

    return ctypes.CDLL(build.build())


def test_argument_validation_without_gpu(lib):
    """Bad arguments are rejected before any CUDA call (PSAM_ERR_ARG = -1, PSAM_ERR_UNSUPPORTED = -2)."""
    f = ctypes.c_float
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below returns before touching the device
    for name in ("psam_mask_stats_f32", "psam_mask_iou_u32", "psam_mask_nms", "psam_mask_unpack_u8"):
        getattr(lib, name).restype = ctypes.c_int
    assert lib.psam_mask_stats_f32(None, None, 4, 32, f(0), f(1), f(0.88), f(0.95), None, None, None, None, None) == -1
    assert lib.psam_mask_stats_f32(fake, fake, 0, 32, f(0), f(1), f(0.88), f(0.95), fake, fake, fake, fake, None) == -1
    assert lib.psam_mask_stats_f32(fake, fake, 4, 0, f(0), f(1), f(0.88), f(0.95), fake, fake, fake, fake, None) == -1
    assert lib.psam_mask_iou_u32(None, 4, fake, 4, 2, fake, None, None) == -1
    assert lib.psam_mask_iou_u32(fake, 4, fake, 0, 2, fake, None, None) == -1
    assert lib.psam_mask_nms(fake, fake, fake, fake, 0, 4, f(0.7), fake, fake, fake, None) == -1
    assert lib.psam_mask_nms(fake, fake, fake, None, 64, 4, f(0.7), fake, fake, fake, None) == -1
    assert lib.psam_mask_nms(fake, fake, fake, fake, 64, 4, f(0.7), fake, fake, ctypes.c_void_p(258), None) == -1  # unaligned
    assert lib.psam_mask_nms(fake, fake, fake, fake, 16385, 4, f(0.7), fake, fake, fake, None) == -2
    assert lib.psam_mask_unpack_u8(fake, 1, None, 2, 33, fake, None) == -1  # 33 points need 2 words
    assert lib.psam_mask_unpack_u8(fake, 2, None, 0, 33, fake, None) == -1
    lib.psam_mask_nms_workspace_bytes.restype = ctypes.c_size_t
    assert lib.psam_mask_nms_workspace_bytes(1536, 1024) == 16 + 384 * 16 + 1536 * 24 * 8


def test_generator_refuses_cpu_tensors_and_bad_parameters():
    from oracle import synth
    from pc_sam.model import PointCloudAutomaticMaskGenerator, build_point_sam

    m = build_point_sam("eva02_test_tiny", 8, 4)
    xyz, feats = synth.make_batch(1, 64, 0)
    with pytest.raises(RuntimeError):
        PointCloudAutomaticMaskGenerator(m, points_per_cloud=8).generate(xyz, feats)
    for bad in (dict(points_per_cloud=0), dict(points_per_batch=-1), dict(points_per_cloud=6000), dict(points_per_cloud=8.0),
                dict(nms_thresh=float("nan")), dict(pred_iou_thresh=float("inf")), dict(stability_score_offset=-1.0)):
        with pytest.raises(ValueError):
            PointCloudAutomaticMaskGenerator(m, **bad)
    import pc_sam.model

    assert pc_sam.model.PointCloudAutomaticMaskGenerator is PointCloudAutomaticMaskGenerator


# ------------------------------------------------------------------------------------------------ GPU: kernels
DEV = "cuda:0"


def _planted_logits(R, N, t, off, rng):
    x = (rng.standard_normal((R, N)) * 2 * off + t).astype(F32)
    special = np.array([t, t + off, t - off], F32)
    plant = np.concatenate([special, np.nextafter(special, F32(np.inf)), np.nextafter(special, F32(-np.inf))]).astype(F32)
    x.reshape(-1)[:: 3][: min(R * N // 3, 10 * N)] = np.resize(plant, min(R * N // 3, 10 * N))
    x[0] = F32(t - 2 * off - 1)  # empty row (stability 0 / 0)
    if R > 1:
        x[1] = F32(t + 2 * off + 1)  # full row
    return x


def _check_stats(out, ref_args, rows=slice(None)):
    bits, area, stab, keep = (o.cpu().numpy()[rows] for o in out)
    masks, r_area, r_stab, r_keep = amg_ref.mask_stats(*ref_args)
    np.testing.assert_array_equal(bits.view(np.uint32), amg_ref.pack_bits(masks))
    np.testing.assert_array_equal(area, r_area)
    np.testing.assert_array_equal(stab, r_stab)
    np.testing.assert_array_equal(keep.astype(bool), r_keep)


@gpu
@pytest.mark.parametrize("N", [1, 31, 32, 33, 4103, 32768])
@pytest.mark.parametrize("t,off", [(0.0, 1.0), (0.25, 0.125)])
def test_mask_stats_exact(N, t, off):
    from psam_b200 import ops

    rng = np.random.default_rng(N)
    R = 9
    x = _planted_logits(R, N, t, off, rng)
    iou = rng.uniform(0.8, 1.0, R).astype(F32)
    iou[2] = F32(0.88)  # exactly at pred_iou_thresh: filtered out (strict)
    args = (x, iou, t, off, 0.88, 0.5)
    out = ops.mask_stats(torch.from_numpy(x).to(DEV), torch.from_numpy(iou).to(DEV), *args[2:])
    _check_stats(out, args)
    # the same rows at a row offset into a larger table; the rows around them stay untouched
    W = ops.mask_words(N)
    table = (torch.full((R + 5, W), 7, dtype=torch.int32, device=DEV), torch.full((R + 5,), 7, dtype=torch.int32, device=DEV),
             torch.full((R + 5,), 7.0, device=DEV), torch.full((R + 5,), 7, dtype=torch.uint8, device=DEV))
    ops.mask_stats(torch.from_numpy(x).to(DEV), torch.from_numpy(iou).to(DEV), *args[2:], out=table, row0=3)
    _check_stats(table, args, rows=slice(3, 3 + R))
    for t_ in table:
        assert (t_[:3].cpu() == 7).all() and (t_[3 + R:].cpu() == 7).all()


@gpu
def test_mask_stats_unaligned_rows_take_the_scalar_path():
    from psam_b200 import ops

    rng = np.random.default_rng(5)
    R, N = 6, 64
    x = _planted_logits(R, N, 0.0, 1.0, rng)
    iou = np.full(R, 0.95, F32)
    buf = torch.zeros(R * N + 1, device=DEV)
    buf[1:] = torch.from_numpy(x.reshape(-1)).to(DEV)
    out = ops.mask_stats(buf[1:].view(R, N), torch.from_numpy(iou).to(DEV), 0.0, 1.0, 0.88, 0.95)  # 4-byte aligned only
    _check_stats(out, (x, iou, 0.0, 1.0, 0.88, 0.95))


def _random_masks(K, N, rng):
    dens = np.array([0.0, 0.001, 0.01, 0.1, 0.5, 0.9, 0.99, 1.0])
    m = rng.random((K, N)) < dens[np.arange(K) % len(dens)][:, None]
    if K >= 6:
        m[3] = m[4]  # identical rows
        m[5] = ~m[4]  # disjoint from row 4
    return m


@gpu
@pytest.mark.parametrize("K", [1, 63, 64, 65, 1536])
def test_mask_iou_exact(K):
    from psam_b200 import ops

    rng = np.random.default_rng(K)
    N = 4103
    a = _random_masks(K, N, rng)
    b = _random_masks(max(1, K // 2 + 1), N, rng)
    ab, bb = (torch.from_numpy(amg_ref.pack_bits(m).view(np.int32)).to(DEV) for m in (a, b))
    for x, xb in ((a, ab), (b, bb)):
        iou, inter = ops.mask_iou(ab, xb, want_inter=True)
        r_inter, r_iou = amg_ref.pairwise_iou(a, x)
        np.testing.assert_array_equal(inter.cpu().numpy(), r_inter)
        np.testing.assert_array_equal(iou.cpu().numpy(), r_iou)


def _ball_masks(K, N, rng):
    """Overlapping regions of one synthetic cloud: nested and neighbouring balls, so IoUs spread around the thresholds."""
    from oracle import synth

    xyz = synth.make_cloud(N, 3)[0].numpy()
    centres = xyz[rng.integers(0, N, K)]
    radii = rng.uniform(0.1, 0.8, K)
    return np.linalg.norm(xyz[None] - centres[:, None], axis=-1) < radii[:, None]


@gpu
@pytest.mark.parametrize("case", ["ties", "k_150", "k_1000", "all_suppressed", "none_suppressed", "no_survivors", "k_1536"])
def test_mask_nms_exact(case):
    from psam_b200 import ops

    rng = np.random.default_rng(len(case))
    K = {"k_150": 150, "k_1000": 1000, "k_1536": 1536}.get(case, 200)
    N = 2000
    masks = _ball_masks(K, N, rng)
    scores = rng.uniform(0.0, 1.0, K).astype(F32)
    pred_thresh, nms = 0.2, 0.7
    if case == "ties":
        scores = np.round(scores * 4).astype(F32) / F32(4)
    elif case == "all_suppressed":
        masks[:] = masks[0] | True
    elif case == "none_suppressed":
        masks = np.zeros((K, N), dtype=bool)
        masks[np.arange(K), np.arange(K) * (N // K)] = True
    elif case == "no_survivors":
        pred_thresh = 2.0
    logits = _logits(masks)
    params = dict(pred_iou_thresh=pred_thresh, stability_score_thresh=0.5, nms_thresh=nms)
    ref = amg_ref.generate(logits, scores, **params)
    bits, area, stab, keep = ops.mask_stats(torch.from_numpy(logits).to(DEV), torch.from_numpy(scores).to(DEV), 0.0, 1.0,
                                            pred_thresh, 0.5)
    keep_idx, count = ops.mask_nms(bits, area, torch.from_numpy(scores).to(DEV), keep, nms)
    n = int(count.item())
    got = keep_idx.cpu().numpy()
    print(f"[nms] {case}: K={K} passed={ref['passed']} kept={n}")
    np.testing.assert_array_equal(got[:n], ref["candidates"])
    assert (got[n:] == -1).all()
    if case == "all_suppressed":
        assert n == 1
    elif case == "none_suppressed":
        assert n == ref["passed"] > 0
    elif case == "no_survivors":
        assert n == 0
    else:
        assert 0 < n < ref["passed"]
    u = ops.mask_unpack(bits, N, keep_idx[:n]).cpu().numpy()
    np.testing.assert_array_equal(u, masks[ref["candidates"]])


# ------------------------------------------------------------------------------------------------ GPU: end to end
LOW = dict(pred_iou_thresh=-10.0, stability_score_thresh=0.0, nms_thresh=0.5)  # random weights rarely reach SAM's defaults


def _record_decoder(monkeypatch):
    from psam_b200 import engine

    rec = []
    orig = engine.run_mask_decoder

    def wrapped(*a, **k):
        masks, iou = orig(*a, **k)
        rec.append((masks.detach().clone(), iou.detach().clone()))
        return masks, iou

    monkeypatch.setattr(engine, "run_mask_decoder", wrapped)
    return rec


def _check_against_recording(out, rec, gen, N):
    logits = torch.cat([m.reshape(-1, N) for m, _ in rec]).cpu().numpy()
    ious = torch.cat([i.reshape(-1) for _, i in rec]).cpu().numpy()
    assert logits.shape[0] == 3 * gen.points_per_cloud
    ref = amg_ref.generate(logits, ious, **gen.params)
    cand = (out["prompt_index"] * 3 + out["mask_index"]).cpu().numpy()
    print(f"[amg] N={N} P={gen.points_per_cloud} ppb={gen.params['points_per_batch']} passed={ref['passed']} kept={len(cand)}")
    np.testing.assert_array_equal(cand, ref["candidates"])
    np.testing.assert_array_equal(out["masks"].cpu().numpy(), ref["masks"])
    np.testing.assert_array_equal(out["areas"].cpu().numpy(), ref["areas"])
    np.testing.assert_array_equal(out["iou_preds"].cpu().numpy(), ref["iou_preds"])
    np.testing.assert_array_equal(out["stability_scores"].cpu().numpy(), ref["stability_scores"])
    assert out["masks"].dtype == torch.bool and out["areas"].dtype == torch.int64
    return ref


@gpu
@pytest.mark.parametrize("N", [3000, 4096])
@pytest.mark.parametrize("ppb", [7, 64])
@pytest.mark.parametrize("thresholds", ["low", "default"])
def test_generator_end_to_end_tiny(N, ppb, thresholds, monkeypatch):
    from oracle import synth, tokenizer_ref, torch_ref
    from pc_sam.model import PointCloudAutomaticMaskGenerator, build_point_sam

    oracle = torch_ref.build_model("eva02_test_tiny", 96, 16, seed=11)
    model = build_point_sam("eva02_test_tiny", 96, 16)
    model.load_state_dict(oracle.state_dict(), strict=True)
    model = model.cuda().eval()
    xyz, feats = synth.make_batch(1, N, 21)
    P = 64
    gen = PointCloudAutomaticMaskGenerator(model, points_per_cloud=P, points_per_batch=ppb,
                                           **(LOW if thresholds == "low" else {}))
    rec = _record_decoder(monkeypatch)
    out = gen.generate(xyz.to(DEV), feats.to(DEV))
    assert len(rec) == (P + ppb - 1) // ppb
    # prompts: the FPS sample of the cloud
    prompts = xyz[0, torch.from_numpy(tokenizer_ref.fps(xyz.numpy(), P)[0])]
    # (a) decoder parity at 64 prompts per cloud against the fp32 oracle
    with torch.no_grad():
        want_m, want_i = oracle.predict_masks(xyz, feats, prompts.unsqueeze(1), torch.ones((P, 1), dtype=torch.int64), None, True)
    got_m = torch.cat([m for m, _ in rec]).cpu()
    got_i = torch.cat([i for _, i in rec]).cpu()
    np.testing.assert_allclose(got_m.numpy(), want_m.numpy(), atol=1e-3, rtol=1e-2)
    np.testing.assert_allclose(got_i.numpy(), want_i.numpy(), atol=1e-3, rtol=1e-2)
    # (b) the generator's output = amg_ref on exactly the decoder outputs it consumed
    ref = _check_against_recording(out, rec, gen, N)
    np.testing.assert_array_equal(out["prompt_coords"].cpu().numpy(), prompts.numpy()[ref["prompt_index"]])
    if thresholds == "low":
        assert 0 < len(ref["candidates"]) < ref["passed"]  # NMS did real work


@pytest.fixture(scope="module")
def vit_l_model():
    from pc_sam.model import build_point_sam

    torch.manual_seed(1234)
    return build_point_sam("eva02_large_patch14_448", 512, 64).cuda().eval()


@gpu
@pytest.mark.parametrize("thresholds", ["low", "default"])
def test_generator_c2_size_against_recording(thresholds, vit_l_model, monkeypatch):
    """ViT-L, N = 32768, G = 512, P = 512 (K = 1536 candidates), default points_per_batch."""
    from oracle import synth
    from pc_sam.model import PointCloudAutomaticMaskGenerator

    model = vit_l_model
    xyz, feats = synth.make_batch(1, 32768, 31)
    gen = PointCloudAutomaticMaskGenerator(model, **(LOW if thresholds == "low" else {}))
    rec = _record_decoder(monkeypatch)
    out = gen.generate(xyz.to(DEV), feats.to(DEV))
    assert len(rec) == 8
    _check_against_recording(out, rec, gen, 32768)


@gpu
def test_generator_reuses_the_demo_session_encoding_and_checks_inputs():
    from oracle import synth
    from pc_sam.model import PointCloudAutomaticMaskGenerator, build_point_sam
    from psam_b200 import engine

    model = build_point_sam("eva02_test_tiny", 96, 16).cuda().eval()
    xyz, feats = (t.to(DEV) for t in synth.make_batch(1, 2048, 4))
    model.set_pointcloud(xyz, feats)
    cloud = model._cloud
    gen = PointCloudAutomaticMaskGenerator(model, points_per_cloud=32, **LOW)
    out = gen.generate(xyz, feats)
    assert model._cloud is cloud  # not encoded again
    assert out["masks"].shape[1] == 2048
    # prompts beyond the encoder's G come from their own FPS (same points: FPS is prefix-stable)
    big = PointCloudAutomaticMaskGenerator(model, points_per_cloud=128, **LOW).generate(xyz, feats)
    assert big["masks"].shape[1] == 2048
    p = engine.run_amg_prompts(cloud, 128)
    assert torch.equal(p[:, :96], cloud["patches"]["centers"])
    with pytest.raises(ValueError):
        gen.generate(xyz.expand(2, -1, -1), feats.expand(2, -1, -1))
    with pytest.raises(ValueError):
        PointCloudAutomaticMaskGenerator(model, points_per_cloud=4096).generate(xyz, feats)
    model.train()
    with pytest.raises(ValueError):
        gen.generate(xyz, feats)
    model.eval()
    with pytest.raises(ValueError):  # prompts outside [-1, 1] are reported like predict_masks does
        gen.generate(xyz * 3, feats)
