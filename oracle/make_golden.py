"""ORACLE tooling (NOT product code): mint golden vectors by running the REFERENCE's own Python
modules (imported unmodified from /root/reference) on CPU.

Only two things are substituted, because the reference cannot provide them offline:
  * ``torkit3d._C`` (CUDA-only FPS)  -> oracle.tokenizer_ref.fps, the C restatement of that kernel;
  * ``timm`` (not installed)          -> oracle.torch_ref.Eva, the restatement of timm's EVA blocks.
Everything else (KNNGrouper, PatchEncoder, PointCloudEncoder, Point/MaskEncoder, MaskDecoder,
TwoWayTransformer, PointCloudSAM.predict_masks) is the reference code itself.

Run here (needs /root/reference):   python -m oracle.make_golden
Writes tests/golden/*.npz.  Weights are NOT stored (tens of MB); they are re-created from
``oracle.torch_ref.build_model(seed=...)`` and pinned by a checksum stored in the fixture.

``python -m oracle.make_golden --ref-kernels`` writes tests/golden/ref_kernels.npz instead: outputs of the reference's
CUDA kernels built into oracle/_ref by oracle/build_ref.py, on a GPU.
"""
from __future__ import annotations

import hashlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
REF = "/root/reference"
sys.path.insert(0, REPO)

from oracle import synth, tokenizer_ref, torch_ref  # noqa: E402


def import_reference():
    """Import the reference packages with the two substitutions described above."""
    fake_c = types.ModuleType("torkit3d._C")

    def _fps_cuda(points, num_samples):
        return torch.from_numpy(tokenizer_ref.fps(points.detach().cpu().numpy(), int(num_samples)))

    fake_c.sample_farthest_points_cuda = _fps_cuda
    sys.path.insert(0, os.path.join(REF, "third_party", "torkit3d"))
    sys.modules["torkit3d._C"] = fake_c
    import torkit3d  # noqa: F401

    torkit3d._C = fake_c
    timm = types.ModuleType("timm")
    timm.create_model = torch_ref.create_model
    timm.models = types.ModuleType("timm.models")
    timm.models.eva = types.ModuleType("timm.models.eva")
    timm.models.eva.Eva = torch_ref.Eva
    timm.models.vision_transformer = types.ModuleType("timm.models.vision_transformer")
    timm.models.vision_transformer.VisionTransformer = torch_ref.Eva
    for name in ("timm", "timm.models", "timm.models.eva", "timm.models.vision_transformer"):
        sys.modules[name] = eval(name)
    sys.path.insert(0, REF)
    import pc_sam.model.pc_sam as ref_sam  # noqa: F401
    import pc_sam.model.common as ref_common
    import pc_sam.model.pc_encoder as ref_enc
    import pc_sam.model.prompt_encoder as ref_prompt
    import pc_sam.model.mask_decoder as ref_dec
    import pc_sam.model.transformer as ref_tr

    return dict(sam=ref_sam, common=ref_common, enc=ref_enc, prompt=ref_prompt, dec=ref_dec, tr=ref_tr)


def state_checksum(sd) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()[:16]


def build_reference_model(ref, encoder, G, K, seed):
    oracle_model = torch_ref.build_model(encoder, G, K, seed=seed)
    pe = ref["enc"].PatchEmbed(6, 512, G, K)
    enc = ref["enc"].PointCloudEncoder(pe, torch_ref.create_model(encoder), 256)
    me = ref["prompt"].MaskEncoder(256)
    md = ref["dec"].MaskDecoder(256, ref["tr"].TwoWayTransformer(2, 256, 8, 2048))
    model = ref["sam"].PointCloudSAM(enc, me, md, 5).eval()
    model.load_state_dict(oracle_model.state_dict(), strict=True)  # pins the state-dict key contract
    return model, oracle_model


CASES = [
    # name, B, N, G, K, encoder, prompts, kind, seed
    ("tiny", 2, 1024, 32, 16, "eva02_test_tiny", 2, "ball", 0),
    ("tiny_fused_qkv", 1, 777, 24, 8, "eva_test_tiny_fused", 1, "ball", 1),
    ("tiny_ties", 1, 2048, 64, 32, "eva02_test_tiny", 1, "grid", 2),
]


def sampler_cases():
    """Inputs for the prompt-sampler fixture: (points [B,N,3], gt [B,M,N] bool, list of pred_logits [B*M,N] | None)."""
    B, M, N = 2, 3, 1500
    xyz, _ = synth.make_batch(B, N, 40, "ball")
    g = torch.Generator().manual_seed(41)
    gt = torch.stack([torch.stack([xyz[b, :, m % 3] > (-0.2 + 0.25 * m) for m in range(M)]) for b in range(B)])
    sign = gt.reshape(B * M, N).float() * 2 - 1
    noisy = sign * (torch.rand(B * M, N, generator=g) * 2 - 0.35)          # ~17% of the points flip
    only_fn = torch.where(gt.reshape(B * M, N) & (torch.rand(B * M, N, generator=g) < 0.2), -torch.ones(1), sign)
    only_fp = torch.where(~gt.reshape(B * M, N) & (torch.rand(B * M, N, generator=g) < 0.2), torch.ones(1), sign)
    mixed = noisy.clone()
    mixed[0] = sign[0]              # perfect prediction for one mask -> ground-truth fallback (common.py:420-428)
    mixed[1] = only_fn[1]
    mixed[2] = only_fp[2]
    return xyz, gt, [None, noisy, only_fn, only_fp, sign, mixed]


@torch.no_grad()
def sampler_fixture(ref, out_dir):
    """sample_prompts_adapter of the reference (pc_sam/model/common.py:287-318) with the CUDA-only chamfer wrapper
    replaced by the oracle's exact nearest-neighbour (same arithmetic as chamfer_distance_kernel.cu:62-76)."""
    common = ref["common"]

    def fake_chamfer(xyz1, xyz2, **kw):
        _, d12 = tokenizer_ref.knn(xyz1.numpy(), xyz2.numpy(), 1)
        _, d21 = tokenizer_ref.knn(xyz2.numpy(), xyz1.numpy(), 1)
        return torch.from_numpy(d12[..., 0]), torch.from_numpy(d21[..., 0])

    common.chamfer_distance = fake_chamfer
    xyz, gt, preds = sampler_cases()
    pack = dict(xyz=xyz.numpy(), gt=gt.numpy(), n=len(preds))
    for i, pr in enumerate(preds):
        c, l = common.sample_prompts_adapter(xyz, gt, pr, is_eval=True)
        oc, ol = torch_ref.sample_prompts_eval(xyz, gt, pr)
        assert torch.equal(c, oc) and torch.equal(l, ol), f"oracle sampler differs from the reference in case {i}"
        if pr is not None:
            pack[f"pred{i}"] = pr.numpy()
        pack[f"coords{i}"] = c.numpy()
        pack[f"labels{i}"] = l.numpy()
    np.savez_compressed(os.path.join(out_dir, "prompt_sampler.npz"), **pack)
    print("prompt sampler fixture written:", [tuple(pack[f"coords{i}"].shape) for i in range(len(preds))])


VORONOI = dict(B=2, N=3000, G=96, hidden=64, out=96, seed=7)      # PatchEmbedNN(7, hidden, out, G)
HIER = dict(B=2, N=2000, G=(128, 32), K=(32, 16), radius=(0.2, 0.4), out=96, seed=9)  # PatchEmbedHier(6, out, G, K, radius)
GROUPER_OPTS = dict(B=2, N=1500, G=40, K=24, radius=0.3, seed=8)   # KNNGrouper(use_fps=False, centralize_features=True)


@torch.no_grad()
def variant_fixture(ref, out_dir):
    """Outputs of the reference's own NNGrouper / PatchEmbedNN (Voronoi tokenizer, common.py:190-236, pc_encoder.py:147-197) and
    of KNNGrouper with use_fps=False / centralize_features=True (common.py:93-96, :116-118), exact-distance cdist."""
    orig = torch.cdist
    torch.cdist = lambda a, b, **kw: orig(a, b, compute_mode="donot_use_mm_for_euclid_dist")
    try:
        v = VORONOI
        xyz, feats = synth.make_batch(v["B"], v["N"], v["seed"], "ball")
        torch.manual_seed(4321)
        oracle = torch_ref.PatchEmbedNN(7, v["hidden"], v["out"], v["G"]).eval()
        model = ref["enc"].PatchEmbedNN(7, v["hidden"], v["out"], v["G"]).eval()
        model.load_state_dict(oracle.state_dict(), strict=True)
        patches = model(xyz, feats)
        want = oracle(xyz, feats)
        for k in ("features", "centers", "nn_idx", "embeddings"):
            assert torch.allclose(patches[k].double(), want[k].double(), atol=1e-6), k
        h = HIER
        xyz3, feats3 = synth.make_batch(h["B"], h["N"], h["seed"], "ball")
        torch.manual_seed(4322)
        oracle_h = torch_ref.PatchEmbedHier(6, h["out"], list(h["G"]), list(h["K"]), list(h["radius"])).eval()
        model_h = ref["enc"].PatchEmbedHier(6, h["out"], list(h["G"]), list(h["K"]), list(h["radius"])).eval()
        model_h.load_state_dict(oracle_h.state_dict(), strict=True)
        p1, p2 = model_h(xyz3, feats3)
        w1, w2 = oracle_h(xyz3, feats3)
        assert torch.allclose(p1["embeddings"], w1["embeddings"], atol=1e-5) and torch.allclose(p2["embeddings"], w2["embeddings"], atol=1e-5)
        g = GROUPER_OPTS
        xyz2, feats2 = synth.make_batch(g["B"], g["N"], g["seed"], "ball")
        grp = ref["common"].KNNGrouper(g["G"], g["K"], radius=g["radius"], centralize_features=True)
        out2 = grp(xyz2, feats2, use_fps=False)
        np.savez_compressed(
            os.path.join(out_dir, "variants.npz"),
            voronoi_meta=np.array([v["B"], v["N"], v["G"], v["hidden"], v["out"], v["seed"]]),
            voronoi_weights_checksum=state_checksum(model.state_dict()),
            voronoi_xyz=xyz.numpy(), voronoi_feats=feats.numpy(), voronoi_features=patches["features"].numpy(),
            voronoi_centers=patches["centers"].numpy(), voronoi_nn_idx=patches["nn_idx"].numpy().astype(np.int32),
            voronoi_embeddings=patches["embeddings"].numpy(),
            hier_weights_checksum=state_checksum(model_h.state_dict()), hier_xyz=xyz3.numpy(), hier_feats=feats3.numpy(),
            hier_centers1=p1["centers"].numpy(), hier_centers2=p2["centers"].numpy(), hier_emb1=p1["embeddings"].numpy(),
            hier_emb2=p2["embeddings"].numpy(), hier_knn2_sorted=torch.sort(p2["knn_idx"], -1).values.numpy().astype(np.int32),
            grouper_meta=np.array([g["B"], g["N"], g["G"], g["K"], g["seed"]]), grouper_radius=g["radius"],
            grouper_xyz=xyz2.numpy(), grouper_feats=feats2.numpy(), grouper_features_sorted=_sorted_groups(out2).numpy(),
            grouper_centers=out2["centers"].numpy(), grouper_fps_idx=out2["fps_idx"].numpy().astype(np.int32),
        )
        print("variant fixture written: voronoi embeddings", tuple(patches["embeddings"].shape), "grouper features",
              tuple(out2["features"].shape))
    finally:
        torch.cdist = orig


REF_FPS_CASES = [(2, 4096, 128, "grid", 1), (1, 700, 64, "grid", 2), (4, 1024, 512, "ball", 3), (1, 32768, 512, "ball", 4),
                 (2, 3000, 300, "grid", 5), (1, 50, 50, "grid", 6)]                   # B, N, G, kind, seed
REF_FPS_STREAMING_CASES = [(200000, 48, "ball"), (200000, 40, "grid"), (524288, 40, "ball"), (524288, 24, "grid")]  # N, G, kind
REF_FPS_STREAMING_SEED = 13                                                          # B = 1
REF_NN = dict(N=5000, split=1800, seed=9)  # nearest-neighbour distance from xyz[0, :split] to xyz[0, split:]


@torch.no_grad()
def ref_kernel_fixture(out_dir):
    """Outputs of the reference's own CUDA kernels (sample_farthest_points_kernel.cu, chamfer_distance_kernel.cu) as
    oracle/build_ref.py compiles them for sm_100a into oracle/_ref; needs a GPU.  Inputs come from oracle/synth."""
    from oracle import build_ref

    ref = build_ref.load_ref()
    if ref is None:
        raise RuntimeError("oracle/_ref is not built: run `python -m oracle.build_ref` next to the reference sources")
    d = torch.device("cuda", 0)
    pack = {}
    for i, (B, N, G, kind, seed) in enumerate(REF_FPS_CASES):
        xyz, _ = synth.make_batch(B, N, seed, kind)
        pack[f"fps{i}"] = ref.sample_farthest_points_cuda(xyz.to(d), G).cpu().numpy()
    for N, G, kind in REF_FPS_STREAMING_CASES:
        xyz, _ = synth.make_batch(1, N, REF_FPS_STREAMING_SEED, kind)
        pack[f"fps_streaming_{N}_{G}_{kind}"] = ref.sample_farthest_points_cuda(xyz.to(d), G).cpu().numpy()
    xyz, _ = synth.make_batch(1, REF_NN["N"], REF_NN["seed"])
    a, b = xyz[0, :REF_NN["split"]].to(d), xyz[0, REF_NN["split"]:].to(d)
    pack["nn_dist"] = ref.chamfer_distance_forward_cuda(a[None], b[None])[0][0].cpu().numpy()
    np.savez_compressed(os.path.join(out_dir, "ref_kernels.npz"), **pack)
    print("reference kernel fixture written:", {k: v.shape for k, v in pack.items()})


def _sorted_groups(out):
    """Group features with the K members of every group ordered by key index (the reference's topk order is unspecified)."""
    order = torch.argsort(out["knn_idx"], dim=-1)
    return torch.gather(out["features"], 2, order.unsqueeze(-1).expand_as(out["features"]))


@torch.no_grad()
def main():
    torch.set_num_threads(8)
    out_dir = os.path.join(REPO, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    if "--ref-kernels" in sys.argv:
        return ref_kernel_fixture(out_dir)
    ref = import_reference()
    if "--only-variants" in sys.argv:
        return variant_fixture(ref, out_dir)
    sampler_fixture(ref, out_dir)
    variant_fixture(ref, out_dir)
    if "--only-sampler" in sys.argv:
        return
    for name, B, N, G, K, encoder, P, kind, seed in CASES:
        xyz, feats = synth.make_batch(B, N, seed, kind)
        pc, pl = synth.make_prompts(xyz, P, seed)
        model, _ = build_reference_model(ref, encoder, G, K, seed=1234 + seed)
        # --- the reference's own code path -----------------------------------------------------
        emb, patches = model.pc_encoder(xyz, feats)
        masks, iou = model.predict_masks(xyz, feats, pc, pl, None, True)
        best = torch.argmax(iou, dim=1)
        pm = torch.gather(masks, 1, best[:, None, None].expand(-1, 1, masks.shape[-1]))[:, 0]
        masks2, iou2 = model.predict_masks(xyz, feats, pc, pl, pm, False)
        # exact-distance variant of the same reference code (cdist without the matmul expansion):
        # this is the semantics the CUDA path implements; the difference to the run above is the
        # reference's own backend-dependent rounding noise and is recorded in the fixture.
        orig = torch.cdist
        torch.cdist = lambda a, b, **kw: orig(a, b, compute_mode="donot_use_mm_for_euclid_dist")
        try:
            masks_x, iou_x = model.predict_masks(xyz, feats, pc, pl, None, True)
            masks2_x, iou2_x = model.predict_masks(xyz, feats, pc, pl, pm, False)
            interp_idx, interp_w = ref["common"].compute_interp_weights(xyz, patches["centers"])
        finally:
            torch.cdist = orig
        knn_sorted = torch.sort(patches["knn_idx"], dim=-1).values
        np.savez_compressed(
            os.path.join(out_dir, f"{name}.npz"),
            meta=np.array([B, N, G, K, P, seed]), encoder=encoder, kind=kind,
            weights_checksum=state_checksum(model.state_dict()),
            xyz=xyz.numpy(), feats=feats.numpy(), prompt_coords=pc.numpy(), prompt_labels=pl.numpy(),
            fps_idx=patches["fps_idx"].numpy(), centers=patches["centers"].numpy(),
            knn_idx_sorted=knn_sorted.numpy().astype(np.int32),
            patch_embeddings=patches["embeddings"].numpy(), pc_embeddings=emb.numpy(),
            masks_mm=masks.numpy(), iou_mm=iou.numpy(), masks2_mm=masks2.numpy(), iou2_mm=iou2.numpy(),
            masks=masks_x.numpy(), iou=iou_x.numpy(), masks2=masks2_x.numpy(), iou2=iou2_x.numpy(),
            prompt_mask=pm.numpy(), interp_idx_sorted=torch.sort(interp_idx, -1).values.numpy().astype(np.int32),
            interp_w_sorted=torch.sort(interp_w, -1).values.numpy(),
        )
        print(f"{name}: masks {tuple(masks.shape)} |mm-exact| max {float((masks - masks_x).abs().max()):.3e} "
              f"logit range [{float(masks_x.min()):.2f},{float(masks_x.max()):.2f}]")

    # FPS-only fixtures at the reference test's shapes (test_sample_farthest_points.py:41-49) in
    # float32, plus tie-heavy grids; expected indices come from the literal kernel simulation and are
    # cross-checked against the reference test's numpy oracle where no tie exists.
    fps_cases = [(1, 31, 2, "ball"), (2, 1024, 128, "ball"), (3, 1025, 129, "ball"), (4, 1024, 512, "ball"),
                 (2, 8192, 2048, "ball"), (2, 4096, 128, "grid"), (1, 700, 64, "grid"), (1, 32768, 512, "ball"),
                 (1, 40000, 300, "kitti")]
    pack = {}
    for i, (B, N, G, kind) in enumerate(fps_cases):
        xyz, _ = synth.make_batch(B, N, 100 + i, kind)
        idx = tokenizer_ref.fps(xyz.numpy(), G)
        assert (idx == tokenizer_ref.fps_closed(xyz.numpy(), G)).all()
        if kind != "grid" and N <= 8192:
            assert (idx == tokenizer_ref.fps_numpy(xyz.numpy().astype(np.float64), G)).all(), (B, N, G)
        pack[f"case{i}"] = np.array([B, N, G, 100 + i])
        pack[f"kind{i}"] = kind
        pack[f"idx{i}"] = idx.astype(np.int32)
    np.savez_compressed(os.path.join(out_dir, "fps_cases.npz"), n=len(fps_cases), **pack)
    print("fps fixtures written")


if __name__ == "__main__":
    main()
