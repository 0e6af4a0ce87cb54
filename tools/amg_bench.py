"""Automatic mask generation timing (PointCloudAutomaticMaskGenerator.generate, one cloud, P = 512 FPS prompts, ViT-L).

  c2: N = 32768, G = 512, K = 64, points_per_batch in {32, 64, 128}
  c4: N = 131072, G = 2048, K = 256 (kitti-like cloud), points_per_batch in {16, 32}

Per setting: ms per cloud from CUDA events after warm-up (the cloud is re-encoded every call), split into encoder,
decoder chunks, stats and NMS + unpack (events around each stage, summed per call); candidates before / after the
filter and kept masks, with SAM's default thresholds and with lowered ones (random weights rarely pass the defaults, and
the lowered ones give the NMS real work); per-kernel times of the mask kernels from one torch.profiler pass (separate
from the timed calls), the stats kernel's achieved bytes/s and the pairwise kernel's word-ops/s, both from shapes;
peak device memory; card name and power limit read in the same run.
usage: python tools/amg_bench.py --config c2 --out DIR [--iters 5 --warmup 2]"""
import argparse
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "point-sam_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402

from pc_sam.model import PointCloudAutomaticMaskGenerator, build_point_sam  # noqa: E402
from psam_b200 import engine, ops, synth  # noqa: E402

CONFIGS = {"c2": (32768, 512, 64, "ball", [32, 64, 128]), "c4": (131072, 2048, 256, "kitti", [16, 32])}
LOW = dict(pred_iou_thresh=-10.0, stability_score_thresh=0.0, nms_thresh=0.7)
KERNELS = ("mask_stats_kernel", "mask_sort_kernel", "mask_suppress_kernel", "mask_scan_kernel", "mask_unpack_kernel")


class StageTimer:
    """CUDA event pairs around the stages of one generate() call (wrapping the engine's / ops' entry points)."""

    def __init__(self, model):
        self.ev = {k: [] for k in ("encoder", "decoder", "stats", "nms_unpack")}
        self.info = {}
        self.patches = []

        def wrap(owner, name, stage, hook=None):
            orig = getattr(owner, name)

            def f(*a, **k):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = orig(*a, **k)
                e.record()
                self.ev[stage].append((s, e))
                if hook:
                    hook(a, out)
                return out

            setattr(owner, name, f)
            self.patches.append((owner, name, orig))

        wrap(model, "_encode", "encoder")
        wrap(engine, "run_mask_decoder", "decoder")
        wrap(ops, "mask_stats", "stats", lambda a, out: self.info.__setitem__("stats_rows", self.info.get("stats_rows", 0) + a[0].numel() // a[0].shape[-1]))
        wrap(ops, "mask_nms", "nms_unpack", lambda a, out: self.info.update(K=a[0].shape[0], W=a[0].shape[1], keep=a[3]))
        wrap(ops, "mask_unpack", "nms_unpack")

    def reset(self):
        for v in self.ev.values():
            v.clear()
        self.info.clear()

    def times(self):
        return {k: sum(s.elapsed_time(e) for s, e in v) for k, v in self.ev.items()}

    def close(self):
        for owner, name, orig in reversed(self.patches):
            setattr(owner, name, orig)


def gpu_identity():
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["sm_max_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # the card name above still identifies the device
        out["power_limit"] = f"unavailable ({e!r})"
    return out


def kernel_times(fn):
    """{kernel: device us per call} over one call of fn under torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                t = getattr(ev, "device_time_total", None)
                if t is None:
                    t = ev.cuda_time_total
                out[k] = out.get(k, 0.0) + float(t)
    return out


def run_setting(model, xyz, feats, ppb, thresholds, args):
    gen = PointCloudAutomaticMaskGenerator(model, points_per_cloud=512, points_per_batch=ppb, **thresholds)
    timer = StageTimer(model)
    try:
        def call():
            model._cloud = None  # re-encode every call: the timed figure is a whole cloud
            return gen.generate(xyz, feats)

        for _ in range(args.warmup):
            call()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        totals, stages = [], []
        for _ in range(args.iters):
            timer.reset()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = call()
            e.record()
            torch.cuda.synchronize()
            totals.append(s.elapsed_time(e))
            stages.append(timer.times())
        peak = torch.cuda.max_memory_allocated()
        K, W = timer.info["K"], timer.info["W"]
        passed = int(timer.info["keep"].sum().item())
        kept = int(out["masks"].shape[0])
    finally:
        timer.close()
    kt = kernel_times(call)
    N = xyz.shape[1]
    stats_bytes = 3 * 512 * N * 4 + K * W * 4  # logits read once, bits written once
    TM = (passed + 63) // 64
    word_ops = TM * (TM + 1) // 2 * 64 * 64 * W  # AND + POPC per word of every pair of the tiles launched with work
    med = sorted(totals)[len(totals) // 2]
    rec = dict(points_per_batch=ppb, thresholds=thresholds or "sam_defaults", ms_per_cloud_median=med,
               ms_per_cloud_all=totals, stages_ms_median={k: sorted(st[k] for st in stages)[len(stages) // 2] for k in stages[0]},
               candidates=K, passed_filter=passed, kept=kept, kernel_us_profiler=kt,
               stats_bytes=stats_bytes, pairwise_word_ops=word_ops, peak_device_memory_gb=peak / 1e9)
    if kt.get("mask_stats_kernel"):
        rec["stats_achieved_GBps"] = stats_bytes / (kt["mask_stats_kernel"] * 1e-6) / 1e9
    if kt.get("mask_suppress_kernel") and word_ops:
        rec["pairwise_Gwordops_per_s"] = word_ops / (kt["mask_suppress_kernel"] * 1e-6) / 1e9
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", choices=sorted(CONFIGS), default="c2")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="directory for r03_amg_<config>.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("amg_bench: needs a CUDA device")
    N, G, K, kind, ppbs = CONFIGS[args.config]
    dev = torch.device("cuda:0")
    torch.manual_seed(1234)
    model = build_point_sam("eva02_large_patch14_448", G, K).to(dev).eval()
    xyz, feats = (t.to(dev) for t in synth.make_batch(1, N, 0, kind))
    t0 = time.time()
    runs = [run_setting(model, xyz, feats, ppb, {}, args) for ppb in ppbs]
    runs += [run_setting(model, xyz, feats, ppbs[len(ppbs) // 2], LOW, args)]
    rec = dict(config=args.config, encoder="eva02_large_patch14_448", N=N, G=G, K=K, cloud=kind, points_per_cloud=512,
               warmup=args.warmup, iters=args.iters, gpu=gpu_identity(), runs=runs, wall_s=time.time() - t0,
               note="L2 not flushed between calls; the 3 x 512 x N fp32 logits of a cloud (200 MB at c2) exceed the 126 MB L2")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"r03_amg_{args.config}.json"), "w") as f:
            json.dump(rec, f, indent=1)
    print(json.dumps(dict(config=args.config, gpu=rec["gpu"], ms=[r["ms_per_cloud_median"] for r in runs])))


if __name__ == "__main__":
    main()
