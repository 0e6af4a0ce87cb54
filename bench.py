#!/usr/bin/env python
"""Benchmark of the Point-SAM hot path (BASELINE.json metric: point-clouds/sec, N=32768, ViT-L, 512x64 groups).

  python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--config c2] [--no-graph] [--dump-outputs DIR]

Headline workload (config c2, BASELINE.json configs[1]): independent single-cloud requests (B=1, N=32768, G=512, K=64,
EVA02-L, one point prompt) through FPS + kNN grouping + mini-PointNet + ViT-L encoder + prompt decoder -> mask logits.
Clouds are independent, so `--depth` of them are in flight per GPU on separate streams / CUDA graphs
(PipelinedPredictor).  ONE STEP = `--clouds-per-step` clouds (default 16 = two rounds of the 8 lanes) so that the
driver's short `--steps 20` run still times >= 0.5 s; `value` stays clouds/s.
  value : device-timed, inputs resident in HBM
  e2e   : the same through the public predictor API with HOST (pinned) buffers: H2D of cloud + prompts and D2H of
          logits + IoU inside the timed region, every result read on the host.
Multi-GPU: one process per GPU (torchrun), clouds sharded by rank, weights replicated.

`--dump-outputs DIR` writes what the last timed step of the `value` arm returned: `masks.npy` (mask logits of every
request of the step, [clouds, masks, N]) and `iou.npy` ([clouds, masks]), float32, plus `c3_iou_rows.npy` (per-cloud IoU
of every prompt iteration) when the c3 arm runs; a rank > 0 adds `_rank<r>` to the names.  All files of all ranks stay
within 64 MB: past that, the logits keep a fixed, seeded sample of the N points.  Only the repo arm dumps.  A lane's
outputs are overwritten by its next request within the step, so the last timed step also copies each request's logits
and IoU on the lane's stream: the `value` of a dump run includes those 2 x requests device-to-device copies.  The
inputs depend only on the arguments, so two builds can be compared output for output.  Compare them with a tolerance,
because repeated runs of one build agree only to rounding: split-K GEMMs accumulate with atomics.

The same line carries "c3" (BASELINE.json configs[2], run after the c2 arms unless --no-c3): a FIXED batch of 32 clouds
sharded contiguously over the ranks (strong scaling), 3 prompt iterations of the evaluation loop
(forward(is_eval=True): GT-driven prompt sampling, mask feedback) as CUDA graphs of 4 clouds, and the NCCL all_gather
of the per-cloud IoU rows INSIDE the timed region.

`--impl reference` times the reference's own algorithm on the host cores: the oracle port (oracle/tokenizer_ref.c FPS
+ oracle/torch_ref.py PyTorch fp32 path; the reference has no CPU FPS and timm is not installable offline, DESIGN.md).
The repo arm never imports oracle/: the cpu_baseline and the same-GPU PyTorch reference run in subprocesses.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # a benchmark run writes nothing into the tree (it may be read-only)
for p in (REPO, os.path.join(REPO, "point-sam_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

CONFIGS = {
    # name: (encoder, N, G, K, clouds per request, prompts, kind)
    "c1": ("eva02_base_patch14_448", 4096, 128, 32, 1, 1, "ball"),
    "c2": ("eva02_large_patch14_448", 32768, 512, 64, 1, 1, "ball"),
    "c2b4": ("eva02_large_patch14_448", 32768, 512, 64, 4, 1, "ball"),
    "c2b8": ("eva02_large_patch14_448", 32768, 512, 64, 8, 1, "ball"),
    "c4": ("eva02_large_patch14_448", 131072, 2048, 256, 1, 1, "kitti"),
    "c5": ("eva_giant_patch14_560", 32768, 512, 64, 1, 1, "ball"),
    "tiny": ("eva02_test_tiny", 2048, 64, 16, 1, 1, "ball"),
}
# config c3: (encoder, N, G, K, total clouds, clouds per graph, prompt iterations, masks per cloud)
C3 = {"c3": ("eva02_large_patch14_448", 32768, 512, 64, 32, 4, 3, 1),
      "c3tiny": ("eva02_test_tiny", 2048, 64, 16, 32, 4, 3, 1)}
METRIC = "point-clouds/sec (N=32768, ViT-L, 512x64 groups)"  # BASELINE.json metric; other --config values are side runs


DUMP_BYTES = 64 << 20  # --dump-outputs: cap on the bytes written by all ranks together


def write_outputs(out_dir, arrays, budget, n_points=0, tag=""):
    """Write every array as out_dir/<name><tag>.npy in float32, in at most `budget` bytes.  Past the budget, the arrays
    whose last axis holds the n_points points of a cloud keep a fixed, seeded sample of those points, so runs with the
    same arguments stay comparable element for element."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: a.detach().float().cpu() for k, a in arrays.items()}
    budget -= 1024 * len(arrays)  # .npy headers
    total = sum(a.numel() * 4 for a in arrays.values())
    if n_points and total > budget:
        per_point = sum(a[..., 0].numel() * 4 for a in arrays.values() if a.shape[-1] == n_points)
        keep = max(1, (budget - (total - per_point * n_points)) // per_point)
        idx = torch.randperm(n_points, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        arrays = {k: a[..., idx] if a.shape[-1] == n_points else a for k, a in arrays.items()}
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}{tag}.npy"), a.numpy())


def peaks():
    try:
        return json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    FIELDS = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def workload_config(args, name):
    """IDENTICAL on the repo arm and the reference arm (the driver compares the two `config` objects); everything
    specific to how one arm runs the workload goes into the line's "run" object instead."""
    if name in C3:
        enc, N, G, K, total, chunk, iters, M = C3[name]
        wl = (f"{name}: fixed batch of {total} clouds sharded over the ranks, N={N}, group_number={G}, group_size={K}, {enc}, "
              f"{iters} GT-driven prompt iterations (forward(is_eval=True)), {M} mask/cloud")
    else:
        enc, N, G, K, bpg, P, kind = CONFIGS[name]
        wl = (f"{name}: independent requests of {bpg} cloud(s), N={N}, group_number={G}, group_size={K}, {enc}, "
              f"{P} point prompt, multimask")
    return {"workload": wl, "parallelism": f"dp{args.gpus} (clouds sharded by rank, weights replicated)",
            "l2": "inputs larger than L2: packed weights (1.3 GB for ViT-L) + activations exceed the 126 MB L2 and are "
                  "re-streamed for every cloud; the input clouds rotate"}


def clouds_per_step(args, name):
    if args.clouds_per_step > 0:
        return args.clouds_per_step
    return 2 * max(1, args.depth) * CONFIGS[name][4]


# --------------------------------------------------------------------------------------------------
# reference arm: the oracle port on the host cores (the ONLY part of this file that touches oracle/)
# --------------------------------------------------------------------------------------------------
def cpu_reference_throughput(cfg, steps: int, warmup: int):
    from oracle import synth, torch_ref

    enc, N, G, K, bpg, P, kind = cfg
    # "all the host threads it can use": PyTorch's CPU GEMMs stop scaling (and regress badly) beyond a few dozen
    # threads on many-socket hosts, so the thread count is capped; PSAM_CPU_THREADS overrides.
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(int(os.environ.get("PSAM_CPU_THREADS", min(ncpu, 32))))
    model = torch_ref.build_model(enc, G, K, seed=1234)
    clouds = [synth.make_batch(bpg, N, 0 + 17 * i, kind) for i in range(2)]
    prompts = [synth.make_prompts(c[0], P, i) for i, c in enumerate(clouds)]
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            xyz, feats = clouds[i % 2]
            pc, pl = prompts[i % 2]
            t0 = time.perf_counter()
            model.predict_masks(xyz, feats, pc, pl, None, True)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    tot = sum(times)
    return steps * bpg / tot, tot / steps * 1e3, torch.get_num_threads()


def run_reference(args):
    """One JSON line: --steps requests of the workload after --warmup untimed ones, timed one by one on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.config if args.config in CONFIGS else "c2"
    cfg = CONFIGS[name]
    steps, warm = args.steps, args.warmup
    v, ms, cores = cpu_reference_throughput(cfg, steps, warm)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "clouds/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, name),
            "cpu_baseline": {"value": v, "unit": "clouds/s", "cores": cores, "kind": "port",
                             "sample": f"{steps} requests of the bench workload ({cfg[4]} cloud each, timed one by one) after {warm} warm-up; oracle "
                                       "port: C restatement of the FPS kernel + PyTorch fp32 CPU path, all host threads"},
            "e2e": {"value": v, "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_gpu_reference(args):
    """Subprocess mode (`--impl gpu-reference`): SURVEY.md 8(d) "GPU reference beside it" - the reference's own GPU
    execution model on this box (its FPS kernel compiled for sm_100a from oracle/_ref when it travelled + cdist/topk +
    PyTorch fp32 eager modules = the oracle restatement on cuda:0), plus full-size parity of the CUDA path against it on
    this very workload.  A reported comparison point only; nothing here is product code."""
    from oracle import build_ref, synth, torch_ref
    from pc_sam.model import build_point_sam

    enc, N, G, K, bpg, P, kind = CONFIGS[args.config]
    steps, warmup = args.steps, args.warmup
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ref = build_ref.load_ref()
    if ref is not None:
        torch_ref.sample_farthest_points = lambda pts, g: ref.sample_farthest_points_cuda(pts.float().contiguous(), g)
    out = {"fps": "reference kernel (oracle/_ref)" if ref is not None else "oracle C port on the host (oracle/_ref absent)",
           "kind": "reference execution model: torkit3d FPS + cdist/topk + PyTorch eager modules, same GPU", "steps": steps}
    torch.manual_seed(1234)
    ours = build_point_sam(enc, G, K).to(dev).eval()
    model = torch_ref.build_model(enc, G, K, seed=1234).to(dev)
    model.load_state_dict(ours.state_dict(), strict=True)
    clouds = [tuple(t.to(dev) for t in synth.make_batch(bpg, N, 0 + 17 * i, kind)) for i in range(2)]
    prompts = [tuple(t.to(dev) for t in synth.make_prompts(c[0].cpu(), P, i)) for i, c in enumerate(clouds)]
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        want_m, want_i = model.predict_masks(*clouds[0], *prompts[0], None, True)
        got_m, got_i = ours.predict_masks(*clouds[0], *prompts[0], None, True)
    err = (got_m - want_m).abs()
    out["parity"] = {"max_abs_err_logits": float(err.max()), "mean_abs_err_logits": float(err.mean()),
                     "logit_range": [float(want_m.min()), float(want_m.max())],
                     "max_abs_err_iou": float((got_i - want_i).abs().max()),
                     "within_1e-3_abs_plus_1e-2_rel": bool((err <= 1e-3 + 1e-2 * want_m.abs()).all()),
                     "sign_agreement": float(((got_m > 0) == (want_m > 0)).float().mean())}
    for tag, tf32 in (("fp32", False), ("tf32", True)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        with torch.no_grad():
            for i in range(warmup):
                model.predict_masks(*clouds[i % 2], *prompts[i % 2], None, True)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                model.predict_masks(*clouds[i % 2], *prompts[i % 2], None, True)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[tag] = {"value": bpg / ms * 1e3, "unit": "clouds/s", "ms_per_step": ms}
    print(json.dumps({"impl": "gpu-reference", "gpu_reference": out}), flush=True)


def _sub_json(argv, timeout):
    """Run this file in a fresh interpreter and return the last JSON line it printed (comparison legs only)."""
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__)] + argv, capture_output=True, text=True, timeout=timeout, env=env)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"unavailable": (r.stderr or "no output")[-200:]}
    except Exception as e:
        return {"unavailable": repr(e)[:200]}


# --------------------------------------------------------------------------------------------------
# instrumentation proxies over the C ABI (roofline passes only, never inside a timed region)
# --------------------------------------------------------------------------------------------------
_PASS_THROUGH = ("psam_version", "psam_fps_workspace_bytes", "psam_border_prompt_workspace_bytes")


def _gemm_meta(a):
    A, W = a[0]._obj, a[1]._obj
    nb = max(1, A.nb1) * max(1, A.nb2)
    return dict(flops=2.0 * A.rows * W.rows * A.k * nb, passes=a[3])


class ProfilingLib:
    """CUDA events around every C-ABI launch."""

    def __init__(self, real):
        self._real, self.records = real, []

    def __getattr__(self, name):
        fn = getattr(self._real, name)
        if not name.startswith("psam_") or name in _PASS_THROUGH:
            return fn

        def wrapped(*a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*a)
            e1.record()
            self.records.append((name, e0, e1, _gemm_meta(a) if name == "psam_gemm_bf16x3" else None))
            return rc

        return wrapped


class OnlyLib:
    """Drops every launch except the named entry points: capturing a step through this proxy yields a CUDA graph that holds
    exactly those launches of the step (same shapes, tiles, epilogues and buffers)."""

    def __init__(self, real, keep):
        self._real, self._keep, self.flops, self.launches = real, set(keep), 0.0, 0

    def __getattr__(self, name):
        fn = getattr(self._real, name)
        if not name.startswith("psam_") or name in _PASS_THROUGH:
            return fn
        if name in self._keep:
            def wrapped(*a):
                if name == "psam_gemm_bf16x3":
                    self.flops += _gemm_meta(a)["flops"]
                self.launches += 1
                return fn(*a)

            return wrapped
        return lambda *a: 0


def only_regime(pp, keep, reps: int):
    """One kernel family in the regime of the timed region, with everything else removed: every lane's step is captured
    once more through OnlyLib into the lane's own graph memory pool (so the kernels run on the buffers the full graphs
    populate), then all `depth` reduced graphs are replayed concurrently `reps` times.
    Returns (elapsed ms per cloud of machine time, launches per cloud, algorithmic GEMM flops per cloud)."""
    from psam_b200 import engine, native as nv, ops

    real = nv.lib()
    graphs, flops, launches = [], 0.0, 0
    prev, ops.GEMM_TILE_HINT = ops.GEMM_TILE_HINT, (1 if pp.depth > 1 and pp.throughput_tiles else 0)
    try:
        for lane in pp.lanes:
            proxy = OnlyLib(real, keep)
            nv._lib = proxy
            g = torch.cuda.CUDAGraph()
            with torch.no_grad(), torch.cuda.graph(g, pool=lane.graph.pool(), stream=lane.stream), engine.block_ln_fold(pp.ln_fold):
                lane._run()
            nv._lib = real
            graphs.append(g)
            flops, launches = proxy.flops, proxy.launches
    finally:
        nv._lib = real
        ops.GEMM_TILE_HINT = prev
    main = torch.cuda.current_stream()

    def go(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(main)
        for lane in pp.lanes:
            lane.stream.wait_event(e0)
        for _ in range(n):
            for lane, g in zip(pp.lanes, graphs):
                with torch.cuda.stream(lane.stream):
                    g.replay()
        for lane in pp.lanes:
            ev = torch.cuda.Event()
            ev.record(lane.stream)
            main.wait_event(ev)
        e1.record(main)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for lane in pp.lanes:  # populate the buffers with real activations
        with torch.cuda.stream(lane.stream):
            lane.graph.replay()
    go(2)
    ms = go(reps)
    return ms / (reps * len(pp.lanes)), launches, flops


# --------------------------------------------------------------------------------------------------
# config c3: fixed batch sharded over the ranks, evaluation loop, all_gather of the IoU rows inside the timed region
# --------------------------------------------------------------------------------------------------
def run_c3(name, args, model, dev, dist, rank, world, barrier, outputs=None):
    from pc_sam.model.loss import compute_iou
    from psam_b200 import synth
    from psam_b200.parallel import gather_metric, plan_graph_chunks, shard_range

    enc, N, G, K, total, chunk, iters, M = C3[name]
    lo, hi = shard_range(total, rank, world)
    n_local = hi - lo
    # clouds per CUDA graph: at most C3's 4, fewer when the rank's shard is small, so that `c3_lanes` graphs stay in flight on
    # every rank count (8 ranks x 4 clouds: four 1-cloud graphs overlap instead of one 4-cloud graph running alone)
    chunk, n_chunks = plan_graph_chunks(n_local, args.c3_lanes, chunk)
    saved = model.prompt_iters
    model.prompt_iters = iters
    n_lanes = min(n_chunks, args.c3_lanes)
    lanes = [model.make_iterative_predictor(chunk, M, N, use_graph=not args.no_graph, throughput_tiles=n_lanes > 1) for _ in range(n_lanes)]
    host = []
    for ci in range(n_chunks):
        xyz = torch.cat([synth.make_batch(1, N, 5000 + lo + ci * chunk + b, "ball")[0] for b in range(chunk)])
        feats = torch.cat([synth.make_batch(1, N, 5000 + lo + ci * chunk + b, "ball")[1] for b in range(chunk)])
        gt = synth.make_region_masks(xyz, M)
        host.append(tuple(t.pin_memory() for t in (xyz, feats, gt)))
    devin = [tuple(t.to(dev) for t in h) for h in host]
    for ln in lanes:
        ln.warmup(*devin[0])
    main = torch.cuda.current_stream()
    rows = torch.zeros((n_local, iters), dtype=torch.float32, device=dev)
    rows_host = torch.zeros((total, iters), dtype=torch.float32).pin_memory()
    done = [torch.cuda.Event() for _ in lanes]
    gathered = torch.cuda.Event()
    gathered.record(main)

    def one_step(inputs, to_host):
        """The whole sharded batch once: chunks round-robin over the lanes, IoU rows on the device, one all_gather."""
        for ln in lanes:
            ln.stream.wait_event(gathered)  # the previous step's gather has consumed `rows`
        for ci in range(n_chunks):
            ln = lanes[ci % len(lanes)]
            outs = ln(*inputs[ci], check=False)
            with torch.no_grad(), torch.cuda.stream(ln.stream):
                gtf = ln.gt.flatten(0, 1)
                for t, o in enumerate(outs):
                    rows[ci * chunk:(ci + 1) * chunk, t] = compute_iou(o["prompt_masks"], gtf).view(chunk, M).mean(dim=1)
                done[ci % len(lanes)].record(ln.stream)
        for ev in done:
            main.wait_event(ev)
        full = gather_metric(rows, total) if world > 1 else rows  # NCCL all_gather of the per-cloud IoU rows
        if to_host:
            rows_host.copy_(full, non_blocking=True)
        gathered.record(main)
        return full

    def timed(inputs, to_host, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(main)
        for ln in lanes:
            ln.stream.wait_event(e0)
        chk = 0.0
        for _ in range(steps):
            one_step(inputs, to_host)
            if to_host:
                main.synchronize()            # the host reads every step's result
                chk += float(rows_host[0, 0])
        e1.record(main)
        barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    steps = max(1, args.steps)
    timed(devin, False, max(3, min(args.warmup, 5)))
    ms_dev = timed(devin, False, steps)
    if outputs is not None:  # this rank's per-cloud IoU rows of the last timed step
        outputs[f"{name}_iou_rows"] = rows.clone()
    timed(host, True, 3)
    ms_e2e = timed(host, True, steps)
    for ln in lanes:
        ln.check()  # deferred validity flags of the whole run (ValueError / RuntimeError like the reference)
    full = one_step(devin, True)
    main.synchronize()
    model.prompt_iters = saved
    h2d = sum(t.numel() * t.element_size() for h in host for t in h)
    return {"config": workload_config(args, name),
            "run": dict(clouds_per_step=total, clouds_per_rank=n_local, clouds_per_graph=chunk, graphs_in_flight=len(lanes),
                        cuda_graph=lanes[0].graph is not None, timed_region_s=ms_dev / 1e3),
            "value": total / (ms_dev / steps / 1e3), "unit": "clouds/s", "ms_per_step": ms_dev / steps, "scaling": "strong",
            "n_gpus": world, "steps": steps,
            "e2e": {"value": total / (ms_e2e / steps / 1e3), "unit": "clouds/s", "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": rows_host.numel() * 4},
            "collective": ("NCCL all_gather of the per-cloud IoU rows [32, %d] inside the timed region" % iters) if world > 1 else
                          "none (single rank)",
            "gpu_launches": lanes[0].launches_per_step * n_chunks * steps, "launches_per_graph": lanes[0].launches_per_step,
            "mean_iou_per_iteration": [float(v) for v in full.mean(dim=0).cpu()]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="c2")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--depth", type=int, default=8, help="clouds in flight per GPU (independent streams/graphs)")
    ap.add_argument("--clouds-per-step", type=int, default=0, help="default: two rounds of the lanes (16 at depth 8)")
    ap.add_argument("--c3-lanes", type=int, default=4, help="config c3: evaluation-loop graphs in flight per GPU")
    ap.add_argument("--no-c3", action="store_true", help="skip the sharded-batch evaluation-loop arm (config c3)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the same-GPU PyTorch-eager reference timing")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy "
                    "(repo arm only; its copies run inside that step)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the repo arm (--impl ours) only")
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "gpu-reference":
        return run_gpu_reference(args)
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dump_tag = f"_rank{rank}" if rank else ""
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from pc_sam.model import build_point_sam
    from psam_b200 import native as nv, synth

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if args.config in C3:  # the sharded evaluation loop as the main (only) arm
        enc, N, G, K = C3[args.config][:4]
        torch.manual_seed(1234)
        model = build_point_sam(enc, G, K).to(dev).eval()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        outputs = {} if args.dump_outputs else None
        r = run_c3(args.config, args, model, dev, dist, rank, world, barrier, outputs)
        if outputs:
            write_outputs(args.dump_outputs, outputs, DUMP_BYTES // world, tag=dump_tag)
        if rank == 0:
            r.update({"metric": "point-clouds/sec (fixed batch of 32 clouds sharded over the ranks, 3 prompt iterations)",
                      "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None, "dtype": "bf16x3",
                      "data": "synthetic", "clocks": sampler.stop()})
            print(json.dumps(r), flush=True)
        if dist is not None:
            dist.destroy_process_group()
        return

    cfg = CONFIGS[args.config]
    enc, N, G, K, bpg, P, kind = cfg
    cps = clouds_per_step(args, args.config) // bpg  # requests per step
    torch.manual_seed(1234)
    model = build_point_sam(enc, G, K).to(dev).eval()
    n_rot = 4
    clouds = [synth.make_batch(bpg, N, 1000 * rank + 17 * i, kind) for i in range(n_rot)]
    prompts = [synth.make_prompts(c[0], P, i) for i, c in enumerate(clouds)]
    host = [tuple(t.pin_memory() for t in (c[0], c[1], p[0], p[1])) for c, p in zip(clouds, prompts)]
    devin = [tuple(t.to(dev) for t in h) for h in host]

    pp = model.make_pipelined_predictor(bpg, N, P, depth=max(1, args.depth), use_graph=not args.no_graph)
    pp.warmup(*devin[0])
    pp.enable_host_results(3)
    pred = pp.lanes[0]
    stream = pred.stream
    main_s = torch.cuda.current_stream()

    def timed(fn, steps):
        """Device-side time of `steps` steps: e0 on the main stream gates every lane, e1 follows all lanes."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(main_s)
        for lane in pp.lanes:
            lane.stream.wait_event(e0)
        for i in range(steps):
            fn(i)
        for lane in pp.lanes:
            done = torch.cuda.Event()
            done.record(lane.stream)
            main_s.wait_event(done)
        e1.record(main_s)
        barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- arm 1: inputs resident in HBM ---------------------------------------------------------
    kept_step, kept = [-1], []  # --dump-outputs: (masks, iou) of every request of the last timed step

    def step_dev(i):
        for c in range(cps):
            t = pp.submit(*devin[(i * cps + c) % n_rot])
            if i == kept_step[0]:  # copied on the lane's stream before the lane's next request overwrites its outputs
                lane = pp.lanes[t % pp.depth]
                with torch.cuda.stream(lane.stream):
                    kept.append((lane.masks.clone(), lane.iou.clone()))

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # samples clocks / throttle reasons over the warm-up and both timed arms
    timed(step_dev, args.warmup)
    if args.dump_outputs:
        kept_step[0] = args.steps - 1
    ms_dev = timed(step_dev, args.steps)
    kept_step[0] = -1
    outputs = {"masks": torch.cat([m for m, _ in kept]).cpu(), "iou": torch.cat([i for _, i in kept]).cpu()} if kept else None
    kept.clear()

    # single-stream latency of one cloud (no overlap between clouds), for the record
    n_single = max(3, min(24, args.steps))
    ms_single = timed(lambda i: pred(*devin[i % n_rot]), n_single) / n_single

    # ---- arm 2: end to end with host buffers (H2D inputs, D2H logits + IoU, every result read) ----
    chk = [0.0]

    def step_e2e(i):
        for c in range(cps):
            t = pp.count
            if t >= pp.slots:  # the result that occupies this ticket's slot (ticket t - slots) has landed: the host reads it
                _, iou_h = pp.result(t - pp.slots, to_host=True)
                chk[0] += float(iou_h[0, 0])
            pp.submit(*host[(i * cps + c) % n_rot], to_host=True)

    timed(step_e2e, args.warmup)
    ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    out_m, out_i = pp.host_out[0]
    h2d = sum(t.numel() * t.element_size() for t in host[0]) * cps
    d2h = (out_m.numel() * 4 + out_i.numel() * 4 + 4) * cps

    # ---- metric reduction over ranks -------------------------------------------------------------
    checksum = torch.tensor([float(out_i.mean())], device=dev)
    if dist is not None:
        gathered = [torch.zeros_like(checksum) for _ in range(world)]
        dist.all_gather(gathered, checksum)
        checksum = torch.stack(gathered).mean()

    total_clouds = args.steps * cps * bpg * world
    value = total_clouds / (ms_dev / 1e3)
    e2e = total_clouds / (ms_e2e / 1e3)
    ms_per_cloud = ms_dev / (args.steps * cps * bpg)

    line = {"metric": METRIC, "value": value, "unit": "clouds/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16x3", "data": "synthetic", "config": workload_config(args, args.config),
            "run": {"clouds_per_step": cps * bpg, "clouds_in_flight": pp.depth, "cuda_graph": pred.graph is not None, "layernorm_free_blocks": pp.ln_fold,
                    "numerics": "split-bf16 x3 tensor-core contractions (fp32-parity mode), fp32 everywhere else",
                    "single_stream_ms_per_cloud": ms_single, "ms_per_cloud": ms_per_cloud,
                    "timed_region_s": ms_dev / 1e3},
            "e2e": {"value": e2e, "unit": "clouds/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": pred.launches_per_step * cps * args.steps, "launches_per_cloud": pred.launches_per_step,
            "clocks": clocks, "mean_iou_pred": float(checksum)}

    # ---- config c3 on the same ranks (the sharded workload: strong scaling, collective inside the timed region) ----
    if not args.no_c3 and args.config == "c2" and os.environ.get("PSAM_PROFILE_STAGE") is None:
        try:
            line["c3"] = run_c3("c3", args, model, dev, dist, rank, world, barrier, outputs)
        except Exception as e:  # must never break the headline line
            line["c3"] = {"unavailable": repr(e)[:200]}
            if dist is not None:
                raise
    if outputs:  # one budget for the outputs of both arms on every rank
        write_outputs(args.dump_outputs, outputs, DUMP_BYTES // world, n_points=N, tag=dump_tag)

    # ---- roofline of the dominant kernel (rank 0) ---------------------------------------------------
    if rank == 0 and not args.no_roofline and pred.graph is not None:
        from psam_b200 import engine, ops

        pk, pk_src = peaks()
        peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        real = nv.lib()
        hint = 1 if pp.depth > 1 and pp.throughput_tiles else 0

        def instrumented(busy_lanes):
            """One eager, event-bracketed pass of lane 0 with the tile policy of the captured graphs; `busy_lanes` other
            lanes keep replaying their graphs meanwhile (the regime of the timed region) or stay idle (serial)."""
            prof = ProfilingLib(real)
            prev, ops.GEMM_TILE_HINT = ops.GEMM_TILE_HINT, hint
            nv._lib = prof
            try:
                with torch.no_grad():
                    for rep in range(2):
                        prof.records.clear()
                        torch.cuda.synchronize()
                        for lane in pp.lanes[1:1 + busy_lanes]:
                            with torch.cuda.stream(lane.stream):
                                for _ in range(10):
                                    lane.graph.replay()
                        with torch.cuda.stream(stream), engine.block_ln_fold(pp.ln_fold):
                            pred._load(*devin[rep % n_rot])
                            if busy_lanes == 0:
                                torch.cuda._sleep(int(25e-3 * 1.9e9))  # let the host run ahead of the device
                            pred._run()
                torch.cuda.synchronize()
            finally:
                nv._lib = real
                ops.GEMM_TILE_HINT = prev
            stages = {}
            for name, a, b, meta in prof.records:
                st = stages.setdefault(name, dict(ms=0.0, n=0, flops=0.0))
                st["ms"] += a.elapsed_time(b)
                st["n"] += 1
                if meta:
                    st["flops"] += meta["flops"]
            return stages

        serial = instrumented(0)
        contended = instrumented(pp.depth - 1)
        gs = serial.get("psam_gemm_bf16x3", dict(ms=1e-9, n=1, flops=0.0))
        gc = contended.get("psam_gemm_bf16x3", dict(ms=1e-9, n=1, flops=0.0))
        tot_serial = sum(s["ms"] for s in serial.values())
        ms_gemm, n_gemm, flops_cloud = only_regime(pp, ("psam_gemm_bf16x3",), reps=12)
        tf_regime, us_launch = flops_cloud / (ms_gemm / 1e3) / 1e12, ms_gemm * 1e3 / max(1, n_gemm)
        traffic, traffic_src = None, None
        for f in ("r02_gemm_traffic.json",):
            try:
                tj = json.load(open(os.path.join(REPO, "profiles", f)))
                traffic, traffic_src = tj["dram_bytes_per_launch"], f"profiles/{f}: {tj.get('how', 'ncu --set full')}"
            except Exception:
                pass
        line["roofline"] = {
            "bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 split-bf16)", "achieved": tf_regime, "peak": peak,
            "unit": "TFLOP/s", "frac": tf_regime / peak, "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": f"{pk_src} sustained bf16",
            "regime": f"the step's {n_gemm} GEMM launches (same tiles, epilogues, buffers as the timed graphs) replayed alone on "
                      f"{pp.depth} concurrent streams; achieved = algorithmic flops 2MNK / elapsed",
            "executed_tflops": 3 * tf_regime, "executed_frac": 3 * tf_regime / peak,
            "launches": n_gemm, "avg_launch_us": us_launch, "algorithmic_gflop_per_cloud": flops_cloud / 1e9,
            "gemm_machine_ms_per_cloud": us_launch * n_gemm / 1e3, "ms_per_cloud": ms_per_cloud,
            "share_of_step": min(1.0, us_launch * n_gemm / 1e3 / ms_per_cloud),
            "whole_step_lower_bound": {"achieved": flops_cloud / (ms_per_cloud / 1e3) / 1e12,
                                       "frac": flops_cloud / (ms_per_cloud / 1e3) / 1e12 / peak,
                                       "note": "all GEMM flops of a cloud / ms_per_cloud of the timed region (everything else counted as GEMM time)"},
            "contended": {"launches": gc["n"], "avg_launch_us": gc["ms"] / gc["n"] * 1e3, "sum_ms": gc["ms"],
                          "bound_ms": ms_per_cloud * pp.depth, "within_bound": bool(gc["ms"] <= ms_per_cloud * pp.depth * 1.25),
                          "note": f"lane 0 event-bracketed (throughput tiles) while the other {pp.depth - 1} lanes replay their graphs"},
            "serial": {"launches": gs["n"], "avg_launch_us": gs["ms"] / gs["n"] * 1e3, "sum_ms": gs["ms"],
                       "achieved": gs["flops"] / (gs["ms"] / 1e3) / 1e12, "share_of_serial_step": gs["ms"] / tot_serial,
                       "note": "same tiles, lane 0 alone: one 48-CTA GEMM at a time cannot fill 148 SMs"},
            "note": "achieved counts the ALGORITHMIC fp32 flops 2MNK; the kernel executes 3 bf16 MMA passes per product (executed_* = x3)"}
        f = serial.get("psam_fps_f32")
        if f:
            fb = (G - 1) * N * 20.0 * bpg
            ms_r, _, _ = only_regime(pp, ("psam_fps_f32",), reps=6)
            line["fps"] = {"ms": f["ms"] / f["n"], "us_per_iter": f["ms"] / f["n"] * 1e3 / (G - 1),
                           "stream_model_gbs": fb / (f["ms"] / f["n"] / 1e3) / 1e9, "hbm_peak_gbs": pk["hbm_gbs"],
                           "frac_of_hbm": fb / (f["ms"] / f["n"] / 1e3) / 1e9 / pk["hbm_gbs"],
                           "in_regime": {"machine_ms_per_cloud": ms_r, "stream_model_gbs": fb / (ms_r / 1e3) / 1e9,
                                         "frac_of_hbm": fb / (ms_r / 1e3) / 1e9 / pk["hbm_gbs"],
                                         "note": f"FPS launches of {pp.depth} clouds in flight (the timed regime): one 8-CTA cluster per "
                                                 "cloud, the clusters of different clouds run side by side"},
                           "note": "byte model (G-1)*N*20 B of SURVEY 8(d) = what the reference kernel streams; this kernel keeps the "
                                   "cloud in registers (real DRAM traffic = the cloud once) and is a latency chain: us_per_iter is the "
                                   "figure of merit for one cloud"}
        k = serial.get("psam_knn_f32")
        if k:
            kb = (2.0 * G * N * 4 + N * 12 + G * K * 12) * bpg
            line["knn"] = {"ms": k["ms"] / k["n"], "ref_equiv_gbs": kb / (k["ms"] / k["n"] / 1e3) / 1e9,
                           "frac_of_hbm": kb / (k["ms"] / k["n"] / 1e3) / 1e9 / pk["hbm_gbs"],
                           "pairs_per_s": G * N * bpg / (k["ms"] / k["n"] / 1e3),
                           "note": "byte model = what cdist + topk move (distance matrix written and read back); this kernel writes "
                                   "no distance matrix, real DRAM traffic is the cloud once"}
        if f and k:
            fb = (G - 1) * N * 20.0 * bpg
            kb = (2.0 * G * N * 4 + N * 12 + G * K * 12) * bpg
            ms_r, _, _ = only_regime(pp, ("psam_fps_f32", "psam_knn_f32"), reps=6)
            line["tokenizer_in_regime"] = {
                "machine_ms_per_cloud": ms_r, "byte_model_gbs": (fb + kb) / (ms_r / 1e3) / 1e9,
                "frac_of_hbm": (fb + kb) / (ms_r / 1e3) / 1e9 / pk["hbm_gbs"], "hbm_peak_gbs": pk["hbm_gbs"],
                "note": f"the FPS + kNN launches of {pp.depth} clouds in flight replayed alone (the timed regime); bytes = SURVEY 8(d) "
                        "byte models (FPS streaming model + kNN reference-equivalent), not DRAM traffic"}
        at = serial.get("psam_attention_bf16x3")
        if at:
            L = bpg * G
            from pc_sam.model.eva import EVA_CONFIGS

            De, depth_e, heads = EVA_CONFIGS[enc][:3]
            aflops = 4.0 * G * G * De * bpg  # 4 L^2 dh H per layer
            line["attention"] = {"us_per_layer": at["ms"] / at["n"] * 1e3, "layers": at["n"],
                                 "algorithmic_tflops": aflops / (at["ms"] / at["n"] / 1e3) / 1e12,
                                 "executed_frac_of_peak": 3 * aflops / (at["ms"] / at["n"] / 1e3) / 1e12 / peak,
                                 "note": "serial, lone launch; tensor-pipe % of the kernel is in profiles/ (ncu)"}
        line["stage_ms_serial"] = {n: round(s["ms"], 4) for n, s in sorted(serial.items(), key=lambda kv: -kv[1]["ms"])}

    if rank == 0:
        # ---- comparison legs in fresh interpreters (the repo arm's process maps only libpsam_b200.so) ----
        if world == 1 and not args.no_cpu_baseline:
            r = _sub_json(["--impl", "reference", "--config", args.config, "--steps", "3", "--warmup", "1"], 900)
            line["cpu_baseline"] = r.get("cpu_baseline", r)
        if world == 1 and not args.no_gpu_reference:
            r = _sub_json(["--impl", "gpu-reference", "--config", args.config, "--steps", "10", "--warmup", "3"], 900)
            line["gpu_reference"] = r.get("gpu_reference", r)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
