"""bench.py: --steps / --warmup are used as given, and --dump-outputs writes the results of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_times_the_requested_steps(tmp_path):
    """The host reference arm times --steps requests after --warmup untimed ones, whatever their number."""
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--config", "tiny", "--steps", "23",
                        "--warmup", "0"], check=True, capture_output=True, text=True, cwd=str(tmp_path))
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 23 and line["warmup"] == 0
    assert line["cpu_baseline"]["sample"].startswith("23 requests")


@pytest.mark.gpu
def test_bench_dump_outputs_hold_the_last_timed_step(tmp_path):
    from pc_sam.model import build_point_sam
    from psam_b200 import synth

    steps, cps, N = 2, 3, 2048
    out = tmp_path / "outputs"
    subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--config", "tiny", "--steps", str(steps), "--warmup", "1",
                    "--depth", "2", "--clouds-per-step", str(cps), "--no-roofline", "--no-cpu-baseline", "--no-gpu-reference",
                    "--dump-outputs", str(out)], check=True, cwd=str(tmp_path))
    masks, iou = np.load(out / "masks.npy"), np.load(out / "iou.npy")
    assert masks.dtype == np.float32 and masks.shape == (cps, 3, N) and iou.shape == (cps, 3)
    # the same weights and inputs as the bench's tiny config: seed 1234, four seeded clouds used in rotation
    torch.manual_seed(1234)
    model = build_point_sam("eva02_test_tiny", 64, 16).cuda().eval()
    d = torch.device("cuda:0")
    for c in range(cps):
        j = ((steps - 1) * cps + c) % 4
        xyz, feats = synth.make_batch(1, N, 17 * j)
        pc, pl = synth.make_prompts(xyz, 1, j)
        with torch.no_grad():
            want_m, want_i = model.predict_masks(xyz.to(d), feats.to(d), pc.to(d), pl.to(d), None, True)
        np.testing.assert_allclose(masks[c:c + 1], want_m.cpu().numpy(), atol=1e-3, rtol=1e-2)
        np.testing.assert_allclose(iou[c:c + 1], want_i.cpu().numpy(), atol=1e-3, rtol=1e-2)
