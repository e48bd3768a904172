"""SURVEY.md 8 a12 / INTEGRATION.md section 1: the reference's training loop (``train.train_moco``) runs on the GPU with
ONLY the import swap -- MemoryMoCo, NCESoftmaxLoss, DistributedShufle, moment_update from moco_b200 -- and reproduces
the pure reference run from the same seeds (tests/golden/dropin.npz): same losses, same queue contents and ring
position, same trained and EMA weights."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_train_moco_with_the_import_swap_matches_the_reference():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_train_py.py")], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert p.returncode == 0 and lines, p.stderr[-3000:]
    r = json.loads(lines[-1])
    # three steps of fp32 ResNet-18 on 16 images: the head sees bf16-rounded negatives / queries (2^-9 per operand),
    # everything else is the same arithmetic
    assert abs(r["ref_loss"] - r["new_loss"]) < 5e-3 * max(1.0, abs(r["ref_loss"])), r
    assert abs(r["ref_prob"] - r["new_prob"]) < 5e-2 * r["ref_prob"] + 1e-6, r
    assert r["ref_index"] == r["new_index"] == 48, r
    assert r["memory_max_abs_diff"] < 2e-3, r            # enqueued keys come from an EMA encoder 3 SGD steps apart at most
    assert r["fc_rel_diff"] < 2e-2 and r["ema_fc_rel_diff"] < 1e-3, r
