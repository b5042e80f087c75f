"""The UNMODIFIED reference harness — ``CDEvaluator.eval_models`` (reference models/evaluator.py:166-180) and the body of
``CDTrainer.train_models``' inner loop (models/trainer.py:299-310) — run from the reference copy under
``baseline/_ref/ref`` on the shipped LEVIR sample images and a fabricated ``best_ckpt.pt``:

  * CPU (here): on the reference's own class — pins the oracle and the harness driver against the reference's evaluator
    (identical confusion matrix and scores);
  * GPU: on the native drop-in class through ``dahitra_b200.launch.install`` — the ``log_test.txt`` scores must be the
    oracle's, and the native forward must pick up the weights the reference trainer just updated.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("DAHITRA_REFERENCE", os.path.join(ROOT, "baseline", "_ref", "ref"))
have_ref = os.path.exists(os.path.join(REF, "models", "evaluator.py")) and os.path.isdir(os.path.join(REF, "data", "LEVIR_CD", "train", "A"))


def run_harness(impl, device, what="eval,train"):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "ref_harness.py"), "--ref", REF, "--impl", impl,
                        "--device", device, "--what", what], cwd=ROOT, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    line = [l for l in r.stdout.splitlines() if "HARNESS_JSON " in l][-1]
    return json.loads(line.split("HARNESS_JSON ", 1)[1])


@pytest.mark.skipif(not have_ref, reason=f"original DAHiTra sources and LEVIR samples not found at {REF} "
                                         "(set DAHITRA_REFERENCE or run baseline/install_reference.py)")
def test_reference_evaluator_on_reference_class_equals_oracle_cpu():
    out = run_harness("reference", "cpu", what="eval")
    assert out["eval_net_class"] == "models.networks"
    assert out["eval_cm"] == out["oracle_cm"]
    for k, v in out["oracle_scores"].items():
        assert out["eval_scores"][k] == pytest.approx(v, rel=1e-12, abs=1e-12)
    assert out["logits_max_abs_diff_vs_oracle"] < 1e-5 and out["argmax_agree_vs_oracle"] == 1.0
    assert "mf1: %.5f" % out["oracle_scores"]["mf1"] in out["eval_log"]


@pytest.mark.gpu
@pytest.mark.skipif(not have_ref, reason=f"original DAHiTra sources and LEVIR samples not found at {REF} "
                                         "(set DAHITRA_REFERENCE or run baseline/install_reference.py)")
def test_unmodified_evaluator_and_trainer_on_native_module():
    out = run_harness("native", "cuda")
    print("[harness]", {k: out[k] for k in ("eval_net_class", "eval_cm", "oracle_cm", "logits_max_abs_diff_vs_oracle",
                                            "argmax_agree_vs_oracle", "train_losses", "train_eval_after_max_abs_diff_vs_oracle")})
    assert out["net_class"] == "dahitra_b200.networks.BASE_Transformer_UNet"
    assert out["eval_net_class"] == "dahitra_b200.networks" and out["train_net_class"] == "dahitra_b200.networks"
    cm, ocm = np.array(out["eval_cm"]), np.array(out["oracle_cm"])
    assert cm.sum() == ocm.sum() == 4 * 256 * 256
    assert np.abs(cm - ocm).sum() <= 2e-3 * ocm.sum()              # >= 99.9 % of the pixels in the same cell
    assert out["argmax_agree_vs_oracle"] >= 0.999
    assert out["logits_max_abs_diff_vs_oracle"] <= 1e-4 + 1e-3 * 0.1   # define_G logits are O(0.05)
    for k, v in out["oracle_scores"].items():
        assert out["eval_scores"][k] == pytest.approx(v, abs=3e-3)
    assert "mf1: %.5f" % out["eval_scores"]["mf1"] in out["eval_log"]
    # three steps of the reference trainer's loop body: loss goes down, 425-key checkpoint, and the native eval-mode
    # forward afterwards runs on the UPDATED weights (fp64 oracle on the trainer's state_dict as the yardstick)
    ls = out["train_losses"]
    assert ls[-1] < ls[0] and out["ckpt_keys"] == 425
    assert out["train_eval_after_max_abs_diff_vs_oracle"] <= 1e-4 + 2e-3 * out["train_eval_after_ref_absmax"]
