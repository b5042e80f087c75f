"""Device-side confusion matrix / scores (SURVEY.md §8 f1) against the numpy restatement of misc/metric_tool.py,
which is itself pinned against the reference module when the original DAHiTra sources are present ($DAHITRA_REFERENCE,
else the copy baseline/install_reference.py places under baseline/_ref/ref)."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as MO

REF_DIR = os.environ.get("DAHITRA_REFERENCE", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                           "baseline", "_ref", "ref"))
REF = os.path.join(REF_DIR, "misc", "metric_tool.py")


def _maps(seed, n, nc, ignore=True):
    rng = np.random.RandomState(seed)
    gt = rng.randint(0, nc, size=n).astype(np.int64)
    pr = rng.randint(0, nc, size=n).astype(np.int64)
    if ignore:
        gt[rng.rand(n) < 0.05] = 255
    return pr, gt


@pytest.mark.skipif(not os.path.exists(REF), reason=f"original DAHiTra sources not found: {REF} "
                                                   "(set DAHITRA_REFERENCE or run baseline/install_reference.py)")
def test_oracle_matches_reference_metric_tool():
    spec = importlib.util.spec_from_file_location("ref_metric_tool", REF)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    for nc in (2, 5):
        pr, gt = _maps(nc, 50_000, nc)
        cm_ref = ref.get_confuse_matrix(nc, [gt.reshape(100, 500)], [pr.reshape(100, 500)])
        cm = MO.confuse_matrix(nc, [gt.reshape(100, 500)], [pr.reshape(100, 500)])
        assert np.array_equal(cm, cm_ref)
        s_ref, s = ref.cm2score(cm_ref), MO.cm2score(cm)
        assert s.keys() == s_ref.keys()
        for k in s:
            assert s[k] == s_ref[k], k
        assert ref.cm2F1(cm_ref) == s["mf1"]


def test_scores_match_oracle_formulas():
    from dahitra_b200.metrics import cm2score, cm2F1
    cm = np.array([[9_000_000, 12_345], [54_321, 700_000]], dtype=np.float64)   # LEVIR-like imbalance
    a, b = cm2score(cm), MO.cm2score(cm)
    assert a.keys() == b.keys()
    for k in a:
        assert a[k] == b[k], k                                                 # bit-identical float64
    assert cm2F1(cm) == b["mf1"]
    z = np.zeros((5, 5))                                                       # empty matrix: all-zero scores, no NaN
    assert all(v == 0 for v in cm2score(z).values())


@pytest.mark.gpu
@pytest.mark.parametrize("nc,n", [(2, 64 * 256 * 256), (5, 1024 * 1024), (2, 1000003), (5, 17), (3, 0)])
def test_device_confusion_matrix_bit_exact(nc, n):
    from dahitra_b200.metrics import confusion_matrix, DeviceConfuseMatrixMeter
    pr, gt = _maps(7 + nc, max(n, 1), nc)
    pr, gt = pr[:n], gt[:n]
    ref = MO.confuse_matrix(nc, [gt], [pr]) if n else np.zeros((nc, nc))
    p_dev = torch.from_numpy(pr).cuda()
    cm = confusion_matrix(p_dev.to(torch.uint8), torch.from_numpy(gt).cuda(), nc)        # int64 labels with 255 = ignore
    assert np.array_equal(cm.cpu().numpy(), ref.astype(np.int64))
    cm2 = confusion_matrix(p_dev, torch.from_numpy(gt).cuda().to(torch.uint8), nc, out=cm.clone())   # accumulates
    assert np.array_equal(cm2.cpu().numpy(), 2 * ref.astype(np.int64))
    if n:
        meter = DeviceConfuseMatrixMeter(nc)
        f1 = meter.update_cm(p_dev, torch.from_numpy(gt).cuda())
        assert f1 == MO.cm2score(ref)["mf1"]
        assert meter.get_scores()["miou"] == MO.cm2score(ref)["miou"]


@pytest.mark.gpu
def test_fused_argmax_feeds_the_meter(levir_template):
    """classifier's fused uint8 argmax -> device confusion matrix == torch.argmax -> host bincount (the reference path)."""
    from dahitra_b200.metrics import confusion_matrix
    from dahitra_b200.networks import BASE_Transformer_UNet
    from oracle import synth
    net = BASE_Transformer_UNet(3, 2, 'learned', resnet_stages_num=4, with_decoder_pos='learned', enc_depth=1, dec_depth=8)
    net.load_state_dict(synth.synth_state_dict(levir_template, seed=3, style="default"))
    net = net.cuda().eval()
    x1, x2 = synth.synth_pair(4, 256, 256, seed=2, kind="uniform")
    gt = torch.randint(0, 2, (4, 256, 256), generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        y = net._engine.forward_pair(net, x1.cuda(), x2.cuda(), want_argmax=True)
    cm = confusion_matrix(net._engine.last_argmax, gt.cuda(), 2).cpu().numpy()
    ref = MO.confuse_matrix(2, [gt.numpy()], [y.argmax(1).cpu().numpy()])
    assert np.array_equal(cm, ref.astype(np.int64))
