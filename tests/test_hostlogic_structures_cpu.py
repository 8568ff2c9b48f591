"""Wiring of the derived network for structures the shipped genotypes do not exercise -- three branches, a branch that ends
at 1/8 (its feature is copied straight into the fusion buffer), single-branch networks, eval and train builds -- on random
architectures: ours (CPU stand-in backend) against the UNMODIFIED reference network (CPU fp32) given the same state_dict and the
same input, through goldens (oracle/make_golden_fuzz.py, tests/golden/fuzz_forward.npz: the reference's outputs at fixed
sample positions, its full argmax map).  Random genotypes with random weights are badly conditioned (zoomed operators on 4x8
feature maps: the reference's own logits move by several % when it is merely run in torch fp16), so the gate is two-sided: our
deviation from the fp32 reference must not exceed 1.5 x the deviation of the reference run in fp16 -- a mis-wired branch or
concat offset produces O(1) errors and is far outside that band for the well-conditioned cases."""
import numpy as np
import pytest
import torch

from oracle import make_golden_decode as mk
from oracle import make_golden_fuzz as fz
from tests import cpu_backend
from tests import helpers as H


@pytest.fixture(scope="module")
def golden():
    return H.load_npz("fuzz_forward.npz")


@pytest.mark.parametrize("seed,lasts", fz.EVAL_CASES)
def test_eval_logits_match_the_reference_on_random_structures(golden, seed, lasts):
    from fasterseg_b200.model_seg import Network_Multi_Path_Infer
    cid = fz.case_id("eval", seed, lasts)
    ours = fz.build_derived(Network_Multi_Path_Infer, mk.draw_case(seed), lasts, False)
    assert fz.keys_digest(list(ours.state_dict())) == str(golden[cid + "/keys"])
    fz.init_weights(ours, seed)
    x = fz.input_frame(seed, 1)
    with torch.no_grad(), cpu_backend.installed():
        got = ours(x)
        labels = ours.predict_labels(x)
    assert tuple(got.shape) == tuple(golden[cid + ".0/shape"]) == (1, 19, 128, 256)
    err = fz.rel_err(fz.sample(got), golden[cid + ".0/want"].astype(np.float64))
    err16 = float(golden[cid + ".0/err16"])
    print("seed %d lasts %s: norm-wise rel err ours %.3e | reference in fp16 %.3e" % (seed, lasts, err, err16))
    assert err <= 1.5 * err16 + 2e-3
    agree = float((labels.long().numpy() == golden[cid + "/argmax"]).mean())
    assert agree >= float(golden[cid + "/agree16"]) - 0.02


@pytest.mark.parametrize("seed,lasts", fz.TRAIN_CASES)
def test_train_mode_auxiliary_heads_match_the_reference_on_random_structures(golden, seed, lasts):
    """Train-mode build (auxiliary 1/16 and 1/32 heads, model_seg.py:217-226,298-335) for `lasts` combinations the shipped
    genotypes do not cover: which features feed heads16 / heads32, in which order, and which predictions are None."""
    from fasterseg_b200.model_seg import Network_Multi_Path_Infer
    cid = fz.case_id("train", seed, lasts)
    ours = fz.build_derived(Network_Multi_Path_Infer, mk.draw_case(seed), lasts, True)
    assert fz.keys_digest(list(ours.state_dict())) == str(golden[cid + "/keys"])
    fz.init_weights(ours, seed)
    x = fz.input_frame(seed, 2)
    with torch.no_grad(), cpu_backend.installed():
        got = ours(x)
    assert len(got) == len(golden[cid + "/none"]) == 3
    for i, (name, g) in enumerate(zip(("pred8", "pred16", "pred32"), got)):
        assert (g is None) == bool(golden[cid + "/none"][i]), name
        if g is None:
            continue
        assert tuple(g.shape) == tuple(golden["%s.%d/shape" % (cid, i)])
        err = fz.rel_err(fz.sample(g), golden["%s.%d/want" % (cid, i)].astype(np.float64))
        err16 = float(golden["%s.%d/err16" % (cid, i)])
        print("seed %d lasts %s %s: ours %.3e | reference in fp16 %.3e" % (seed, lasts, name, err, err16))
        assert err <= 1.5 * err16 + 5e-3, name
