"""Host logic of the boundary on the build machine: the REAL `fasterseg_b200` operator classes, networks and autograd
functions run on CPU tensors with the tensor-level wrappers of `fasterseg_b200.functional` swapped for the torch stand-ins of
tests/cpu_backend.py (test infrastructure; the product itself has no CPU path), and are compared with the same reference
goldens / oracle the GPU parity tests use.  What this pins without a GPU: which unit every operator calls and with which
channel slices (zero-copy concat offsets, FactorizedReduce's shifted second conv), the branch / cell sharing and the
arm-refine-fusion wiring of the derived network, MixedOp / beta aggregation and width sampling of the supernet, the autograd
graph of the training units (including accumulation of weight gradients straight into `param.grad` and the set of parameters
that must stay grad-less), running-statistic updates, and GRAD_SCALE bookkeeping."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import fasterseg_oracle as orc
from oracle import supernet_oracle as sno
from tests import cpu_backend
from tests import helpers as H
from tests.test_boundary_cpu import _build_student, _build_supernet
from tests.test_supernet_oracle import CASE, FWD, META, cfg, inputs, make_sd, oracle_loss_and_grads


@pytest.fixture(autouse=True)
def _cpu_backend():
    with cpu_backend.installed():
        yield


def _load_seeded(model, g, seed, key="state_dict_shapes"):
    full = {k: tuple(v) for k, v in g[key].items() if not k.endswith("num_batches_tracked")}
    sd = orc.random_state_dict(full, seed=seed)
    own = model.state_dict()
    seen = set()
    for k in sorted(sd):  # shared cells: first key wins (same rule as oracle/make_golden.py)
        if own[k].data_ptr() in seen:
            continue
        seen.add(own[k].data_ptr())
        own[k].copy_(sd[k])
    for m in model.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.eps, m.momentum = orc.BN_EPS, orc.BN_MOMENTUM
    return sd


@pytest.mark.parametrize("arch_idx,hw", [(1, (64, 128)), (0, (64, 128)), (1, (96, 160))])
def test_student_eval_wiring_vs_reference_golden(arch_idx, hw):
    z = H.load_npz("student.npz")
    model, g = _build_student(arch_idx)
    model = model.eval()
    _load_seeded(model, g, 2024 + arch_idx)
    x = orc.random_input((1, 3) + hw, seed=99 + arch_idx)
    with torch.no_grad():
        y = model(x)
        lab = model.predict_labels(x)
    assert y.dtype == torch.float32 and tuple(y.shape) == (1, 19) + hw and y.is_contiguous()
    tag = "arch%d.%dx%d.eval" % (arch_idx, hw[0], hw[1])
    yn = y.numpy()
    ref = z[tag + "/logits.s4"]
    nerr = H.rel_err(yn[:, :, ::4, ::4], ref)
    print(tag, "norm-wise rel err vs the reference (fp16-storage emulation on CPU): %.3e" % nerr)
    assert nerr < 3e-3
    assert (lab.numpy() == z[tag + "/argmax"]).mean() > 0.995
    assert np.array_equal(lab.numpy(), yn.argmax(1).astype(np.uint8))


def test_student_train_forward_and_running_stats_vs_reference_golden():
    z = H.load_npz("student.npz")
    model, g = _build_student(1, training=True)
    model = model.train()
    _load_seeded(model, g, 2025, key="state_dict_shapes_train")
    x = orc.random_input((2, 3, 192, 384), seed=100)
    with torch.no_grad():
        preds = model(x)
    tag = "arch1.192x384.train"
    for name, o in zip(("pred8", "pred16", "pred32"), preds):
        nerr = H.rel_err(o.float().numpy()[:, :, ::4, ::4], z[tag + "/" + name + ".s4"])
        print(tag, name, "%.3e" % nerr)
        assert nerr < 6e-2, name  # ill-conditioned train-mode chain, see tests/test_student_gpu.py
    sd = model.state_dict()
    for k in ("stem.0.conv.1.running_mean", "stem.0.conv.1.running_var", "heads8.conv_3x3.bn.running_var"):
        np.testing.assert_allclose(sd[k].numpy(), z[tag + "/after:" + k], rtol=3e-3, atol=3e-4)
    assert int(sd["stem.0.conv.1.num_batches_tracked"]) == 1


def test_student_train_step_autograd_wiring_vs_oracle():
    """forward + backward of the train-mode student through the real autograd Functions; gradients against CPU autograd
    through the fp16-storage-emulating oracle (same storage semantics -> tight) and the set of grad-less parameters."""
    model, g = _build_student(1, training=True)
    model = model.train()
    sd = _load_seeded(model, g, 31, key="state_dict_shapes_train")
    st, _ = H.student_structure(1)
    x = orc.random_input((2, 3, 96, 192), seed=32)
    tgt = [orc.random_input((2, 19, 96, 192), seed=33 + i) for i in range(3)]

    def run_oracle(emulate):
        orc.EMULATE_FP16["on"] = emulate
        try:
            sd_ref = {k: v.clone().requires_grad_(not ("running" in k)) for k, v in sd.items()}
            outs = orc.student_forward(x, sd_ref, st, training=True)
            sum((o * t).mean() for o, t in zip(outs, tgt)).backward()
        finally:
            orc.EMULATE_FP16["on"] = False
        return {k: v.grad.numpy() for k, v in sd_ref.items() if v.grad is not None}

    g32, g16 = run_oracle(False), run_oracle(True)
    outs = model(x)
    sum((o * t).mean() for o, t in zip(outs, tgt)).backward()
    e_ours, e_emu = [], []
    for k, p in model.named_parameters():
        if k not in g32 or np.linalg.norm(g32[k]) < 1e-12:
            continue
        assert p.grad is not None and p.grad.dtype == torch.float32 and p.grad.shape == p.shape, k
        e_ours.append(H.rel_err(p.grad.numpy(), g32[k]))
        e_emu.append(H.rel_err(g16[k], g32[k]))
    med_ours, med_emu = float(np.median(e_ours)), float(np.median(e_emu))
    print("checked %d gradients: median err vs fp32 oracle ours %.3e | fp16-emulating oracle %.3e" % (len(e_ours), med_ours, med_emu))
    assert len(e_ours) > 100
    assert med_ours <= 1.5 * med_emu + 1e-2
    assert max(e_ours) <= 4.0 * max(max(e_emu), med_emu) + 5e-2
    no_grad_ours = {k for k, p in model.named_parameters() if p.grad is None}
    no_grad_ref = {k for k in dict(model.named_parameters()) if k not in g32}
    assert no_grad_ours == no_grad_ref, sorted(no_grad_ours ^ no_grad_ref)


@pytest.mark.parametrize("tag,arch_idx,mode,train,np_seed,torch_seed", FWD)
def test_supernet_forward_wiring_vs_reference_golden(tag, arch_idx, mode, train, np_seed, torch_seed):
    z = H.load_npz("supernet.npz")
    model = _build_supernet(CASE["layers"])
    own = model.state_dict()
    for k, v in make_sd().items():
        own[k].copy_(v)
    for m in model.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.eps, m.momentum = orc.BN_EPS, orc.BN_MOMENTUM
    model.train(train)
    x, _ = inputs()
    if np_seed is not None:
        np.random.seed(np_seed)
    if torch_seed is not None:
        torch.manual_seed(torch_seed)
    model.arch_idx, model.prun_mode = arch_idx, mode
    with torch.no_grad():
        preds = model(x)
    worst = 0.0
    for i, p in enumerate(preds):
        assert p.dtype == torch.float32 and p.is_contiguous()
        ref = z["%s/pred%d" % (tag, i)]
        got = p.numpy() if train else p.numpy()[:, :, ::8, ::8]
        worst = max(worst, H.rel_err(got, ref))
    print("%s: worst norm-wise rel err over the 5 logits %.3e" % (tag, worst))
    assert worst < (5e-3 if not train else 5e-2)
    if train:
        sd = model.state_dict()
        for k in z.files:
            if k.startswith(tag + "/after:"):
                np.testing.assert_allclose(sd[k.split("after:")[1]].numpy(), z[k], rtol=2e-2, atol=2e-3)


@pytest.mark.parametrize("tag,pretrain,np_seed,torch_seed", [("loss.pretrain", True, 11, 12), ("loss.search", "some-dir", 13, 14)])
def test_supernet_loss_backward_wiring(tag, pretrain, np_seed, torch_seed):
    """`_loss` (4 forwards) + backward through WsumFn / ConvBnActFn / FactorizedReduceFn / CatFn / ToNCHWFn on CPU: the loss,
    the set of parameters that receive no gradient, and the gradients against the fp32 oracle within the fp16-storage band."""
    x, tgt = inputs()
    crit = nn.CrossEntropyLoss(ignore_index=255)

    def run_oracle(emulate):
        loss, sd = oracle_loss_and_grads(pretrain, np_seed, torch_seed, emulate)
        return float(loss), {k: v.grad.numpy() for k, v in sd.items() if v.requires_grad and v.grad is not None}

    l32, g32 = run_oracle(False)
    l16, g16 = run_oracle(True)
    model = _build_supernet(CASE["layers"])
    own = model.state_dict()
    for k, v in make_sd().items():
        own[k].copy_(v)
    for m in model.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.eps, m.momentum = orc.BN_EPS, orc.BN_MOMENTUM
    model.train(True)
    np.random.seed(np_seed)
    torch.manual_seed(torch_seed)
    loss = model._loss(x, tgt, pretrain)
    loss.backward()
    lo = float(loss.detach())
    print("%s: loss ours(CPU stand-in) %.5f | fp32 oracle %.5f | fp16-emulating oracle %.5f" % (tag, lo, l32, l16))
    assert abs(lo - l32) <= 1.5 * abs(l16 - l32) + 2e-3 * abs(l32)
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert sorted(k for k, g in grads.items() if g is None) == sorted(k for k in grads if k not in g32)
    assert len([k for k, g in grads.items() if g is None]) == META[tag + ".no_grad_count"]
    e_ours, e_emu = [], []
    for k, g in grads.items():
        if g is None or np.linalg.norm(g32[k]) < 1e-10 or k.startswith("ratio_"):
            continue  # ratio_*: pure cancellation noise, see tests/test_supernet_gpu.py
        e_ours.append(H.rel_err(g.float().numpy(), g32[k]))
        e_emu.append(H.rel_err(g16[k], g32[k]))
    med_ours, med_emu = float(np.median(e_ours)), float(np.median(e_emu))
    print("%s: %d gradients, median err vs fp32 oracle ours %.3e | emulation %.3e" % (tag, len(e_ours), med_ours, med_emu))
    assert len(e_ours) > 300
    assert med_ours <= 1.5 * med_emu + 1e-2


def test_weight_and_bn_caches_follow_parameter_updates():
    """Packed-weight / folded-BN caches are keyed by the tensors' version counters and storage: an optimizer step, an
    in-place edit, a `.data` swap and `load_state_dict` must all be visible to the next forward (train/train.py:262-264
    steps the optimizer between forwards; train_search.py:73 loads checkpoints partially)."""
    model, g = _build_student(1)
    model = model.eval()
    _load_seeded(model, g, 2024)
    x = orc.random_input((1, 3, 64, 128), seed=5)

    def fresh_output():
        twin, _ = _build_student(1)
        twin = twin.eval()
        twin.load_state_dict(model.state_dict())
        for a, b in zip(model.modules(), twin.modules()):
            if isinstance(a, nn.BatchNorm2d):
                b.eps, b.momentum = a.eps, a.momentum
        with torch.no_grad():
            return twin(x)

    with torch.no_grad():
        y0 = model(x)
        assert torch.equal(y0, fresh_output())
        # 1. optimizer-style in-place update of every parameter
        opt = torch.optim.SGD(model.parameters(), lr=0.05)
        for p in model.parameters():
            p.grad = torch.ones_like(p) * 0.01
        opt.step()
        y1 = model(x)
        assert not torch.equal(y1, y0) and torch.equal(y1, fresh_output())
        # 2. running statistics edited in place (BN fold cache), one conv weight replaced through .data
        model.stem[1].bn1.running_var.mul_(1.5)
        model.heads8.conv_3x3.conv.weight.data = model.heads8.conv_3x3.conv.weight.data * 0.9
        y2 = model(x)
        assert not torch.equal(y2, y1) and torch.equal(y2, fresh_output())
        # 3. load_state_dict back to the original weights reproduces the original output bit for bit
        _load_seeded(model, g, 2024)
        assert torch.equal(model(x), y0)


def test_uint8_frame_path_matches_normalised_fp32_path_and_gpu_free_metrics():
    """Evaluator path (N4): feeding the uint8 HWC image + set_input_normalization must give the labels of feeding
    normalize(img) as fp32 CHW (tools/engine/evaluator.py:329); the device confusion matrix must equal metric.hist_info."""
    from fasterseg_b200 import metric
    model, g = _build_student(1)
    model = model.eval()
    _load_seeded(model, g, 77)
    rs = np.random.RandomState(3)
    img = rs.randint(0, 256, size=(1, 64, 128, 3)).astype(np.uint8)
    mean, std = np.array([0.485, 0.456, 0.406]), np.array([0.229, 0.224, 0.225])
    ref_in = ((img.astype(np.float32) / 255.0 - mean) / std).astype(np.float32).transpose(0, 3, 1, 2)      # img_utils.normalize
    model.set_input_normalization(mean, std)
    with torch.no_grad():
        lab_u8 = model.predict_labels(torch.from_numpy(img).permute(0, 3, 1, 2))
        lab_f32 = model.predict_labels(torch.from_numpy(np.ascontiguousarray(ref_in)))
    assert torch.equal(lab_u8, lab_f32)
    gt = torch.from_numpy(rs.randint(0, 19, size=(1, 64, 128)).astype(np.int64))
    gt[0, :5] = 255
    hist, labeled, correct = metric.hist_info(19, lab_u8, gt)
    p, t = lab_u8.numpy(), gt.numpy()
    k = (t >= 0) & (t < 19)
    want = np.bincount(19 * t[k].astype(int) + p[k].astype(int), minlength=19 ** 2).reshape(19, 19)
    assert np.array_equal(hist, want) and labeled == int(k.sum()) and correct == int((p[k] == t[k]).sum())
    iu, miou, _, acc = metric.compute_score(hist, correct, labeled)
    assert 0 <= acc <= 1 and iu.shape == (19,)


# ---------------------------------------------------------------------------------------------------------------------------
# evaluator path (N4) pinned to the reference's own metric / normalisation code (tests/golden/metric.json, oracle/make_golden_metric.py)
# ---------------------------------------------------------------------------------------------------------------------------
def _same_or_both_nan(a, b, tol=1e-12):
    if b is None:
        return a is None or (isinstance(a, float) and np.isnan(a))
    return abs(float(a) - float(b)) <= tol * max(1.0, abs(float(b)))


@pytest.mark.parametrize("name", sorted(H.load_json("metric.json")["metric"]))
def test_device_confusion_matrix_and_scores_match_the_reference_goldens(name):
    """fasterseg_b200/metric.py against tools/seg_opr/metric.py:7-27 run unmodified (goldens): the confusion matrix, labeled / correct
    counts (ignore label 255 and negative labels), per-class IoU with absent classes (nan), mean IoU with / without class 0, pixel
    accuracy -- one image at a time through `ConfusionMatrix.update`, as the evaluator accumulates them."""
    from fasterseg_b200 import metric
    from oracle import make_golden_metric as mk
    want = H.load_json("metric.json")["metric"][name]
    n_cl, pred, gt = mk.metric_inputs(name)
    hist, labeled, correct = metric.hist_info(n_cl, torch.from_numpy(pred), torch.from_numpy(gt))
    assert hist.dtype == np.int64 and hist.tolist() == want["hist"] and labeled == want["labeled"] and correct == want["correct"]
    cm = metric.ConfusionMatrix(n_cl, device="cpu")
    for i in range(pred.shape[0]):
        cm.update(torch.from_numpy(pred[i]), torch.from_numpy(gt[i]))
    h2, l2, c2 = cm.result()
    assert h2.tolist() == want["hist"] and (l2, c2) == (labeled, correct)
    iu, miou, miou_nb, acc = metric.compute_score(hist, correct, labeled)
    assert len(iu) == n_cl and all(_same_or_both_nan(float(a), b) for a, b in zip(iu, want["iu"]))
    assert _same_or_both_nan(float(miou), want["mean_IU"]) and _same_or_both_nan(float(miou_nb), want["mean_IU_no_back"])
    assert _same_or_both_nan(float(acc), want["mean_pixel_acc"])


@pytest.mark.parametrize("name", sorted(H.load_json("metric.json")["normalize"]))
def test_normalisation_table_matches_the_reference_normalize(name):
    """the 3 x 256 table the stem kernel gathers through (functional.normalization_lut) holds, for every byte value, the fp16 rounding
    of what tools/utils/img_utils.py:179-185 makes of that byte (goldens: sum / head / tail of the reference's normalised frames)"""
    from fasterseg_b200 import functional as F_
    from oracle import make_golden_metric as mk
    want = H.load_json("metric.json")["normalize"][name]
    img, mean, std = mk.normalize_inputs(name)
    lut = F_.normalization_lut(mean, std, "cpu")
    assert lut.dtype == torch.float16 and tuple(lut.shape) == (3, 256)
    exact = np.stack([((np.arange(256, dtype=np.uint8).astype(np.float32) / 255.0) - mean[c]) / std[c] for c in range(3)]).astype(np.float32)
    assert torch.equal(lut, torch.from_numpy(exact).half())
    frame = np.stack([exact[c][img[..., c]] for c in range(3)], axis=-1)          # gather, like the kernel; HWC fp32 before the fp16 rounding
    assert abs(float(frame.astype(np.float64).sum()) - want["sum"]) <= 1e-6 * max(1.0, abs(want["sum"]))
    np.testing.assert_allclose(frame.reshape(-1)[:12], np.array(want["first"], dtype=np.float32), rtol=0, atol=0)
    np.testing.assert_allclose(frame.reshape(-1)[-12:], np.array(want["last"], dtype=np.float32), rtol=0, atol=0)
