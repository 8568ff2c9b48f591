"""CPU checks of the reference-facing Python boundary: class/attribute/state_dict parity with the reference
(from golden metadata), decoder KATs and latency-table KAT.  No kernels are launched."""
import numpy as np
import pytest
import torch

from tests import helpers as H


def _build_student(arch_idx, training=False, lasts=None):
    from fasterseg_b200.model_seg import Network_Multi_Path_Infer
    g = H.load_json("genotypes.json")["arch_%d" % arch_idx]
    a = g["arch"]
    t = lambda k: torch.tensor(a[k], dtype=torch.float32)
    model = Network_Multi_Path_Infer(
        [t("alpha_%d_%d" % (arch_idx, s)) for s in range(3)],
        [None, t("beta_%d_1" % arch_idx), t("beta_%d_2" % arch_idx)],
        [t("ratio_%d_%d" % (arch_idx, s)) for s in range(3)],
        num_classes=19, layers=16, Fch=12, width_mult_list=[4. / 12, 6. / 12, 8. / 12, 10. / 12, 1.],
        stem_head_width=(1., 1.) if arch_idx == 0 else (8. / 12, 8. / 12), ignore_skip=(arch_idx == 0))
    model.train(training)
    model.build_structure(lasts if lasts is not None else g["lasts"])
    return model, g


@pytest.mark.parametrize("arch_idx", [0, 1])
def test_student_state_dict_matches_reference(arch_idx):
    model, g = _build_student(arch_idx)
    sd = model.state_dict()
    assert {k: list(v.shape) for k, v in sd.items()} == g["state_dict_shapes"]
    for last in (0, 1, 2):
        r = g["decoded"][str(last)]
        assert [int(o) for o in getattr(model, "ops%d" % last)] == r["ops"]
        assert list(getattr(model, "path%d" % last)) == r["path"]
        assert list(getattr(model, "downs%d" % last)) == r["downs"]
        assert np.allclose(getattr(model, "widths%d" % last), r["widths"])
    assert model.branch_groups == g["branch_groups"]
    assert (model.ch_16, model.ch_8_2, model.ch_8_1) == (g["ch_16"], g["ch_8_2"], g["ch_8_1"])
    for k, (ci, co, down, cls) in g["cells"].items():
        c = model.cells[k]
        assert (c._C_in, c._C_out, int(bool(c._down)), type(c._op._op).__name__) == (ci, co, down, cls)
    assert sum(p.numel() for p in model.parameters()) == g["param_count_eval_build"]


def test_student_train_build_state_dict():
    model, g = _build_student(1, training=True)
    assert {k: list(v.shape) for k, v in model.state_dict().items()} == g["state_dict_shapes_train"]


def test_forward_latency_kat(tmp_path, monkeypatch):
    """latency12 / latency02 stored in arch_1.pt are reproduced from the reference's lookup table
    (SURVEY section 4 KAT ii; the table's data is stored in tests/golden/latency_lookup_table.json)."""
    from fasterseg_b200 import operations, seg_oprs  # noqa: F401
    monkeypatch.setattr(operations, "latency_lookup_table", H.load_json("latency_lookup_table.json"))
    g = H.load_json("genotypes.json")["arch_1"]
    model, _ = _build_student(1)
    lat, size = model.forward_latency((3, 1024, 2048))
    assert abs(lat - g["arch"]["latency12"]) < 1e-9 and tuple(size) == (19, 128, 256)
    assert abs(lat - g["forward_latency_1024x2048"][0]) < 1e-12
    model2, _ = _build_student(1, lasts=[2, 0])
    lat2, _ = model2.forward_latency((3, 1024, 2048))
    assert abs(lat2 - g["arch"]["latency02"]) < 1e-9


def test_op_classes_state_dict_and_api():
    from fasterseg_b200 import operations as ops
    metas = H.load_json("ops_meta.json")
    wml = [4. / 12, 6. / 12, 8. / 12, 10. / 12, 1.]
    assert ops.__all__ == ['ConvNorm', 'BasicResidual1x', 'BasicResidual_downup_1x', 'BasicResidual2x',
                           'BasicResidual_downup_2x', 'FactorizedReduce', 'OPS', 'OPS_name', 'OPS_Class']
    assert list(ops.OPS) == ['skip', 'conv', 'conv_downup', 'conv_2x', 'conv_2x_downup']
    assert [c.__name__ for c in ops.OPS_Class.values()] == ops.OPS_name
    for name, m in metas.items():
        cls = m["cls"]
        if cls in ("Head", "FeatureFusion"):
            continue
        if cls == "ConvNorm":
            mod = ops.ConvNorm(m["C_in"], m["C_out"], kernel_size=m["kernel_size"], stride=m["stride"],
                               slimmable=m["slimmable"], width_mult_list=wml)
        elif cls == "FactorizedReduce":
            mod = ops.FactorizedReduce(m["C_in"], m["C_out"], m["stride"], m["slimmable"], wml)
        else:
            mod = getattr(ops, cls)(m["C_in"], m["C_out"], 3, m["stride"], 1, 1, m["slimmable"], wml)
        got = {k: list(v.shape) for k, v in mod.state_dict().items() if not k.endswith("num_batches_tracked")}
        assert got == m["shapes"], name
        assert (mod.C_in, mod.C_out, mod.stride, mod.slimmable) == (m["C_in"], m["C_out"], m["stride"], m["slimmable"])
        if m["slimmable"]:
            mod.set_ratio(tuple(m["ratio"]))
            assert tuple(mod.ratio) == tuple(m["ratio"])
    import torch.nn as nn
    from fasterseg_b200.slimmable_ops import USBatchNorm2d, USConv2d
    assert issubclass(USConv2d, nn.Conv2d) and issubclass(USBatchNorm2d, nn.BatchNorm2d)


def _build_supernet(layers):
    import torch.nn as nn
    from fasterseg_b200.model_search import Network_Multi_Path
    return Network_Multi_Path(19, layers, nn.CrossEntropyLoss(ignore_index=255), Fch=12,
                              width_mult_list=[4. / 12, 6. / 12, 8. / 12, 10. / 12, 1.], prun_modes=['max', 'arch_ratio'],
                              stem_head_width=[(1, 1), (8. / 12, 8. / 12)])


def test_supernet_state_dict_and_parameter_order_match_reference():
    meta = H.load_json("supernet_meta.json")
    m = _build_supernet(meta["case"]["layers"])
    got = {k: list(v.shape) for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    assert got == meta["shapes"]
    assert [k for k, _ in m.named_parameters()] == meta["param_order"]
    assert len(m._arch_parameters) == 2 and len(m._arch_parameters[0]) == 8
    assert m._arch_names[1]["ratios"] == ["ratio_1_0", "ratio_1_1", "ratio_1_2"]
    # teacher ('max') has a single width choice, the student ('arch_ratio') five (model_search.py:522-529)
    assert tuple(m.ratio_0_0.shape) == (meta["case"]["layers"] - 1, 1) and tuple(m.ratio_1_2.shape) == (meta["case"]["layers"] - 2, 5)


def test_launcher_shadows_reference_module_names():
    """`from operations import *` / `from model_search import Network_Multi_Path` in the unmodified drivers must resolve to
    our modules (fasterseg_b200/launch.py)."""
    import importlib
    import sys
    from fasterseg_b200 import launch
    saved = {n: sys.modules.get(n) for n in launch.SHADOWED}
    try:
        launch.install_compat_patches()
        launch.install_shadow_modules()
        ops = importlib.import_module("operations")
        ms = importlib.import_module("model_search")
        mseg = importlib.import_module("model_seg")
        assert ops.__name__ == "fasterseg_b200.operations" and hasattr(ops, "OPS")
        assert ms.Network_Multi_Path.__module__ == "fasterseg_b200.model_search"
        assert mseg.Network_Multi_Path_Infer.__module__ == "fasterseg_b200.model_seg"
        ns = {}
        exec("from operations import *\nfrom slimmable_ops import USConv2d, USBatchNorm2d\nfrom seg_oprs import Head, FeatureFusion\n"
             "from genotypes import PRIMITIVES", ns)
        assert set(ops.__all__) <= set(ns) and ns["PRIMITIVES"][0] == "skip"
    finally:
        for n, m in saved.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m


def test_reference_citations_point_into_the_reference_tree():
    """docstrings, the header and the docs cite the reference as `dir/file.py:LINE[-LINE]`; every one must name an existing reference
    file and lines inside it (tools/check_citations.py, against the reference's line counts in tests/golden/reference_line_counts.json)
    -- a stale citation sends the parity reviewer to the wrong place"""
    from tools import check_citations
    bad, total = check_citations.stale(H.load_json("reference_line_counts.json"))
    assert total > 300 and not bad, bad[:10]
