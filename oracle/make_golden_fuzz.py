#!/usr/bin/env python
"""TEST INFRASTRUCTURE ONLY -- goldens of the random-structure tests (tests/test_hostlogic_structures_cpu.py: derived networks of
random genotypes, eval and train builds; tests/test_hostlogic_supernet_fuzz_cpu.py: supernets with random architecture
parameters).  The UNMODIFIED reference network gets the weights `init_weights` draws for OUR network of the same structure (the
state_dicts must agree key for key) and the input `input_frame` draws; it is run in fp32 and, for the two-sided gate of the tests,
once more in torch fp16.  Stored per output: the fp32 values at `SAMPLES` fixed positions (`sample`) and the deviation of the fp16
run from the fp32 run on those positions; for the eval builds also the full fp32 argmax map and the fp16 run's agreement with it.
Written to tests/golden/fuzz_forward.npz.  Run where the reference tree is available:  python oracle/make_golden_fuzz.py"""
import copy
import hashlib
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import make_golden_decode as mkd  # noqa: E402
from oracle import make_golden_latency as mkl  # noqa: E402

SAMPLES = 256
EVAL_CASES = [(1003, [0, 1, 2]), (1010, [2, 0]), (1017, [1]), (1024, [0]), (1031, [1, 0]), (1038, [2]), (1045, [2, 1])]
TRAIN_CASES = [(1003, [0, 1, 2]), (1010, [2, 0]), (1017, [1]), (1045, [2, 1]), (1052, [1, 2])]
SUPERNET_CASES = [(5, 0, "max", 1), (5, 1, None, 2), (6, 1, "min", 3), (8, 1, None, 4), (8, 0, "random", 5)]
PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "fuzz_forward.npz")


def init_weights(model, seed):
    """Variance-preserving conv weights (torch's default init shrinks the signal into fp16 subnormals over 40 layers) and
    non-trivial BatchNorm statistics / affine, like a trained net; drawn per state_dict entry in order, architecture
    parameters left alone."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, v in model.state_dict().items():
            if name.endswith("num_batches_tracked") or name.split("_")[0] in ("alpha", "beta", "ratio"):
                continue
            if v.dim() == 4:
                v.copy_(torch.randn(v.shape, generator=g) * (2.0 / v[0].numel()) ** 0.5)
            elif name.endswith("running_mean"):
                v.copy_(0.1 * torch.randn(v.shape, generator=g))
            elif name.endswith("running_var"):
                v.copy_(0.5 + torch.rand(v.shape, generator=g))
            elif name.endswith("weight"):
                v.copy_(1.0 + 0.1 * torch.randn(v.shape, generator=g))
            else:
                v.copy_(0.1 * torch.randn(v.shape, generator=g))


def input_frame(seed, n):
    return torch.randn(n, 3, 128, 256, generator=torch.Generator().manual_seed(seed))


def keys_digest(names):
    return hashlib.sha256("\n".join(names).encode()).hexdigest()[:16]


def sample(t):
    """the values at SAMPLES fixed positions of an output (the same positions for every output of that size), float64"""
    flat = t.detach().float().reshape(-1)
    idx = np.sort(np.random.RandomState(flat.numel() % (2 ** 31)).choice(flat.numel(), min(SAMPLES, flat.numel()), replace=False))
    return flat[torch.from_numpy(idx)].double().numpy()


def rel_err(got, want):
    return float(np.linalg.norm(got - want) / np.linalg.norm(want))


def build_derived(Net, case, lasts, training):
    alphas, betas, ratios = mkd.clone_params(case)
    m = Net(alphas, betas, ratios, num_classes=19, layers=case["layers"], Fch=12, width_mult_list=mkd.WML,
            stem_head_width=case["stem_head_width"], ignore_skip=case["ignore_skip"])
    m.train(training)
    m.build_structure(list(lasts))
    return m


def run_supernet(model, inp, arch_idx, mode, seed):
    model.arch_idx, model.prun_mode = arch_idx, mode
    np.random.seed(seed)           # 'random' widths
    torch.manual_seed(100 + seed)  # gumbel noise of 'arch_ratio'
    with torch.no_grad():
        return model(inp)


def case_id(kind, *params):
    return ".".join([kind] + ["".join(map(str, p)) if isinstance(p, list) else str(p) for p in params])


def _record(out, cid, preds, preds16):
    for i, (w, h) in enumerate(zip(preds, preds16)):
        if w is None:
            continue
        out["%s.%d/shape" % (cid, i)] = np.array(w.shape, dtype=np.int64)
        out["%s.%d/want" % (cid, i)] = sample(w).astype(np.float32)
        out["%s.%d/err16" % (cid, i)] = np.array(rel_err(sample(h), sample(w)))


def main():
    from fasterseg_b200.model_search import Network_Multi_Path
    from fasterseg_b200.model_seg import Network_Multi_Path_Infer
    from oracle import ref_harness
    ref_seg = ref_harness.load_reference("train", "model_seg").model_seg.Network_Multi_Path_Infer
    ref_search = ref_harness.load_reference("search", "slimmable_ops", "operations", "seg_oprs", "genotypes",
                                            "model_search").model_search.Network_Multi_Path
    out = {}
    for seed, lasts in EVAL_CASES:
        cid = case_id("eval", seed, lasts)
        case = mkd.draw_case(seed)
        ours = build_derived(Network_Multi_Path_Infer, case, lasts, False)
        init_weights(ours, seed)
        ref = build_derived(ref_seg, case, lasts, False)
        ref.load_state_dict(ours.state_dict())
        out[cid + "/keys"] = np.array(keys_digest(list(ref.state_dict())))
        x = input_frame(seed, 1)
        with torch.no_grad():
            want = ref(x)
            half = copy.deepcopy(ref).half()(x.half()).float()
        _record(out, cid, [want], [half])
        out[cid + "/argmax"] = want.argmax(1).numpy().astype(np.uint8)
        out[cid + "/agree16"] = np.array(float((half.argmax(1) == want.argmax(1)).float().mean()))
        print(cid, "fp16 deviation %.3e" % float(out[cid + ".0/err16"]))
    for seed, lasts in TRAIN_CASES:
        cid = case_id("train", seed, lasts)
        case = mkd.draw_case(seed)
        ours = build_derived(Network_Multi_Path_Infer, case, lasts, True)
        init_weights(ours, seed)
        ref = build_derived(ref_seg, case, lasts, True)
        ref.load_state_dict(ours.state_dict())
        out[cid + "/keys"] = np.array(keys_digest(list(ref.state_dict())))
        half = copy.deepcopy(ref).half()
        x = input_frame(seed, 2)
        with torch.no_grad():
            want = ref(x)
            got16 = half(x.half())
        out[cid + "/none"] = np.array([w is None for w in want])
        _record(out, cid, want, got16)
        print(cid, "predictions present", [w is not None for w in want])
    for layers, arch_idx, mode, seed in SUPERNET_CASES:
        cid = case_id("supernet", layers, arch_idx, mode, seed)
        ours = mkl.build(Network_Multi_Path, layers).eval()
        mkl.randomise_arch(ours, 900 + seed)
        init_weights(ours, seed)
        ref = mkl.build(ref_search, layers).eval()
        ref.load_state_dict(ours.state_dict())
        out[cid + "/keys"] = np.array(keys_digest([k for k, _ in ref.named_parameters()]))
        half = copy.deepcopy(ref).half()
        x = input_frame(seed, 1)
        want = run_supernet(ref, x, arch_idx, mode, seed)
        got16 = run_supernet(half, x.half(), arch_idx, mode, seed)
        _record(out, cid, want, got16)
        print(cid, "fp16 deviation", ["%.3e" % float(out["%s.%d/err16" % (cid, i)]) for i in range(len(want))])
    np.savez_compressed(PATH, **out)
    print("wrote", PATH, os.path.getsize(PATH) // 1024, "KiB")


if __name__ == "__main__":
    main()
