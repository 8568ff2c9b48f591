"""Supernet wiring with RANDOM architecture parameters (the goldens use the constant 1e-3 initialisation): MixedOp weights,
beta mixing of the two cell invocations, width selection in every mode incl. gumbel-sampled `arch_ratio`, for several
depths -- ours on the CPU stand-in backend against the UNMODIFIED reference (CPU fp32) given the same state_dict and the same
RNG seeds, through goldens (oracle/make_golden_fuzz.py, tests/golden/fuzz_forward.npz), with a two-sided gate against the
reference run in torch fp16 (random supernets are ill-conditioned, see tests/test_hostlogic_structures_cpu.py)."""
import numpy as np
import pytest

from oracle import make_golden_fuzz as fz
from oracle import make_golden_latency as mkl
from tests import cpu_backend
from tests import helpers as H


@pytest.fixture(scope="module")
def golden():
    return H.load_npz("fuzz_forward.npz")


@pytest.mark.parametrize("layers,arch_idx,mode,seed", fz.SUPERNET_CASES)
def test_eval_forward_matches_reference_with_random_arch_parameters(golden, layers, arch_idx, mode, seed):
    from fasterseg_b200.model_search import Network_Multi_Path
    cid = fz.case_id("supernet", layers, arch_idx, mode, seed)
    ours = mkl.build(Network_Multi_Path, layers).eval()
    assert fz.keys_digest([k for k, _ in ours.named_parameters()]) == str(golden[cid + "/keys"])
    mkl.randomise_arch(ours, 900 + seed)
    fz.init_weights(ours, seed)
    with cpu_backend.installed():
        got = fz.run_supernet(ours, fz.input_frame(seed, 1), arch_idx, mode, seed)
    assert len(got) == 5
    for i, g in enumerate(got):
        assert tuple(g.shape) == tuple(golden["%s.%d/shape" % (cid, i)])
        err = fz.rel_err(fz.sample(g), golden["%s.%d/want" % (cid, i)].astype(np.float64))
        err16 = float(golden["%s.%d/err16" % (cid, i)])
        print("layers %d arch %d mode %s pred%d: ours %.3e | reference in fp16 %.3e" % (layers, arch_idx, mode, i, err, err16))
        assert err <= 1.5 * err16 + 3e-3, i
