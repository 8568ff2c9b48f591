"""N3 preparation: the key space enumerated by tools/build_latency_table.py is exactly the key set of the reference's
shipped lookup table (stored in tests/golden/latency_lookup_table.json), and every key parses into one of our operators."""
import pytest

from tests import helpers as H
from tools import build_latency_table as blt


def test_enumerated_keys_equal_the_reference_table():
    ref = set(H.load_json("latency_lookup_table.json"))
    ours = blt.table_keys()
    assert len(ours) == len(set(ours))
    assert set(ours) == ref, (sorted(ref - set(ours))[:5], sorted(set(ours) - ref)[:5])


def test_every_key_builds_one_of_our_operators():
    keys = blt.table_keys()
    kinds = set()
    for key in keys[::7] + keys[-40:]:
        module, shape = blt.build_module(key)
        assert shape[0] == 1 and len(shape) == 4
        kinds.add(type(module).__name__)
    assert {"ConvNorm", "BasicResidual1x", "BasicResidual_downup_1x", "BasicResidual2x", "BasicResidual_downup_2x",
            "FactorizedReduce", "FeatureFusion", "Head"} <= kinds
    with pytest.raises(ValueError):
        blt.build_module("Pooling_H1_W1")
