"""``TreeSpec`` regenerates the reference's contraction IR bit-exactly
(integer/string work: pinned to golden records from the unmodified reference)."""

import pytest

from cotengra_b200 import TreeSpec
from tests.helpers import RecordedTree, decode_ir, decode_sliced, load_json

TREES = load_json("trees.json") + load_json("sycamore_m20.json")


def _split(ir):
    pre = sorted(r for r in ir if r[1] is None and r[2] is None)
    rest = tuple(r for r in ir if not (r[1] is None and r[2] is None))
    return pre, rest


@pytest.mark.parametrize("rec", TREES, ids=[r["name"] for r in TREES])
def test_ir_matches_reference(rec):
    n_in = len(rec["inputs"])
    node_inds = {int(k): v for k, v in rec["inds"].items() if int(k) >= n_in}
    spec = TreeSpec(rec["inputs"], rec["output"], rec["size_dict"], rec["path"],
                    decode_sliced(rec["sliced"]), node_inds)
    if "_root" not in rec["name"] and "_flops" not in rec["name"]:
        # default index order is derivable from the path alone
        plain = TreeSpec(rec["inputs"], rec["output"], rec["size_dict"], rec["path"],
                         decode_sliced(rec["sliced"]))
        assert plain.contractions() == spec.contractions()
    got_pre, got = _split(spec.contractions())
    want_pre, want = _split(decode_ir(rec["contractions"]))
    # preprocessing steps are independent in-place ops: order is irrelevant
    assert got_pre == want_pre
    assert got == want
    for k, v in rec["inds"].items():
        if int(k) in spec.inds and n_in > 1:
            assert spec.inds[int(k)] == v, k
    assert spec.nslices == rec["nslices"]
    assert sorted(spec.sliced_inputs) == rec["sliced_inputs"]
    assert spec.slice_strides() == rec["slice_strides"]
    for i, key in rec["slice_keys"].items():
        assert spec.slice_key(int(i)) == key
    # JSON round trip
    again = TreeSpec.from_dict(spec.to_dict())
    assert again.contractions() == spec.contractions()


def test_live_reference_random_trees():
    """Freshly searched greedy trees of random equations (random index orders, slicing,
    removed indices), captured through ``TreeSpec.from_cotengra`` as the reference
    recorded them (``random_trees.json``), against the reference's own IR and slice keys."""
    for rec in load_json("random_trees.json"):
        spec = TreeSpec.from_cotengra(RecordedTree(rec))
        want_pre, want = _split(decode_ir(rec["contractions"]))
        got_pre, got = _split(spec.contractions())
        assert got == want and got_pre == want_pre, rec["name"]
        assert spec.nslices == rec["nslices"]
        for i, key in rec["slice_keys"].items():
            assert spec.slice_key(int(i)) == key, (rec["name"], i)
