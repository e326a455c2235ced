"""The drop-in boundary against what the reference's REAL control flow computed and cached
(``tests/golden/dropin.json``, written by ``oracle/gen_golden.py``; the GPU launch is
emulated by tests/emu_device.py).

    ctg.einsum(eq, *arrays, implementation=cb.implementation())   interface.py -> Contractor
    cb.install(tree); tree.contract(arrays)                       core.py:3943 -> contraction_cores
    tree.contract_slice(arrays, i) / tree.contract_core(...)      core.py:3802-3823, 3723-3773

on BASELINE.json config 1 (10-tensor random einsum, bond 4) and its hyper-index variant,
plus sliced trees.  Trees are ``RecordedTree`` stand-ins of the reference's greedy trees;
the reference's node loop and slice loop are the oracle's ports of them."""

import numpy as np
import pytest

import cotengra_b200 as cb
from oracle import ctg_oracle as orc
from tests import emu_device
from tests.helpers import (RecordedTree, decode_ir, decode_sliced, load_json, load_npz, make_arrays,
                           rel_err)

RECS = load_json("dropin.json")
VALS = load_npz("dropin_values.npz")


@pytest.fixture()
def emu(monkeypatch):
    emu_device.install(monkeypatch)


def _config1(hyper):
    tag = f"config1_hyper{int(hyper)}"
    rec = RECS[tag]
    shapes = [tuple(rec["size_dict"][ix] for ix in t) for t in rec["inputs"]]
    return tag, rec, make_arrays(shapes, "complex128", seed=0)


@pytest.mark.parametrize("hyper", [False, True])
def test_einsum_with_b200_implementation(emu, hyper):
    """BASELINE config 1: the reference's node loop on numpy CPU arrays with
    ``implementation=cb.implementation()``, pairwise nodes through the product."""
    tag, rec, arrays = _config1(hyper)
    want = VALS[f"{tag}_einsum"]                          # ctg.einsum(eq, *arrays)
    before = emu_device.FakeLib.launches
    got = orc.run_contractions(decode_ir(rec["contractions"]), arrays,
                               implementation=cb.implementation())
    assert emu_device.FakeLib.launches - before >= 9      # every node went through the C-ABI call
    assert np.shape(got) == np.shape(want)
    assert rel_err(got, want) < 1e-12


@pytest.mark.parametrize("hyper", [False, True])
@pytest.mark.parametrize("strip", [False, True])
def test_install_routes_tree_contract(emu, hyper, strip):
    tag, rec, arrays = _config1(hyper)
    tree = RecordedTree(rec)
    fn = cb.install(tree, strip_exponent=strip)
    # the key tree.contract(arrays, strip_exponent=strip) looked up in the reference's cache
    key = next(tuple(k) for s, k in rec["contractor_keys"] if s == strip)
    assert tree.contraction_cores == {key: fn}
    before = emu_device.FakeLib.launches
    got = fn(*arrays)
    assert emu_device.FakeLib.launches > before
    if strip:
        got = got[0] * 10.0 ** got[1]
        want = VALS[f"{tag}_strip_m"] * 10.0 ** float(VALS[f"{tag}_strip_e"])
        assert rel_err(got, want) < 1e-12
    assert rel_err(got, VALS[f"{tag}_contract"]) < 1e-12


def test_install_on_a_sliced_tree(emu):
    _tag, _rec, arrays = _config1(True)
    rec = RECS["sliced"]
    tree = RecordedTree(rec)
    assert rec["nslices"] > 1
    want = VALS["sliced_contract"]
    fn = cb.install(tree)
    inputs, sliced = [tuple(t) for t in rec["inputs"]], decode_sliced(rec["sliced"])
    before = emu_device.FakeLib.launches
    # the reference's own slice loop + gather_slices around the product's contractor
    slices = [fn(*orc.slice_arrays(inputs, sliced, arrays, i)) for i in range(rec["nslices"])]
    got = orc.gather_slices(tuple(rec["output"]), sliced, slices)
    assert emu_device.FakeLib.launches > before
    assert rel_err(got, want) < 1e-12
    for i in (0, rec["nslices"] - 1):
        assert rel_err(slices[i], VALS[f"sliced_slice{i}"]) < 1e-12
    # whole-tree path of the product on the same tree (slice loop inside ctgb_plan_execute)
    assert rel_err(cb.contract_tree(tree, arrays), want) < 1e-12


def test_make_contractor_signature_matches_reference(emu):
    tag, rec, arrays = _config1(False)
    tree = RecordedTree(rec)
    fn = cb.make_contractor(tree)
    assert rel_err(fn(*arrays), VALS[f"{tag}_contract"]) < 1e-12
    m, e = fn(*arrays, strip_exponent=True, check_zero=True, backend=None)
    rm, re_ = VALS[f"{tag}_strip_m"], float(VALS[f"{tag}_strip_e"])
    assert rel_err(m * 10.0**e, rm * 10.0**re_) < 1e-12
    with pytest.raises(TypeError):
        fn(*arrays, nonsense=True)


def test_benchmark_flops_match_total_flops(emu):
    """ADVICE r1: cb.benchmark's flop count is tree.total_flops(dtype) (core.py:1196-1227),
    hoisted slice-invariant nodes included."""
    rec = RECS["lattice4x4"]
    total_flops = rec["total_flops_float64"]
    ex = cb.TreeExecutor(RecordedTree(rec), dtype="float64")
    macs_v, macs_i, _ = ex.reference_work
    assert macs_i > 0                                     # there are hoisted nodes
    assert 2 * (macs_v + macs_i) * rec["nslices"] == total_flops
    res = cb.benchmark(None, executor=ex, max_time=0.0, min_reps=1, max_reps=1, warmup=False)
    assert np.isclose(res["est_gigaflops"], total_flops / (1e9 * res["est_time_total"]))
