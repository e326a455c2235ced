"""Generate the golden vectors under ``tests/golden/`` from the UNMODIFIED
reference (jcmgray/cotengra at ``/root/reference``), imported in the build
container through the numpy-only ``autoray`` stand-in in ``oracle/refshim``.

Run (build container only; the GPU box has no ``/root/reference``):

    python oracle/gen_golden.py

Everything written here is *data*: equations, shapes, the reference's own
planner outputs (``_parse_eq_to_batch_matmul`` etc.), its linear contraction
IR (``extract_contractions``), slice keys, and numerical results of the
reference's numpy path on seeded inputs (``tests/helpers.make_arrays``).
No reference source is copied.
"""

import json
import os
import random
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(HERE, "refshim"), "/root/reference"]

import numpy as np  # noqa: E402

import cotengra as ctg  # noqa: E402
from cotengra import contract as refc  # noqa: E402  (module, not the alias)

refc = sys.modules["cotengra.contract"]

from tests.helpers import GOLDEN_DIR, make_arrays  # noqa: E402

os.makedirs(GOLDEN_DIR, exist_ok=True)


def jsonable(x):
    if isinstance(x, (tuple, list)):
        return [jsonable(v) for v in x]
    if isinstance(x, (np.integer,)):
        return int(x)
    if isinstance(x, slice):
        return "slice"
    if isinstance(x, range):
        return list(x)
    return x


def enc_prep(e):
    """eq_a / eq_b entry of a plan: None | str | tuple(perm)."""
    if isinstance(e, tuple):
        return {"perm": list(e)}
    return e


def enc_plan(plan):
    eq_a, eq_b, na, nb, nab, perm, pure = plan
    return {
        "eq_a": enc_prep(eq_a),
        "eq_b": enc_prep(eq_b),
        "new_shape_a": jsonable(na),
        "new_shape_b": jsonable(nb),
        "new_shape_ab": jsonable(nab),
        "perm_ab": jsonable(perm),
        "pure": bool(pure),
    }


# --------------------------------------------------------------------------
# 1. parser vectors
# --------------------------------------------------------------------------


def random_pair_case(rng):
    letters = "abcdefghij"
    n_ix = rng.randint(1, 7)
    pool = rng.sample(letters, n_ix)
    sizes = {c: rng.choice([1, 2, 2, 3, 4]) for c in pool}
    la = rng.randint(0, min(4, n_ix))
    lb = rng.randint(0, min(4, n_ix))
    ta = [rng.choice(pool) for _ in range(la)]
    tb = [rng.choice(pool) for _ in range(lb)]
    if rng.random() < 0.7:
        # make repeated indices rarer
        ta = list(dict.fromkeys(ta))
        tb = list(dict.fromkeys(tb))
    present = list(dict.fromkeys(ta + tb))
    out = [c for c in present if rng.random() < 0.5]
    rng.shuffle(out)
    sa = [sizes[c] for c in ta]
    sb = [sizes[c] for c in tb]
    # broadcasting: occasionally collapse one side's extent to 1
    if rng.random() < 0.2 and ta:
        k = rng.randrange(len(ta))
        if ta.count(ta[k]) == 1:
            sa[k] = 1
    if rng.random() < 0.2 and tb:
        k = rng.randrange(len(tb))
        if tb.count(tb[k]) == 1:
            sb[k] = 1
    # occasionally a genuine mismatch
    if rng.random() < 0.04 and tb:
        k = rng.randrange(len(tb))
        sb[k] = sb[k] + 3
    eq = f"{''.join(ta)},{''.join(tb)}->{''.join(out)}"
    return eq, tuple(sa), tuple(sb)


def gen_parsers():
    rng = random.Random(1234)
    pair, pair_vals = [], {}
    seen = set()
    while len(pair) < 400:
        eq, sa, sb = random_pair_case(rng)
        if (eq, sa, sb) in seen:
            continue
        seen.add((eq, sa, sb))
        rec = {"eq": eq, "shape_a": list(sa), "shape_b": list(sb)}
        try:
            plan = refc._parse_eq_to_batch_matmul(eq, sa, sb)
        except ValueError as e:
            rec["error"] = "ValueError"
            pair.append(rec)
            continue
        rec["plan"] = enc_plan(plan)
        # numerical value through the reference's own lowering
        a, b = make_arrays([sa, sb], "complex128", seed=len(pair))
        try:
            val = refc.einsum(eq, a, b)
        except Exception as e:  # e.g. numpy refusing a broadcast in reshape
            rec["value_error"] = type(e).__name__
        else:
            # cross-check against numpy.einsum where numpy accepts the eq
            try:
                chk = np.einsum(eq, a, b)
                assert np.allclose(chk, val), eq
            except ValueError:
                pass
            pair_vals[f"pair_{len(pair)}"] = np.asarray(val)
        pair.append(rec)

    single, single_vals = [], {}
    seen = set()
    while len(single) < 120:
        n_ix = rng.randint(1, 4)
        pool = rng.sample("abcde", n_ix)
        sizes = {c: rng.choice([1, 2, 3, 4]) for c in pool}
        term = [rng.choice(pool) for _ in range(rng.randint(0, 5))]
        present = list(dict.fromkeys(term))
        out = [c for c in present if rng.random() < 0.6]
        rng.shuffle(out)
        eq = f"{''.join(term)}->{''.join(out)}"
        shape = tuple(sizes[c] for c in term)
        if (eq, shape) in seen:
            continue
        seen.add((eq, shape))
        diag, axes, perm = refc._parse_einsum_single(eq, shape)
        (x,) = make_arrays([shape], "complex128", seed=1000 + len(single))
        val = refc._einsum_single(eq, x)
        single_vals[f"single_{len(single)}"] = np.asarray(val)
        single.append(
            {
                "eq": eq,
                "shape": list(shape),
                "n_diag": None if diag is None else len(diag),
                "diag": jsonable(diag),
                "sum_axes": jsonable(axes),
                "perm": jsonable(perm),
            }
        )

    tdot = []
    while len(tdot) < 120:
        na, nb = rng.randint(0, 4), rng.randint(0, 4)
        ncon = rng.randint(0, min(na, nb))
        ax_a = tuple(rng.sample(range(na), ncon))
        ax_b = tuple(rng.sample(range(nb), ncon))
        sa = [rng.choice([1, 2, 3]) for _ in range(na)]
        sb = [rng.choice([1, 2, 3]) for _ in range(nb)]
        for i, j in zip(ax_a, ax_b):
            sb[j] = sa[i]
        rec = {
            "axes": [list(ax_a), list(ax_b)],
            "shape_a": sa,
            "shape_b": sb,
        }
        plan = refc._parse_tensordot_axes_to_matmul(
            (ax_a, ax_b), tuple(sa), tuple(sb)
        )
        rec["plan"] = enc_plan(plan)
        tdot.append(rec)

    with open(os.path.join(GOLDEN_DIR, "parsers.json"), "w") as f:
        json.dump({"pair": pair, "single": single, "tdot": tdot}, f)
    np.savez_compressed(
        os.path.join(GOLDEN_DIR, "parsers_values.npz"), **pair_vals, **single_vals
    )
    print("parsers:", len(pair), len(single), len(tdot))


# --------------------------------------------------------------------------
# 2. the reference's basic equations (tests/test_compute.py:8-99)
# --------------------------------------------------------------------------


def gen_equations():
    sys.path.insert(0, "/root/reference/tests")
    import importlib

    tc = importlib.import_module("test_compute")
    eqs = list(tc.test_case_eqs)
    recs, vals = [], {}
    for n, eq in enumerate(eqs):
        for d_min in (2, 1):
            shapes = ctg.utils.make_shapes_from_inputs(
                *(lambda io: (io[0], io[2]))(_eq_inputs_sizes(eq, n, d_min))
            )
            arrays = make_arrays(shapes, "complex128", seed=5000 + n)
            val = ctg.einsum(eq, *arrays)
            chk = np.einsum(eq, *arrays)
            assert np.allclose(val, chk), eq
            m, e = ctg.einsum(eq, *arrays, strip_exponent=True)
            key = f"eq{n}_d{d_min}"
            vals[key] = np.asarray(val)
            vals[key + "_m"] = np.asarray(m)
            vals[key + "_e"] = np.asarray(float(e))
            recs.append(
                {
                    "key": key,
                    "eq": eq,
                    "shapes": [list(s) for s in shapes],
                    "seed": 5000 + n,
                }
            )
    with open(os.path.join(GOLDEN_DIR, "equations.json"), "w") as f:
        json.dump(recs, f)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "equations_values.npz"), **vals)
    print("equations:", len(recs))


def _eq_inputs_sizes(eq, n, d_min):
    lhs, out = eq.split("->") if "->" in eq else (eq, None)
    inputs = [tuple(t) for t in lhs.split(",")]
    rng = random.Random(77 + n)
    size_dict = {}
    for t in inputs:
        for c in t:
            if c not in size_dict:
                size_dict[c] = rng.randint(d_min, 4)
    return inputs, out, size_dict


# --------------------------------------------------------------------------
# 3. trees: IR, index metadata, slice keys, values
# --------------------------------------------------------------------------


def tree_record(name, tree, dtype, seed, strip_exponent=False, extra=None):
    """Serialise everything the drop-in must reproduce for ``tree``."""
    inputs = [list(t) for t in tree.inputs]
    output = list(tree.output)
    size_dict = dict(tree.size_dict)
    contractions = refc.extract_contractions(tree)

    # traversal as ordered (left, right) SSA pairs + per-node index strings
    ssas = {leaf: i for i, leaf in enumerate(tree.gen_leaves())}
    inds = {i: tree.get_inds(leaf) for leaf, i in list(ssas.items())}
    path = []
    ssa = len(ssas)
    for p, l, r in tree.traverse():
        li, ri = ssas.pop(l), ssas.pop(r)
        ssas[p] = ssa
        inds[ssa] = tree.get_inds(p)
        path.append([li, ri])
        ssa += 1

    sliced = [
        [si.ind, si.size, si.project] for si in tree.sliced_inds.values()
    ]
    nsl = tree.nslices
    ids = sorted({0, nsl - 1, nsl // 2, nsl // 3, min(nsl - 1, 5)})
    keys = {str(i): tree.slice_key(i) for i in ids}

    rec = {
        "name": name,
        "inputs": inputs,
        "output": output,
        "size_dict": size_dict,
        "path": path,
        "sliced": sliced,
        "sliced_inputs": sorted(tree.sliced_inputs),
        "nslices": int(nsl),
        "multiplicity": int(tree.multiplicity),
        "contractions": jsonable(contractions),
        "preprocessing": {str(k): v for k, v in tree.preprocessing.items()},
        "inds": {str(k): v for k, v in inds.items()},
        "slice_keys": keys,
        "slice_strides": [
            int(s) for s in ctg.core.get_slice_strides(tree.sliced_inds)
        ],
        "dtype": dtype,
        "seed": seed,
        "strip_exponent": bool(strip_exponent),
        "contraction_cost": int(tree.contraction_cost()),
    }
    if extra:
        rec.update(extra)
    return rec


def tree_values(tree, rec, vals, max_slices_full=4096):
    shapes = [
        tuple(tree.size_dict[ix] for ix in term) for term in tree.inputs
    ]
    arrays = make_arrays(shapes, rec["dtype"], seed=rec["seed"])
    name = rec["name"]
    if tree.nslices <= max_slices_full:
        val = tree.contract(arrays)
        vals[name] = np.asarray(val)
        if rec["strip_exponent"]:
            m, e = tree.contract(arrays, strip_exponent=True)
            vals[name + "_m"] = np.asarray(m)
            vals[name + "_e"] = np.asarray(float(e))
    # always a few individual slices
    for i in list(rec["slice_keys"])[:3]:
        vals[f"{name}_slice{i}"] = np.asarray(tree.contract_slice(arrays, int(i)))


def gen_trees():
    recs, vals = [], {}
    rng = random.Random(99)
    np.random.seed(99)

    def add(name, tree, dtype="complex128", strip=False, extra=None):
        rec = tree_record(name, tree, dtype, seed=len(recs) + 1, strip_exponent=strip, extra=extra)
        tree_values(tree, rec, vals)
        recs.append(rec)

    # 3a. BASELINE config 1 (plumbing): 10-tensor random einsum, bond dim 4
    c = ctg.utils.rand_equation(10, 3, d_min=4, d_max=4, seed=0)
    tree = ctg.array_contract_tree(c.inputs, c.output, c.size_dict, optimize="greedy")
    add("config1_rand10", tree, strip=True)
    c = ctg.utils.rand_equation(10, 3, n_out=2, n_hyper_in=1, n_hyper_out=1, d_min=4, d_max=4, seed=0)
    tree = ctg.array_contract_tree(c.inputs, c.output, c.size_dict, optimize="greedy")
    add("config1_rand10_hyper", tree, strip=True)

    # 3b. random (hyper) networks, sliced and with sliced output indices
    k = 0
    for reg in (2, 3):
        for n_out in (0, 1, 2):
            for n_hi in (0, 1):
                for n_ho in (0, 1, 2):
                    for isort in (None, "root"):
                        k += 1
                        if k % 3 == 2:
                            continue
                        seed = rng.choice([42, 666, 7, 12])
                        c = ctg.utils.rand_equation(
                            n=10, reg=reg, n_out=n_out, n_hyper_in=n_hi,
                            n_hyper_out=n_ho, d_min=2, d_max=4, seed=seed,
                        )
                        tree = ctg.array_contract_tree(
                            c.inputs, c.output, c.size_dict, optimize="greedy",
                            sort_contraction_indices=isort,
                        )
                        name = f"rand_r{reg}_o{n_out}_hi{n_hi}_ho{n_ho}_{isort}_s{seed}"
                        add(name, tree, dtype=rng.choice(["float64", "complex128"]))
                        size = tree.max_size()
                        if size >= 64:
                            tree.slice_(target_size=max(size // 6, 1))
                            if isort:
                                tree.sort_contraction_indices(isort)
                            add(name + "_sliced", tree, strip=(k % 2 == 0))
                            rem = list(tree.get_legs(tree.root))
                            if rem:
                                tree.remove_ind_(rng.choice(rem))
                                if isort:
                                    tree.sort_contraction_indices(isort)
                                add(name + "_sliced_out", tree, strip=(k % 4 == 0))

    # 3c. projection (SliceInfo.project) and preprocessing x slicing
    c = ctg.utils.rand_equation(8, 3, n_out=1, d_min=2, d_max=3, seed=3)
    tree = ctg.array_contract_tree(c.inputs, c.output, c.size_dict, optimize="greedy")
    inner = [ix for ix in tree.size_dict if ix not in tree.output]
    tree.remove_ind_(inner[0], project=1)
    tree.remove_ind_(inner[1])
    add("projected", tree)

    for eq_name, eq in (("pre_diag", "aab,bc,cdd->a"), ("pre_sum", "ab,bcd,ce->ae")):
        inputs, output, size_dict = _eq_inputs_sizes(eq, 3, 2)
        size_dict = {c_: d + 1 for c_, d in size_dict.items()}
        tree = ctg.array_contract_tree(inputs, tuple(output), size_dict, optimize="greedy")
        add(eq_name, tree, dtype="float64")
        tree.remove_ind_("b")
        add(eq_name + "_sliced", tree, dtype="float64")

    # single-input trees
    for eq_name, eq in (("single_perm", "abc->cab"), ("single_trace", "abab->b"), ("single_sum", "abc->b")):
        inputs, output, size_dict = _eq_inputs_sizes(eq, 9, 2)
        tree = ctg.array_contract_tree(inputs, tuple(output), size_dict)
        add(eq_name, tree, strip=True)

    # 3d. lattices (tests/test_backends.py:105, tests/test_compute.py:222)
    c = ctg.utils.lattice_equation([4, 4])
    tree = ctg.array_contract_tree(c.inputs, c.output, c.size_dict, optimize="greedy")
    add("lattice4x4", tree, strip=True)
    tree.slice_(target_slices=4)
    add("lattice4x4_sliced", tree, strip=True)
    c = ctg.utils.lattice_equation([6, 6], d_min=3)
    tree = ctg.array_contract_tree(c.inputs, c.output, c.size_dict, optimize="greedy")
    tree.slice_(target_slices=8)
    add("lattice6x6_d3_sliced", tree, strip=True)

    # 3e. BASELINE config 2 structure at reduced bond (same topology: 8x8 PEPS)
    c = ctg.utils.lattice_equation([8, 8], d_min=2)
    tree = ctg.array_contract_tree(c.inputs, c.output, c.size_dict, optimize="greedy")
    add("peps8x8_d2", tree, dtype="complex128", strip=True)

    with open(os.path.join(GOLDEN_DIR, "trees.json"), "w") as f:
        json.dump(recs, f)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "trees_values.npz"), **vals)
    print("trees:", len(recs))


# --------------------------------------------------------------------------
# 4. Sycamore n53 m20 (BASELINE north-star workload)
# --------------------------------------------------------------------------


def appendix_b():
    txt = open(os.path.join(ROOT, "SURVEY.md")).read()
    m = re.search(r"SSA path \(380 pairs.*?```\n(.*?)\n```", txt, re.S)
    ssa = [tuple(map(int, p.split(","))) for p in m.group(1).strip().split(";")]
    m2 = re.search(r"index labels used in the JSON \(36\):\n`(.*?)`", txt, re.S)
    sliced = [chr(int(x)) for x in m2.group(1).split(",")]
    return ssa, sliced


def gen_sycamore():
    from cotengra.utils import load_from_json

    inputs, output, size_dict = load_from_json(
        "/root/reference/examples/benchmarks/sycamore_n53_m20_s0_e0_pABCDCDAB.json"
    )
    ssa, sliced = appendix_b()
    tree = ctg.ContractionTree.from_path(inputs, output, size_dict, ssa_path=ssa)
    for ix in sliced:
        tree.remove_ind_(ix)
    stats = tree.contract_stats()
    rec = tree_record(
        "sycamore_m20_appxB", tree, "complex128", seed=2020,
        extra={
            "contract_stats": {k: int(v) for k, v in stats.items()},
            "peak_size": int(tree.peak_size()),
            "ssa_path": [list(p) for p in ssa],
        },
    )
    # values: the same tree sliced further until a slice is oracle-sized
    small = tree.copy()
    small.slice_(target_size=2**16)
    srec = tree_record("sycamore_m20_small", small, "complex128", seed=2020)
    vals = {}
    shapes = [tuple(small.size_dict[ix] for ix in t) for t in small.inputs]
    arrays = make_arrays(shapes, "complex128", seed=2020, scale=1.0)
    for i in list(srec["slice_keys"])[:3]:
        vals[f"sycamore_m20_small_slice{i}"] = np.asarray(
            small.contract_slice(arrays, int(i))
        )
    # medium: W = 2**24 single slice for a heavier GPU-vs-reference check
    med = tree.copy()
    med.slice_(target_size=2**22)
    mrec = tree_record("sycamore_m20_medium", med, "complex128", seed=2020)
    for i in list(mrec["slice_keys"])[:1]:
        m_, e_ = med.contract_slice(arrays, int(i), strip_exponent=True)
        vals[f"sycamore_m20_medium_slice{i}_m"] = np.asarray(m_)
        vals[f"sycamore_m20_medium_slice{i}_e"] = np.asarray(float(e_))
    with open(os.path.join(GOLDEN_DIR, "sycamore_m20.json"), "w") as f:
        json.dump([rec, srec, mrec], f)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "sycamore_m20_values.npz"), **vals)
    print("sycamore:", stats, tree.nslices, small.nslices, med.nslices)


# --------------------------------------------------------------------------
# 5. Freshly searched random trees (tests/test_tree_ir.py)
# --------------------------------------------------------------------------


def gen_random_trees():
    """Greedy trees of random equations with random index orders, slicing and
    removed indices: ``tree_record`` holds what ``TreeSpec.from_cotengra`` reads
    and the reference's IR and slice keys it must reproduce."""
    rng = random.Random(5)
    recs = []
    for trial in range(40):
        c = ctg.utils.rand_equation(
            n=rng.randint(4, 12), reg=rng.randint(2, 4), n_out=rng.randint(0, 3),
            n_hyper_in=rng.randint(0, 2), n_hyper_out=rng.randint(0, 2),
            d_min=1, d_max=4, seed=trial,
        )
        tree = ctg.array_contract_tree(
            c.inputs, c.output, c.size_dict, optimize="greedy",
            sort_contraction_indices=rng.choice([None, "root", "flops"]),
        )
        if tree.max_size() > 16 and rng.random() < 0.7:
            tree.slice_(target_size=max(tree.max_size() // 4, 1))
        rem = [ix for ix in tree.get_legs(tree.root)]
        if rem and rng.random() < 0.5:
            tree.remove_ind_(rng.choice(rem))
        recs.append(tree_record(f"random_tree{trial}", tree, "complex128", seed=trial))
    with open(os.path.join(GOLDEN_DIR, "random_trees.json"), "w") as f:
        json.dump(recs, f)
    print("random trees:", len(recs))


# --------------------------------------------------------------------------
# 6. The drop-in boundary (tests/test_dropin_reference.py)
# --------------------------------------------------------------------------


def gen_dropin():
    """BASELINE config 1 (and its hyper-index variant) through the reference's
    own entry points: ``ctg.einsum``, ``tree.contract`` (plain, stripped,
    sliced), ``tree.contract_slice``, the keys its contractor cache used, and
    ``total_flops`` of a sliced lattice tree."""
    recs, vals = {}, {}
    for hyper in (False, True):
        kw = dict(n_out=2, n_hyper_in=1, n_hyper_out=1) if hyper else {}
        con = ctg.utils.rand_equation(10, 3, d_min=4, d_max=4, seed=0, **kw)
        shapes = [tuple(con.size_dict[ix] for ix in t) for t in con.inputs]
        arrays = make_arrays(shapes, "complex128", seed=0)
        eq = ctg.utils.inputs_output_to_eq(con.inputs, con.output)
        tag = f"config1_hyper{int(hyper)}"
        vals[f"{tag}_einsum"] = np.asarray(ctg.einsum(eq, *arrays))
        tree = ctg.array_contract_tree(con.inputs, con.output, con.size_dict, optimize="greedy")
        vals[f"{tag}_contract"] = np.asarray(tree.contract(arrays))
        m, e = tree.contract(arrays, strip_exponent=True)
        vals[f"{tag}_strip_m"], vals[f"{tag}_strip_e"] = np.asarray(m), np.asarray(e)
        rec = tree_record(tag, tree, "complex128", seed=0)
        rec["eq"] = eq
        # (strip_exponent, key) of every contractor the calls above cached
        rec["contractor_keys"] = [[bool(k[3]), jsonable(k)] for k in tree.contraction_cores]
        recs[tag] = rec
        if hyper:
            tree.slice_(target_size=max(tree.max_size() // 8, 1))
            vals["sliced_contract"] = np.asarray(tree.contract(arrays))
            for i in (0, tree.nslices - 1):
                vals[f"sliced_slice{i}"] = np.asarray(tree.contract_slice(arrays, i))
            recs["sliced"] = tree_record("sliced", tree, "complex128", seed=0)
    con = ctg.utils.lattice_equation([4, 4], d_min=3)
    tree = ctg.array_contract_tree(con.inputs, con.output, con.size_dict, optimize="greedy")
    tree.slice_(target_slices=9)
    recs["lattice4x4"] = tree_record("lattice4x4", tree, "float64", seed=0,
                                     extra={"total_flops_float64": int(tree.total_flops("float64"))})
    with open(os.path.join(GOLDEN_DIR, "dropin.json"), "w") as f:
        json.dump(recs, f)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "dropin_values.npz"), **vals)
    print("dropin:", sorted(recs))


if __name__ == "__main__":
    which = sys.argv[1:] or ["parsers", "equations", "trees", "sycamore", "random_trees", "dropin"]
    if "parsers" in which:
        gen_parsers()
    if "equations" in which:
        gen_equations()
    if "trees" in which:
        gen_trees()
    if "sycamore" in which:
        gen_sycamore()
    if "random_trees" in which:
        gen_random_trees()
    if "dropin" in which:
        gen_dropin()
