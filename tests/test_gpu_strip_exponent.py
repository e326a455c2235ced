"""Fused strip_exponent on the GPU, kernel by kernel and at the ends of the floating-point range.

The device normalises lazily (DESIGN §4): a node stores its raw product and records max|C| in a
factor slot; its consumer multiplies by 1/(fA fB) -- through a scaled copy of a small operand, or in
its own epilogue -- and the exponent is the sum of log10 of the slots.  A product m * 10**e does
not change when a slot holds a wrong value (the consumer's scale and the exponent absorb the error
alike), so these tests check the pieces themselves:

A. every STRIP instantiation, one launch at a time, with the scale and factor words of the
   descriptor pointed at slots the test owns: the scaled product, the recorded maximum, and the
   branches of the epilogue (double fallback of the single-precision kernels, the two-factor scale,
   the hypot path, zero factors, NaN, the integer pre-filter);
B. whole trees: the reference's (mantissa, exponent) pair itself, inputs scaled towards the ends of
   each type's range through every way an operand reaches a node, and an Ising partition function
   whose value overflows every floating-point type against exact enumeration."""

import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import cotengra_b200 as cb  # noqa: E402
from cotengra_b200 import lowering as L  # noqa: E402
from oracle import ctg_oracle as orc  # noqa: E402
from tests.helpers import load_json, load_npz, make_arrays, rel_err  # noqa: E402
from tests.ising import ising_log10_z, ising_network, random_path  # noqa: E402
from tests.test_strip_range_cpu import ISING_CASES  # noqa: E402

# fused strip_exponent words of a pair descriptor (csrc/gett_desc.h): device addresses of doubles
W_SCALE_A, W_SCALE_B, W_FACTOR_C = 36, 37, 38

DOUBLE = ("float64", "complex128")
ALL = ("float64", "complex128", "float32", "complex64")
WIDE = {"float32": np.float64, "float64": np.float64, "complex64": np.complex128, "complex128": np.complex128}


def _single(dtype):
    return dtype not in DOUBLE


# ---------------------------------------------------------------------------------------------
# A. one launch at a time
# ---------------------------------------------------------------------------------------------
# (name, dtypes, (M, K, N), build_pair_desc kwargs, variant the lowering must pick, measure_after)
# measure_after: the executor measures max|C| in a pass of its own (split-K atomics, the
# block-reduction kernels, tcgen05 with more than one TMEM chunk) and leaves W_FACTOR_C = 0
_R = (130, 19, 70)  # ragged in every tile dimension
LAUNCHES = [
    ("simt", ALL, _R, {"variant": L.VAR_SIMT_64x64}, L.VAR_SIMT_64x64, False),
    ("mma_128x64", ALL, _R, {"variant": L.VAR_DMMA_128x64}, L.VAR_DMMA_128x64, False),
    ("mma_64x128", ALL, (70, 33, 130), {"variant": L.VAR_DMMA_64x128}, L.VAR_DMMA_64x128, False),
    ("mma_256x32", ALL, (300, 21, 37), {"variant": L.VAR_DMMA_256x32}, L.VAR_DMMA_256x32, False),
    ("mma_256x16", ALL, (300, 21, 13), {"variant": L.VAR_DMMA_256x16}, L.VAR_DMMA_256x16, False),
    ("dmma_32x32", DOUBLE, (30, 40, 29), {"variant": L.VAR_DMMA_32x32, "force_splitk": 1}, L.VAR_DMMA_32x32, False),
    ("dmma3m_128x32", ("complex128",), _R, {"variant": L.VAR_DMMA3M_128x32}, L.VAR_DMMA3M_128x32, False),
    ("dmma3m_256x16", ("complex128",), (300, 21, 13), {"variant": L.VAR_DMMA3M_256x16}, L.VAR_DMMA3M_256x16,
     False),
    ("row_128x8", ALL, (301, 19, 7), {"variant": L.VAR_ROW_128x8, "force_splitk": 1}, L.VAR_ROW_128x8, False),
    ("row_256x4", ALL, (301, 19, 3), {"variant": L.VAR_ROW_256x4, "force_splitk": 1}, L.VAR_ROW_256x4, False),
    ("rowstream_n4k4", ALL, (4096, 4, 3), {}, L.VAR_ROWSTREAM, False),
    ("rowstream_n2k8", ALL, (4096, 7, 2), {}, L.VAR_ROWSTREAM, False),
    ("rowstream_n8k8", ALL, (4096, 8, 7), {}, L.VAR_ROWSTREAM, False),
    ("rowstream_longk", ("float32", "float64", "complex64"), (4096, 40, 5), {}, L.VAR_ROWSTREAM_K, False),
    ("dmmastream_n8", ("complex128",), (4096, 40, 6), {}, L.VAR_DMMASTREAM, False),
    ("dmmastream_n16", ("complex128",), (4096, 20, 13), {}, L.VAR_DMMASTREAM, False),
    ("dmmastream_n32", ("complex128",), (4096, 20, 29), {"variant": L.VAR_DMMASTREAM}, L.VAR_DMMASTREAM, False),
    ("tc05_lean", ("complex64",), (1024, 64, 128), {"force_splitk": 1}, L.VAR_TC05_128x64, False),
    ("tc05_general_6n", ("complex64",), (216, 36, 216), {"force_splitk": 1}, L.VAR_TC05_128x64, False),
    ("tc05_narrow", ("complex64",), (4096, 32, 16), {}, L.VAR_TC05_128x16, False),
    # measure_after launches: the scaling only
    ("split_k", ALL, (130, 256, 70), {"variant": L.VAR_DMMA_128x64, "force_splitk": 4}, L.VAR_DMMA_128x64, True),
    ("kred", ALL, (1, 65536, 1), {}, L.VAR_KRED, True),
    ("dotstream", ALL, (1, 1 << 20, 1), {}, L.VAR_DOTSTREAM, True),
    ("dotstream4", ALL, (3, 1 << 20, 4), {}, L.VAR_DOTSTREAM4, True),
    ("tc05_chunked", ("complex64",), (256, 512, 64), {"force_splitk": 1}, L.VAR_TC05_128x64, True),
]

# (name, scale of the operands, fA, fB, dtypes)
FACTORS = [
    ("moderate", 1.0, 3.7, 0.21, ALL),
    ("single_fallback_big", 1e15, 1e20, 1e20, ALL),          # 1/(fA fB) = 1e-40: not a normal float
    ("single_fallback_small", 1e-15, 1e-20, 1e-20, ALL),     # 1e+40
    ("double_two", 1e-100, 1e-160, 1e-160, DOUBLE),          # (1/fA)(1/fB) = 1e320 overflows
    ("subnormal_product", 1e100, 1e160, 1e160, DOUBLE),      # (1/fA)(1/fB) = 1e-320 is subnormal
    ("hypot_huge", 1e100, 1.0, 1.0, DOUBLE),                  # |C|^2 ~ 1e400
    ("hypot_tiny", 1e-100, 1.0, 1.0, DOUBLE),                 # |C|^2 ~ 1e-400
    ("zero_factor", 1.0, 0.0, 2.0, ALL),
    ("nan", 1.0, 1.5, 0.5, ALL),
]
PLANTS = ["corner", "negative", "imaginary", "filter_boundary"]


def _operands(dtype, M, K, N, scale, seed):
    a, b = make_arrays([(M, K), (K, N)], dtype, seed=seed)
    return (a * np.asarray(scale, dtype=a.real.dtype)).astype(dtype), (b * np.asarray(scale, a.real.dtype)).astype(dtype)


def _planted(dtype, M, K, N, kind):
    """C = A B is V everywhere but in the last row and column -- the last element of the ragged
    final tile, the last one its thread stores -- where it is P with |P| = V (1 + 1e-3):
    negative, purely imaginary, or with both components just above max/sqrt(2), the edge of the
    integer pre-filter (real types: just above V)."""
    V, eps = 0.75, 1e-3
    if kind == "negative":
        P = -V * (1 + eps)
    elif kind == "imaginary":
        P = 1j * V * (1 + eps)
    elif kind == "filter_boundary":
        P = V * (1 + eps) / math.sqrt(2) * (1 + 1j) if np.dtype(dtype).kind == "c" else V * (1 + eps)
    else:
        P = 0.5 * V + 1j * V if np.dtype(dtype).kind == "c" else 1.5 * V
    a = np.zeros((M, K), dtype=dtype)
    b = np.zeros((K, N), dtype=dtype)
    a[:, 0] = 1
    a[M - 1, 1] = 1
    b[0, :] = V
    b[1, N - 1] = P - V
    return a, b


def _launch(plan, a, b, out_shape, dtype, words_patch):
    import torch

    from cotengra_b200 import _lib

    words = plan.words.copy()
    for k, v in words_patch.items():
        words[k] = v
    ta, tb = torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.from_numpy(np.ascontiguousarray(b)).cuda()
    c = torch.zeros(out_shape, dtype=ta.dtype, device="cuda")
    pa, pb = (tb, ta) if plan.swapped else (ta, tb)
    _lib.check(_lib.load().ctgb_contract_pair(words.ctypes.data, pa.data_ptr(), pb.data_ptr(), c.data_ptr(), 0))
    torch.cuda.synchronize()
    return c.cpu().numpy()


def _run_launch(plan, a, b, dtype, fa, fb, scale, track, seed_slot=0.0):
    """One launch with the slots owned here; returns (C, slot after the launch)."""
    import torch

    slots = torch.tensor([fa, fb, seed_slot], dtype=torch.float64, device="cuda")
    patch = {W_SCALE_A: 0, W_SCALE_B: 0, W_FACTOR_C: 0}
    if scale:
        # both scale words together: the kernels read both as soon as the first is set
        patch[W_SCALE_A] = slots[0].data_ptr()
        patch[W_SCALE_B] = slots[1].data_ptr()
    if track:
        patch[W_FACTOR_C] = slots[2].data_ptr()
    c = _launch(plan, a, b, (a.shape[0], b.shape[1]), dtype, patch)
    return c, float(slots[2].item())


def _check_launch(plan, a, b, dtype, fa, fb, scale, track, tag, fails):
    tol = 1e-5 if _single(dtype) else 1e-12
    wide = WIDE[dtype]
    raw = a.astype(wide) @ b.astype(wide)
    if scale:
        sa = 1.0 / fa if fa != 0 else 0.0
        sb = 1.0 / fb if fb != 0 else 0.0
        with np.errstate(invalid="ignore"):
            want = raw * sa * sb
    else:
        want = raw
    c, slot = _run_launch(plan, a, b, dtype, fa, fb, scale, track)
    fin = np.isfinite(want)
    if not np.array_equal(np.isfinite(c), fin):
        fails.append(f"{tag}: non-finite pattern of C differs from the reference")
        return
    if scale and (fa == 0 or fb == 0):
        if np.any(c != 0):
            fails.append(f"{tag}: zero factor, C has nonzeros (max {np.max(np.abs(c)):.3e})")
    else:
        err = rel_err(c[fin], want[fin]) if fin.any() else 0.0
        if not err <= tol:
            fails.append(f"{tag}: C rel err {err:.3e} > {tol:.0e} (max|C| {np.max(np.abs(c[fin])):.3e}, "
                         f"want {np.max(np.abs(want[fin])):.3e})")
    if not track:
        return
    if not fin.all():
        if not math.isnan(slot):
            fails.append(f"{tag}: NaN in C, slot {slot!r}")
        return
    mx = float(np.max(np.abs(c.astype(wide))))
    if mx == 0.0:
        if slot != 0.0:
            fails.append(f"{tag}: C is zero, slot {slot!r}")
        return
    if not abs(slot - mx) <= 1e-15 * mx:
        fails.append(f"{tag}: slot {slot!r} != max|C| {mx!r} (rel {abs(slot - mx) / mx:.2e})")
        return
    # a slot already above the maximum keeps its value (atomicMax)
    _c, kept = _run_launch(plan, a, b, dtype, fa, fb, scale, track, seed_slot=4.0 * mx)
    if kept != 4.0 * mx:
        fails.append(f"{tag}: pre-seeded slot {4.0 * mx!r} became {kept!r}")


def _plan(dtype, M, K, N, kw):
    from cotengra_b200 import _lib

    dims = L.classify_pair("ab", (M, K), "bc", (K, N), "ac")
    return L.build_pair_desc(dims, dtype, c_dense_elems=M * N, sm_count=_lib.device_info()["sm_count"], **kw)


_LAUNCH_PARAMS = [pytest.param(case, dt, id=f"{case[0]}-{dt}") for case in LAUNCHES for dt in case[1]]


@pytest.mark.parametrize("case,dtype", _LAUNCH_PARAMS)
def test_strip_epilogue_per_launch(case, dtype):
    """Scale + track and track-only, for every factor/magnitude case and planted maximum."""
    name, _dts, (M, K, N), kw, want_variant, measure_after = case
    plan = _plan(dtype, M, K, N, kw)
    print(f"{name} {dtype}: variant {plan.variant} splitk {plan.splitk} swapped {plan.swapped}")
    assert plan.variant == want_variant, (name, dtype, plan.variant)
    if name == "split_k":
        assert plan.splitk > 1
    fails = []
    for fname, mag, fa, fb, dts in FACTORS:
        if dtype not in dts:
            continue
        a, b = _operands(dtype, M, K, N, mag, seed=M + K + N)
        if fname == "nan":
            a = a.copy()
            a[min(1, M - 1), K // 2] = np.nan
        for scale, track in ((False, True), (True, True)):
            if measure_after:
                track = False  # the plan measures these nodes afterwards
                if not scale:
                    continue
            _check_launch(plan, a, b, dtype, fa, fb, scale, track,
                          f"{name}/{dtype}/{fname}/{'scale+track' if scale else 'track'}", fails)
    if not measure_after and min(M, N) > 1 and K >= 2:
        for kind in PLANTS:
            if kind == "imaginary" and np.dtype(dtype).kind != "c":
                continue
            a, b = _planted(dtype, M, K, N, kind)
            for scale, track in ((False, True), (True, True)):
                _check_launch(plan, a, b, dtype, 3.7, 0.21, scale, track,
                              f"{name}/{dtype}/plant_{kind}/{'scale+track' if scale else 'track'}", fails)
    assert not fails, "\n".join(fails)


# ---------------------------------------------------------------------------------------------
# B1. the reference's pair, not only its product
# ---------------------------------------------------------------------------------------------
TREES = load_json("trees.json")
TVALS = load_npz("trees_values.npz")
_STRIP_TREES = [r for r in TREES if r["strip_exponent"] and r["name"] + "_m" in TVALS]


def _spec(rec):
    from tests.helpers import decode_sliced

    n_in = len(rec["inputs"])
    node_inds = {int(k): v for k, v in rec["inds"].items() if int(k) >= n_in}
    return cb.TreeSpec(rec["inputs"], rec["output"], rec["size_dict"], rec["path"],
                       decode_sliced(rec["sliced"]), node_inds)


@pytest.mark.parametrize("rec", _STRIP_TREES, ids=[r["name"] for r in _STRIP_TREES])
def test_golden_mantissa_and_exponent(rec):
    """What ``tree.contract(strip_exponent=True)`` returns, compared as a pair: the root's own
    factor is the only tracker a wrong split between mantissa and exponent would expose here."""
    spec = _spec(rec)
    arrays = make_arrays(spec.shapes(), rec["dtype"], seed=rec["seed"])
    wm, we = TVALS[rec["name"] + "_m"], float(TVALS[rec["name"] + "_e"])
    m, e = cb.contract_tree(spec, arrays, strip_exponent=True)
    assert abs(e - we) <= 1e-10, (e, we)
    assert rel_err(m, wm) <= 1e-10
    if not spec.sliced and spec.N > 1:
        # (the reference strips after pairwise nodes only: a one-input tree keeps its raw values)
        assert abs(float(np.max(np.abs(m))) - 1.0) <= 1e-14


# ---------------------------------------------------------------------------------------------
# B2. range trees
# ---------------------------------------------------------------------------------------------
# (name, inputs, output, size_dict, path, sliced); every operand > 16 MiB in float32 is "large":
# its consumer scales in the epilogue instead of through a scaled copy of the operand
_a, _b, _c = 2048, 2080, 2048
RANGE_TREES = {
    # X = P Q, Y = R S (both large), Z = X Y: an epilogue-scaled matrix product of two raw products
    "gemm_of_products": (["ai", "ib", "bj", "jc"], "ac", dict(a=_a, b=_b, c=_c, i=4, j=4),
                         [(0, 1), (2, 3), (4, 5)], ()),
    # Z = sum X * Y over 2^23 elements: the dot-stream root of two large raw products
    "dot_of_products": (["ai", "ib", "aj", "jb"], "", dict(a=4096, b=2048, i=2, j=2),
                        [(0, 1), (2, 3), (4, 5)], ()),
    # Y small: the consumer takes a scaled copy of it (control)
    "prescaled_control": (["ai", "ib", "bj", "jc"], "ac", dict(a=_a, b=_b, c=8, i=4, j=4),
                          [(0, 1), (2, 3), (4, 5)], ()),
    # the stem (P Q) R with R a large input, in both operand orders
    "stem_big_input": (["ai", "ib", "bc"], "ac", dict(a=_a, b=_b, c=_c, i=4), [(0, 1), (3, 2)], ()),
    "stem_big_input_swapped": (["ai", "ib", "bc"], "ac", dict(a=_a, b=_b, c=_c, i=4), [(0, 1), (2, 3)], ()),
    # sliced over j: X = P Q is slice-invariant (hoisted, computed once, reread by every slice)
    "sliced_hoisted": (["ai", "ib", "bj", "jc"], "ac", dict(a=64, b=65600, c=64, i=4, j=4),
                       [(0, 1), (2, 3), (4, 5)], (("j", 4, None),)),
}
SIGMA = {"float32": 12, "complex64": 12, "float64": 90, "complex128": 90}


def _range_spec(name):
    inputs, output, sizes, path, sliced = RANGE_TREES[name]
    return cb.TreeSpec([tuple(t) for t in inputs], tuple(output), sizes, path, sliced)


def _oracle(spec, arrays):
    return orc.contract_tree([tuple(t) for t in spec.inputs], spec.output, spec.sliced, spec.contractions(),
                             arrays, strip_exponent=True)


def _stripped_err(m, e, m_ref, e_ref):
    return rel_err(np.asarray(m, dtype=np.complex128) * 10.0 ** (e - e_ref), m_ref)


_ORACLE_CACHE = {}


def _range_case(name, dtype, sign):
    key = (name, dtype, sign)
    if key not in _ORACLE_CACHE:
        spec = _range_spec(name)
        s = SIGMA[dtype] * sign
        arrays = make_arrays(spec.shapes(), dtype, seed=7, scale=10.0 ** s)
        wide = [x.astype(WIDE[dtype]) for x in arrays]
        m_ref, e_ref = _oracle(spec, wide)
        tol = 1e-10
        if _single(dtype):
            m32, e32 = _oracle(spec, arrays)
            assert np.all(np.isfinite(m32)) and math.isfinite(e32), "oracle left the single range"
            tol = max(1e-5, 3.0 * _stripped_err(m32, e32, m_ref, e_ref))
        _ORACLE_CACHE[key] = (spec, arrays, m_ref, e_ref, tol)
    return _ORACLE_CACHE[key]


def _check_range(m, e, m_ref, e_ref, tol, tag):
    m = np.asarray(m)
    assert np.all(np.isfinite(m)) and math.isfinite(e), f"{tag}: m finite {np.all(np.isfinite(m))}, e = {e}"
    assert not (np.any(m_ref != 0) and (np.all(m == 0) or e == -math.inf)), f"{tag}: nonzero value returned as zero"
    err = _stripped_err(m, e, m_ref, e_ref)
    assert err <= tol, f"{tag}: rel err {err:.3e} > {tol:.1e} (e {e:.6f}, e_ref {e_ref:.6f})"


@pytest.mark.parametrize("sign", [0, 1, -1], ids=["sigma0", "sigma_plus", "sigma_minus"])
@pytest.mark.parametrize("dtype", ALL)
@pytest.mark.parametrize("name", list(RANGE_TREES))
def test_range_tree(name, dtype, sign):
    spec, arrays, m_ref, e_ref, tol = _range_case(name, dtype, sign)
    for fuse in (False, True):
        m, e = cb.contract_tree(spec, arrays, strip_exponent=True, fuse=fuse)
        _check_range(m, e, m_ref, e_ref, tol, f"{name}/{dtype}/sigma {SIGMA[dtype] * sign}/fuse={fuse}")


@pytest.mark.parametrize("dtype", ["complex128", "float32"])
def test_range_tree_through_contractor(dtype):
    """The ``tree.contract_slice`` path (B200Contractor) on the epilogue-scaled product."""
    spec, arrays, m_ref, e_ref, tol = _range_case("gemm_of_products", dtype, 1)
    fn = cb.B200Contractor(spec.contractions(), strip_exponent=True)
    m, e = fn(*arrays)
    _check_range(m, e, m_ref, e_ref, tol, f"contractor/{dtype}")


# ---------------------------------------------------------------------------------------------
# B3. Ising partition function, exact
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,beta", ISING_CASES)
def test_ising_partition_function(dtype, beta):
    """4 x 5 open lattice, random +-J bonds: log10 Z from the stripped pair against all 2^20
    configurations.  At beta = 40, log10 Z is several hundred: Z overflows float32 and float64
    (single precision runs at beta = 4, log10 Z ~ 54: at 40 the reference's own float32 run ends
    in an inner product that underflows)."""
    inputs, size_dict, tensors, J = ising_network(4, 5, beta, seed=3)
    want = ising_log10_z(4, 5, beta, J)
    arrays = [np.asarray(t, dtype=dtype) for t in tensors]
    for seed in range(3):
        path = random_path(inputs, seed)
        spec = cb.TreeSpec(inputs, (), size_dict, path)
        m, e = cb.contract_tree(spec, arrays, strip_exponent=True, fuse=False)
        got = math.log10(abs(complex(np.asarray(m).reshape(-1)[0]))) + e
        tol = 1e-12
        if _single(dtype):
            m32, e32 = orc.run_contractions(spec.contractions(), arrays, strip_exponent=True)
            ref32 = math.log10(abs(complex(np.asarray(m32).reshape(-1)[0]))) + e32
            tol = max(1e-6 * max(1.0, abs(want)), 3.0 * abs(ref32 - want))
        assert abs(got - want) <= tol, (seed, got, want)
