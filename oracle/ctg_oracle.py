"""CPU oracle: a numpy restatement of cotengra's contraction-execution path.

TEST INFRASTRUCTURE ONLY -- this file is the *checker*, never the product.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import it.  ``cotengra_b200`` (the product) must
never import anything under ``oracle/``.

What is restated (reference = jcmgray/cotengra @ 2182a79, paths relative to
``/root/reference``):

* pairwise lowering to (batched) matmul ......... cotengra/contract.py:167-329, 364-411
* single-term einsum (diag / sum / transpose) ... cotengra/contract.py:61-119, 332-361
* tensordot axes -> equation .................... cotengra/contract.py:472-518
* the per-slice node loop + strip_exponent ...... cotengra/contract.py:718-837
* slice id -> digits, slicing of the inputs ..... cotengra/core.py:114-122, 3775-3819
* gathering slices (sum / stack / exponents) .... cotengra/core.py:125-172, 3825-3882

Parity pinning: ``tests/test_oracle_golden.py`` checks every function here
against golden vectors produced by the *unmodified* reference imported in the
build container through the numpy-only ``autoray`` stand-in
(``oracle/refshim``); the generator is ``oracle/gen_golden.py`` and the vectors
live in ``tests/golden/``.  The arithmetic itself is numpy's (``matmul`` ->
OpenBLAS), exactly as in the reference's default CPU path.

The input "program" is the reference's own linear IR: the tuple of
``(parent, left, right, tdot, arg, perm)`` records that
``cotengra.contract.extract_contractions`` produces (contract.py:573-651).
"""

import functools

import numpy as np

# ----------------------------------------------------------------------------
# equation helpers
# ----------------------------------------------------------------------------


def split_equation(eq):
    """Return ``(lhs, out)``; an implicit output is every index that occurs
    exactly once, sorted (contract.py:34-58)."""
    eq = eq.replace(" ", "")
    if "..." in eq:
        raise NotImplementedError("Ellipsis not supported.")
    if "->" in eq:
        lhs, out = eq.split("->")
        return lhs, out
    flat = eq.replace(",", "")
    out = "".join(c for c in sorted(set(flat)) if flat.count(c) == 1)
    return eq, out


def _symbols():
    """a-z, A-Z, then unicode from chr(192) (contract.py:462-469)."""
    for base, n in (("a", 26), ("A", 26)):
        for i in range(n):
            yield chr(ord(base) + i)
    i = 192
    while True:
        yield chr(i)
        i += 1


# ----------------------------------------------------------------------------
# single-term einsum  (contract.py:61-119 and 332-361)
# ----------------------------------------------------------------------------


@functools.lru_cache(4096)
def plan_single(eq, shape):
    """Plan ``eq`` on one operand as (diagonal selectors, summed axes, perm).

    Mirrors the three-stage order of the reference: repeated indices are taken
    as diagonals by advanced indexing (last-discovered first), then indices that
    are absent from the output are summed, then the survivors are transposed.
    """
    term, out = split_equation(eq)

    repeated, dropped, met = [], [], set()
    for c in term:
        if c in repeated:
            continue
        if c in met:
            repeated.append(c)
            continue
        met.add(c)
        if c not in out:
            dropped.append(c)

    selectors = None
    if repeated:
        selectors = []
        extent = dict(zip(term, shape))
        for c in reversed(repeated):
            ar = tuple(range(extent[c]))
            selectors.append(tuple(ar if x == c else slice(None) for x in term))
            run = c * term.count(c)
            if run in term:
                # occurrences adjacent: numpy leaves the new axis in place
                term = term.replace(run, c)
            else:
                # separated: advanced-index result axis moves to the front
                term = c + term.replace(c, "")

    axes = None
    if dropped:
        axes = tuple(term.index(c) for c in dropped)
        for c in dropped:
            term = term.replace(c, "")

    perm = None if term == out else tuple(term.index(c) for c in out)
    return selectors, axes, perm


def einsum_single(eq, x):
    """One-operand einsum by explicit diag / sum / transpose steps.

    The reference first tries the backend's own ``einsum`` (contract.py:338-341);
    numpy has one, so on the reference's CPU path the result is
    ``numpy.einsum(eq, x)``.  We restate the manual three-step route (which the
    reference uses for backends without einsum) and the two agree to rounding;
    the golden tests check both.
    """
    x = np.asarray(x)
    selectors, axes, perm = plan_single(eq, tuple(x.shape))
    if selectors is not None:
        for sel in selectors:
            x = x[sel]
    if axes is not None:
        x = np.sum(x, axis=axes)
    if perm is not None:
        x = np.transpose(x, perm)
    return x


# ----------------------------------------------------------------------------
# pairwise lowering  (contract.py:122-329)
# ----------------------------------------------------------------------------


def _plan_pure_multiply(ta, sa, tb, sb, out):
    """No contracted index: align both operands to the output order with
    singleton axes and broadcast-multiply (contract.py:122-164)."""
    want_a, want_b, shp_a, shp_b = "", "", [], []
    for c in out:
        if c in ta:
            want_a += c
            shp_a.append(sa[ta.index(c)])
        else:
            shp_a.append(1)
        if c in tb:
            want_b += c
            shp_b.append(sb[tb.index(c)])
        else:
            shp_b.append(1)
    eq_a = None if want_a == ta else f"{ta}->{want_a}"
    eq_b = None if want_b == tb else f"{tb}->{want_b}"
    return (eq_a, eq_b, shp_a, shp_b, None, None, True)


def _prod(xs):
    p = 1
    for x in xs:
        p *= x
    return p


@functools.lru_cache(4096)
def plan_pair(eq, shape_a, shape_b):
    """Plan a two-operand einsum as transpose/reshape -> (batched) matmul ->
    reshape/transpose; returns the reference's 7-tuple
    ``(eq_a, eq_b, new_shape_a, new_shape_b, new_shape_ab, perm_ab, pure_mul)``
    (contract.py:167-329)."""
    lhs, out = eq.split("->")
    ta, tb = lhs.split(",")
    if len(ta) != len(shape_a):
        raise ValueError(f"Term '{ta}' does not match shape {shape_a}.")
    if len(tb) != len(shape_b):
        raise ValueError(f"Term '{tb}' does not match shape {shape_b}.")

    extent = {}
    ones = set()

    def _record(c, d):
        if extent.setdefault(c, d) != d:
            raise ValueError(
                f"Index {c} has mismatched sizes {extent[c]} and {d}."
            )

    # distinct non-trivial indices of each term, insertion ordered
    on_a = {}
    for c, d in zip(ta, shape_a):
        if d == 1:
            ones.add(c)
        else:
            _record(c, d)
            on_a[c] = None
    on_b = {}
    for c, d in zip(tb, shape_b):
        if d == 1:
            # size 1 here but >1 on the left is a broadcast, not a singleton
            if c not in on_a:
                ones.add(c)
        else:
            ones.discard(c)
            _record(c, d)
            on_b[c] = None

    batch, summed, keep_a, keep_b = [], [], [], []
    for c in on_a:
        if c in on_b:
            del on_b[c]
            (batch if c in out else summed).append(c)
        elif c in out:
            keep_a.append(c)
    for c in on_b:
        if c in out:
            keep_b.append(c)

    if not summed:
        return _plan_pure_multiply(ta, shape_a, tb, shape_b, out)

    lead_ones = [c for c in out if c in ones]

    def _prep(term, want):
        if term == want:
            return None
        if set(term) == set(want):
            return tuple(term.index(c) for c in want)
        return f"{term}->{want}"

    want_a = "".join(batch + keep_a + summed)
    want_b = "".join(batch + summed + keep_b)
    eq_a = _prep(ta, want_a)
    eq_b = _prep(tb, want_b)

    if batch:
        groups_a = (batch, keep_a, summed)
        groups_b = (batch, summed, keep_b)
        groups_o = (batch, keep_a, keep_b)
    else:
        groups_a = (keep_a, summed)
        groups_b = (summed, keep_b)
        groups_o = (keep_a, keep_b)

    def _fused(groups):
        if all(len(g) == 1 for g in groups):
            return None
        return tuple(_prod(extent[c] for c in g) for g in groups)

    new_a = _fused(groups_a)
    new_b = _fused(groups_b)
    if lead_ones or any(len(g) != 1 for g in groups_o):
        new_ab = (1,) * len(lead_ones) + tuple(
            extent[c] for g in groups_o for c in g
        )
    else:
        new_ab = None

    produced = "".join(lead_ones + batch + keep_a + keep_b)
    perm_ab = (
        None if produced == out else tuple(produced.index(c) for c in out)
    )
    return (eq_a, eq_b, new_a, new_b, new_ab, perm_ab, False)


@functools.lru_cache(4096)
def plan_tensordot(axes, shape_a, shape_b):
    """Tensordot axes -> synthetic equation -> :func:`plan_pair`
    (contract.py:472-518)."""
    na, nb = len(shape_a), len(shape_b)
    if isinstance(axes, int):
        ax_a = tuple(range(na - axes, na))
        ax_b = tuple(range(axes))
    else:
        ax_a, ax_b = axes
    if len(ax_a) != len(ax_b):
        raise ValueError(
            f"Axes should have the same length, got {ax_a} and {ax_b}."
        )
    sym = _symbols()
    ia = [next(sym) for _ in range(na)]
    ib, io = [], list(ia)
    for j in range(nb):
        if j in ax_b:
            i = ax_a[ax_b.index(j)]
            if shape_a[i] != shape_b[j]:
                raise ValueError(
                    f"Dimension mismatch between axes {i} of {shape_a} and "
                    f"{j} of {shape_b}: {shape_a[i]} != {shape_b[j]}."
                )
            c = ia[i]
            io.remove(c)
        else:
            c = next(sym)
            io.append(c)
        ib.append(c)
    eq = f"{''.join(ia)},{''.join(ib)}->{''.join(io)}"
    return plan_pair(eq, shape_a, shape_b)


def _apply_plan(a, b, plan):
    """Execute a 7-tuple plan with numpy (contract.py:364-411)."""
    eq_a, eq_b, new_a, new_b, new_ab, perm_ab, pure = plan
    a = np.asarray(a)
    b = np.asarray(b)
    if eq_a is not None:
        a = np.transpose(a, eq_a) if isinstance(eq_a, tuple) else einsum_single(eq_a, a)
    if new_a is not None:
        a = np.reshape(a, new_a)
    if eq_b is not None:
        b = np.transpose(b, eq_b) if isinstance(eq_b, tuple) else einsum_single(eq_b, b)
    if new_b is not None:
        b = np.reshape(b, new_b)
    if pure:
        return np.multiply(a, b)
    ab = np.matmul(a, b)
    if new_ab is not None:
        ab = np.reshape(ab, new_ab)
    if perm_ab is not None:
        ab = np.transpose(ab, perm_ab)
    return ab


def einsum(eq, a, b=None):
    """Single or pairwise einsum using only transpose / reshape / matmul / sum
    (contract.py:414-459)."""
    if b is None:
        return einsum_single(eq, a)
    a = np.asarray(a)
    b = np.asarray(b)
    return _apply_plan(a, b, plan_pair(eq, tuple(a.shape), tuple(b.shape)))


def tensordot(a, b, axes=2):
    """Tensordot via matmul (contract.py:521-570)."""
    try:
        axes = tuple(map(int, axes[0])), tuple(map(int, axes[1]))
    except (IndexError, TypeError):
        axes = int(axes)
    a = np.asarray(a)
    b = np.asarray(b)
    return _apply_plan(
        a, b, plan_tensordot(axes, tuple(a.shape), tuple(b.shape))
    )


# ----------------------------------------------------------------------------
# the node loop  (contract.py:718-837)
# ----------------------------------------------------------------------------


def run_contractions(
    contractions, arrays, strip_exponent=False, check_zero=False,
    implementation=None,
):
    """Contract ``arrays`` by walking the linear program ``contractions``.

    Returns the output array, or ``(mantissa, exponent)`` (base-10 exponent) if
    ``strip_exponent``.  ``implementation`` is an ``(einsum, tensordot)`` pair
    that every node is dispatched to instead of this module's own, as the
    reference's ``implementation=`` argument does (contract.py:752-776).
    """
    einsum_, tensordot_ = implementation or (einsum, tensordot)
    live = dict(enumerate(arrays))
    exponent = 0.0 if strip_exponent else None
    out = None
    for p, l, r, tdot, arg, perm in contractions:
        if r is None:
            if l is None:
                # in-place preprocessing of input ``p``
                live[p] = einsum_(arg, live[p])
                continue
            # single-input tree
            out = einsum_(arg, live[l])
            return (out, 0.0) if strip_exponent else out
        x = live.pop(l)
        y = live.pop(r)
        if tdot:
            out = tensordot_(x, y, arg)
            if perm:
                out = np.transpose(out, perm)
        else:
            out = einsum_(arg, x, y)
        if exponent is not None:
            top = np.max(np.abs(out))
            if check_zero and float(top) == 0.0:
                return 0.0, float("-inf")
            exponent = exponent + np.log10(top)
            out = out / top
        live[p] = out
    if exponent is not None:
        return out, exponent
    return out


# ----------------------------------------------------------------------------
# slicing  (core.py:114-122, 3775-3819)
# ----------------------------------------------------------------------------
# ``sliced`` is the ordered list ``[(ind, size, project_or_None), ...]`` in the
# order of ``tree.sliced_inds`` (output indices first, then by name:
# core.py:99-104, 1989-1991).


def slice_strides(sliced):
    """Mixed-radix place values, most significant first (core.py:114-122)."""
    n = len(sliced)
    strides = [1] * n
    for i in range(n - 2, -1, -1):
        strides[i] = strides[i + 1] * sliced[i + 1][1]
    return strides


def slice_key(sliced, i):
    """Digits of slice id ``i`` as ``{ind: value}`` (core.py:3775-3800);
    projected indices keep their fixed value and consume no digit."""
    key = {}
    for (ind, _size, project), stride in zip(sliced, slice_strides(sliced)):
        if project is None:
            key[ind] = i // stride
            i %= stride
        else:
            key[ind] = project
    return key


def slice_arrays(inputs, sliced, arrays, i):
    """Basic-index every input that carries a sliced index (core.py:3802-3819)."""
    key = slice_key(sliced, i)
    out = list(arrays)
    for c, term in enumerate(inputs):
        if any(ix in key for ix in term):
            sel = tuple(key.get(ix, slice(None)) for ix in term)
            out[c] = np.asarray(arrays[c])[sel]
    return out


def num_slices(sliced):
    return _prod(size for _ind, size, project in sliced if project is None)


# ----------------------------------------------------------------------------
# gathering  (core.py:125-172, 3825-3882)
# ----------------------------------------------------------------------------


def add_maybe_stripped(x, y):
    """``x + y`` where either may be ``(mantissa, exponent)`` (core.py:142-172)."""
    xt, yt = isinstance(x, tuple), isinstance(y, tuple)
    if not (xt or yt):
        return x + y
    xm, xe = x if xt else (x, 0.0)
    ym, ye = y if yt else (y, 0.0)
    e = max(xe, ye)
    return (xm * 10 ** (xe - e) + ym * 10 ** (ye - e), e)


def gather_slices(output, sliced, results):
    """Combine per-slice results: plain sum when no sliced index is an output
    index, otherwise sum over inner sliced indices and stack over the outer
    ones (core.py:3825-3882)."""
    where = {
        ix: pos
        for pos, ix in enumerate(output)
        if any(ix == s[0] for s in sliced)
    }
    if not where:
        return functools.reduce(add_maybe_stripped, results)

    chunks = {}
    for i, res in enumerate(results):
        key = slice_key(sliced, i)
        k = tuple(key[ix] for ix in where)
        chunks[k] = add_maybe_stripped(chunks[k], res) if k in chunks else res

    emax = None
    if isinstance(next(iter(chunks.values())), tuple):
        emax = max(e for _m, e in chunks.values())
        chunks = {k: m * 10 ** (e - emax) for k, (m, e) in chunks.items()}

    info = {s[0]: s for s in sliced}

    def _stack(prefix, rest):
        if not rest:
            return chunks[prefix]
        ind, size, project = info[rest[0]]
        values = range(size) if project is None else [project]
        parts = [_stack(prefix + (d,), rest[1:]) for d in values]
        return np.stack(parts, where[rest[0]] - len(prefix))

    result = _stack((), tuple(where))
    return (result, emax) if emax is not None else result


def contract_tree(
    inputs,
    output,
    sliced,
    contractions,
    arrays,
    strip_exponent=False,
    check_zero=False,
    slice_ids=None,
):
    """``ContractionTree.contract`` (core.py:3943-4030): serial slice loop +
    gather.  ``slice_ids`` restricts the loop (used for bounded CPU-baseline
    samples and for emulating a rank's round-robin share, core.py:4070)."""
    if not sliced:
        return run_contractions(contractions, arrays, strip_exponent, check_zero)
    n = num_slices(sliced)
    ids = range(n) if slice_ids is None else slice_ids
    results = (
        run_contractions(
            contractions,
            slice_arrays(inputs, sliced, arrays, i),
            strip_exponent,
            check_zero,
        )
        for i in ids
    )
    if slice_ids is not None:
        # partial sums only make sense when every sliced index is inner
        return functools.reduce(add_maybe_stripped, results)
    return gather_slices(output, sliced, results)


def contraction_cost(contractions, shapes):
    """Scalar multiply-adds of one pass over ``contractions`` given the (sliced)
    input shapes: sum over nodes of the product of all involved index extents
    (core.py:1014-1022, 1362-1364).  Used by bench.py to convert time to flops
    without importing the reference."""
    live = {i: tuple(s) for i, s in enumerate(shapes)}
    total = 0
    elements = 0
    for p, l, r, tdot, arg, perm in contractions:
        if r is None:
            continue
        sa, sb = live.pop(l), live.pop(r)
        if tdot:
            ax_a, ax_b = arg
            k = _prod(sa[i] for i in ax_a)
            keep_a = [d for i, d in enumerate(sa) if i not in ax_a]
            keep_b = [d for i, d in enumerate(sb) if i not in ax_b]
            shp = keep_a + keep_b
            if perm:
                shp = [shp[i] for i in perm]
            total += _prod(shp) * k
        else:
            lhs, out = arg.split("->")
            ta, tb = lhs.split(",")
            ext = {}
            for c, d in list(zip(ta, sa)) + list(zip(tb, sb)):
                ext[c] = max(ext.get(c, 1), d)
            total += _prod(ext.values())
            shp = [ext[c] for c in out]
        elements += _prod(sa) + _prod(sb) + _prod(shp)
        live[p] = tuple(shp)
    return total, elements
