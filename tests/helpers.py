"""Helpers shared by the golden generator (``oracle/gen_golden.py``) and the
tests: deterministic synthetic arrays and golden-file decoding."""

import json
import os
from types import SimpleNamespace

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def make_arrays(shapes, dtype="complex128", seed=0, scale=1.0):
    """Seeded synthetic operands: uniform(-1, 1) real parts (plus imaginary
    parts for complex dtypes), generated in float64 then cast, so that every
    dtype sees the same underlying values."""
    rng = np.random.default_rng(seed)
    dtype = np.dtype(dtype)
    arrays = []
    for shape in shapes:
        shape = tuple(int(d) for d in shape)
        x = rng.uniform(-1.0, 1.0, size=shape)
        if dtype.kind == "c":
            x = x + 1j * rng.uniform(-1.0, 1.0, size=shape)
        arrays.append(np.asarray(x * scale).astype(dtype))
    return arrays


def load_json(name):
    with open(os.path.join(GOLDEN_DIR, name)) as f:
        return json.load(f)


def load_npz(name):
    return np.load(os.path.join(GOLDEN_DIR, name))


def decode_ir(contractions):
    """JSON -> the reference's contraction records ``(p, l, r, tdot, arg,
    perm)`` with tuples restored."""
    out = []
    for p, l, r, tdot, arg, perm in contractions:
        if tdot:
            arg = (tuple(arg[0]), tuple(arg[1]))
        if perm is not None:
            perm = tuple(perm)
        out.append((p, l, r, bool(tdot), arg, perm))
    return tuple(out)


def decode_sliced(sliced):
    return [(ind, int(size), None if project is None else int(project))
            for ind, size, project in sliced]


class RecordedTree:
    """A ``cotengra.ContractionTree`` as ``oracle/gen_golden.tree_record`` stored it: the
    attributes ``TreeSpec.from_cotengra`` reads (nodes are the record's SSA ids) and the
    contractor cache ``cotengra_b200.install`` seeds."""

    def __init__(self, rec):
        self.inputs = [tuple(t) for t in rec["inputs"]]
        self.output = tuple(rec["output"])
        self.size_dict = dict(rec["size_dict"])
        self.sliced_inds = {ix: SimpleNamespace(ind=ix, size=int(size), project=project)
                            for ix, size, project in rec["sliced"]}
        self._path = [tuple(p) for p in rec["path"]]
        self._inds = {int(k): v for k, v in rec["inds"].items()}
        self.contraction_cores = {}

    def gen_leaves(self):
        return iter(range(len(self.inputs)))

    def traverse(self):
        n = len(self.inputs)
        return [(n + k, l, r) for k, (l, r) in enumerate(self._path)]

    def get_inds(self, node):
        return self._inds[node]


def rel_err(x, ref):
    x = np.asarray(x)
    ref = np.asarray(ref)
    den = np.max(np.abs(ref))
    if den == 0:
        return float(np.max(np.abs(x))) if x.size else 0.0
    return float(np.max(np.abs(x - ref)) / den)
