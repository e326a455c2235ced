"""The reference side of the GPU Ising test (tests/test_gpu_strip_exponent.py): the oracle's
stripped (mantissa, exponent) of a partition function that overflows float32 and float64, against
exact enumeration of all 2^20 configurations."""

import math

import numpy as np
import pytest

import cotengra_b200 as cb
from oracle import ctg_oracle as orc
from tests.ising import ising_log10_z, ising_network, random_path

# log10 Z to within these (single precision: relative to log10 Z, the reference accumulates
# its exponent in the dtype); single precision at beta = 4 (log10 Z ~ 54, beyond float32), as at
# beta = 40 the final inner product of two normalised halves underflows float32 in the reference
TOL = {"float64": 1e-12, "complex128": 1e-12, "float32": 1e-6, "complex64": 1e-6}
ISING_CASES = [(dt, beta) for dt in ("float64", "complex128") for beta in (0.5, 40.0)] + \
    [(dt, beta) for dt in ("float32", "complex64") for beta in (0.5, 4.0)]


@pytest.mark.parametrize("dtype,beta", ISING_CASES)
def test_oracle_ising_against_enumeration(dtype, beta):
    inputs, size_dict, tensors, J = ising_network(4, 5, beta, seed=3)
    want = ising_log10_z(4, 5, beta, J)
    if beta > 1.0:
        # Z itself is not representable in the dtype
        assert want > math.log10(np.finfo(np.dtype(dtype).type(0).real.dtype).max)
    arrays = [np.asarray(t, dtype=dtype) for t in tensors]
    for seed in range(3):
        spec = cb.TreeSpec(inputs, (), size_dict, random_path(inputs, seed))
        m, e = orc.run_contractions(spec.contractions(), arrays, strip_exponent=True)
        got = math.log10(abs(complex(np.asarray(m).reshape(-1)[0]))) + e
        tol = TOL[dtype] * (max(1.0, abs(want)) if dtype in ("float32", "complex64") else 1.0)
        assert abs(got - want) <= tol, (seed, got, want)


def test_enumeration_small_lattice():
    """The enumeration itself, on a 2 x 2 lattice summed by hand."""
    beta = 0.7
    inputs, size_dict, tensors, J = ising_network(2, 2, beta, seed=1)
    bonds = [(0, 1), (0, 2), (1, 3), (2, 3)]
    z = 0.0
    for c in range(16):
        s = [1 - 2 * ((c >> k) & 1) for k in range(4)]
        z += math.exp(beta * sum(j * s[u] * s[v] for (u, v), j in zip(bonds, J)))
    assert abs(ising_log10_z(2, 2, beta, J) - math.log10(z)) < 1e-14
