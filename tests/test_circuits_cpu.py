"""Host-side .qsim reader: gate set sanity and the structure of the reference's Sycamore
circuit files (copied under ``tests/golden/``)."""

import os

import numpy as np
import pytest

from cotengra_b200.circuits import amplitude_network, gate_matrix, read_qsim
from tests.helpers import GOLDEN_DIR, load_json


def _qsim(m):
    return os.path.join(GOLDEN_DIR, f"circuit_n53_m{m}_s0_e0_pABCDCDAB.qsim")


def test_gates_are_unitary_and_square_roots():
    X = np.array([[0, 1], [1, 0]], dtype=complex)
    Y = np.array([[0, -1j], [1j, 0]], dtype=complex)
    W = (X + Y) / np.sqrt(2)
    for name, params, target in (("x_1_2", (), X), ("y_1_2", (), Y), ("hz_1_2", (), W)):
        U = gate_matrix(name, params)
        assert np.allclose(U @ U.conj().T, np.eye(2))
        S = U @ U
        phase = S[np.nonzero(np.abs(target) > 0.5)][0] / target[np.nonzero(np.abs(target) > 0.5)][0]
        assert np.allclose(S, phase * target)  # square root up to a global phase
    for t in (0.3, -1.7):
        U = gate_matrix("rz", (t,))
        assert np.allclose(U @ U.conj().T, np.eye(2))
    U = gate_matrix("fs", (1.5157741664069029, 0.5567125777723744))
    assert np.allclose(U @ U.conj().T, np.eye(4))
    with pytest.raises(ValueError):
        gate_matrix("cz", ())


def test_sycamore_m10_network_structure():
    path = _qsim(10)
    n, gates = read_qsim(path)
    assert n == 53 and len(gates) == 1658  # SURVEY.md Appendix C
    inputs, output, size_dict, arrays = amplitude_network(path)
    assert len(inputs) == 1658 + 2 * 53 == len(arrays)
    assert output == () and set(size_dict.values()) == {2}
    # every index appears exactly twice (closed network)
    counts = {}
    for t in inputs:
        for ix in t:
            counts[ix] = counts.get(ix, 0) + 1
    assert set(counts.values()) == {2}
    assert all(a.shape == (2,) * len(t) for a, t in zip(arrays, inputs))


def test_rank_simplify_small_circuit_keeps_the_amplitude(tmp_path):
    """rank_simplify on a random 6-qubit circuit in the .qsim gate set: same amplitude
    (dense contraction of both networks), far fewer tensors."""
    from cotengra_b200.circuits import rank_simplify

    rng = np.random.default_rng(0)
    lines = ["6"]
    for cyc in range(6):
        for q in range(6):
            lines.append(f"{3 * cyc} {rng.choice(['x_1_2', 'y_1_2', 'hz_1_2'])} {q}")
        for q in range(cyc % 2, 5, 2):
            lines.append(f"{3 * cyc + 1} rz {q} {rng.uniform(-3, 3)}")
            lines.append(f"{3 * cyc + 1} rz {q + 1} {rng.uniform(-3, 3)}")
            lines.append(f"{3 * cyc + 2} fs {q} {q + 1} {rng.uniform(0, 2)} {rng.uniform(0, 2)}")
    path = tmp_path / "c.qsim"
    path.write_text("\n".join(lines) + "\n")
    inputs, output, size_dict, arrays = amplitude_network(str(path), bits=[1, 0, 1, 1, 0, 0])
    s_in, s_out, s_sizes, s_arr = rank_simplify(inputs, output, size_dict, arrays)
    assert len(s_in) < len(inputs) // 4
    assert all(a.shape == tuple(s_sizes[ix] for ix in t) for a, t in zip(s_arr, s_in))

    def dense(ins, arrs):
        from oracle import ctg_oracle as orc
        import cotengra_b200 as cb

        n = len(ins)
        path_, cur = [], 0
        for i in range(1, n):
            path_.append((cur, i))
            cur = n + i - 1
        spec = cb.TreeSpec(ins, (), {ix: 2 for t in ins for ix in t}, path_)
        return orc.run_contractions(spec.contractions(), arrs)

    # a linear path over a 6-qubit circuit stays tiny
    a0, a1 = dense(inputs, arrays), dense(s_in, s_arr)
    assert abs(a0 - a1) < 1e-12 * max(1.0, abs(a0))


@pytest.mark.parametrize("m,tensors,indices", [(10, 164, 319), (20, 381, 754)])
def test_rank_simplify_reaches_the_notebook_sizes(m, tensors, indices):
    """The reference notebooks contract networks simplified by quimb: m10 has 164 tensors / 319
    indices (`Quantum Circuit Example Old.ipynb:143`), m20 381 / 754 -- the shipped benchmark JSON
    (`ex_benchmarking.ipynb` cell 4).  rank_simplify reproduces both counts from the .qsim files."""
    from cotengra_b200.circuits import rank_simplify

    path = _qsim(m)
    inputs, output, size_dict, arrays = amplitude_network(path)
    s_in, _o, s_sizes, s_arr = rank_simplify(inputs, output, size_dict, arrays)
    assert len(s_in) == tensors and len(s_sizes) == indices
    assert max(len(t) for t in s_in) <= 4
    counts = {}
    for t in s_in:
        for ix in t:
            counts[ix] = counts.get(ix, 0) + 1
    assert set(counts.values()) == {2}
    if m == 20:
        # same degree sequence as the reference's benchmark structure file, whose network
        # sycamore_m20.json carries
        ref_inputs = next(r for r in load_json("sycamore_m20.json") if r["name"] == "sycamore_m20_appxB")["inputs"]
        assert sorted(len(t) for t in ref_inputs) == sorted(len(t) for t in s_in)
