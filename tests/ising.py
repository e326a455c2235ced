"""Ising partition functions as tensor networks, and their exact values by enumeration.

An open L1 x L2 lattice with random +-J bonds.  Every bond is a 2 x 2 tensor exp(beta J s s');
every spin is a COPY tensor joining the ends of its bonds, so each index appears exactly twice.
At low temperature the bond weights are exp(+-beta) -- unnormalised tensors of magnitude
10^(+-beta/ln 10) -- and Z itself overflows every floating-point type, which is what the
stripped exponent is for."""

import math

import numpy as np

from cotengra_b200.tree import get_symbol


def _bonds(l1, l2):
    out = []
    for i in range(l1):
        for j in range(l2):
            n = i * l2 + j
            if j + 1 < l2:
                out.append((n, n + 1))
            if i + 1 < l1:
                out.append((n, n + l2))
    return out


def ising_network(l1, l2, beta, seed=0):
    """``(inputs, size_dict, tensors, J)``: bond tensors first, then one COPY tensor per spin."""
    bonds = _bonds(l1, l2)
    J = np.random.default_rng(seed).choice([-1.0, 1.0], size=len(bonds))
    s = np.array([1.0, -1.0])
    inputs, tensors = [], []
    ends = {n: [] for n in range(l1 * l2)}
    for k, ((u, v), j) in enumerate(zip(bonds, J)):
        iu, iv = get_symbol(2 * k), get_symbol(2 * k + 1)
        inputs.append((iu, iv))
        tensors.append(np.exp(beta * j * np.outer(s, s)))
        ends[u].append(iu)
        ends[v].append(iv)
    for n in range(l1 * l2):
        d = len(ends[n])
        copy = np.zeros((2,) * d)
        copy[(0,) * d] = copy[(1,) * d] = 1.0
        inputs.append(tuple(ends[n]))
        tensors.append(copy)
    size_dict = {ix: 2 for t in inputs for ix in t}
    return inputs, size_dict, tensors, J


def ising_log10_z(l1, l2, beta, J):
    """Exact log10 Z over all 2^(l1 l2) configurations (logsumexp in float64)."""
    n = l1 * l2
    conf = ((np.arange(1 << n)[:, None] >> np.arange(n)[None, :]) & 1).astype(np.int8)
    spins = 1 - 2 * conf
    energy = np.zeros(1 << n)
    for (u, v), j in zip(_bonds(l1, l2), J):
        energy += j * (spins[:, u] * spins[:, v])
    x = beta * energy
    top = x.max()
    return (top + math.log(np.exp(x - top).sum())) / math.log(10.0)


def random_path(inputs, seed):
    """A seeded SSA contraction path that merges two tensors sharing an index whenever it can."""
    rng = np.random.default_rng(seed)
    live = {i: set(t) for i, t in enumerate(inputs)}
    nxt, path = len(inputs), []
    while len(live) > 1:
        ids = sorted(live)
        pairs = [(a, b) for x, a in enumerate(ids) for b in ids[x + 1:] if live[a] & live[b]]
        if not pairs:
            pairs = [(ids[0], ids[1])]
        a, b = pairs[rng.integers(len(pairs))]
        live[nxt] = live.pop(a) ^ live.pop(b)
        path.append((a, b))
        nxt += 1
    return path
