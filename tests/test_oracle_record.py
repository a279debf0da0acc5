"""CPU: the oracle of the steady-state record contract (oracle/record_oracle.py) against a per-env Python loop, for
one-word and two-word states."""
import numpy as np
import pytest

from oracle.record_oracle import record_states


def _loop(states, n, genes):
    gene_on = [0] * n
    hist = None if genes is None else [0] * (1 << len(genes))
    for row in states:
        v = 0
        for k, w in enumerate(row):
            v |= int(w) << (64 * k)
        for g in range(n):
            gene_on[g] += (v >> g) & 1
        if genes is not None:
            hist[sum(((v >> g) & 1) << j for j, g in enumerate(genes))] += 1
    return gene_on, hist


@pytest.mark.parametrize("n,genes", [(7, None), (7, []), (7, [6, 0, 3]), (10, list(range(10))), (28, [27, 1, 14, 5]),
                                     (70, [69, 3, 64, 12, 40, 0, 65, 31, 32, 63, 7, 50]), (128, [127, 0, 64, 63])])
def test_record_states_matches_a_python_loop(n, genes):
    rng = np.random.default_rng(n)
    w = (n + 63) // 64
    st = rng.integers(0, 2**63, size=(301, w), dtype=np.int64).astype(np.uint64) * np.uint64(2) + \
        rng.integers(0, 2, size=(301, w)).astype(np.uint64)
    if n % 64:
        st[:, -1] &= np.uint64((1 << (n % 64)) - 1)
    st[:40] = st[0]   # a concentrated part: many equal states
    gene_on, hist = record_states(st, n, genes)
    ref_on, ref_hist = _loop(st, n, genes)
    assert gene_on.dtype == np.uint64 and gene_on.tolist() == ref_on
    if genes is None:
        assert hist is None
    else:
        assert hist.dtype == np.uint64 and hist.tolist() == ref_hist and int(hist.sum()) == st.shape[0]


@pytest.mark.parametrize("genes", [list(range(13)), [1, 1], [-1], [7]])
def test_record_states_rejects_bad_projections(genes):
    with pytest.raises(ValueError):
        record_states(np.zeros((3, 1), dtype=np.uint64), 7, genes)
