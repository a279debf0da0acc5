"""CPU: the prioritised-replay restatement (oracle/per_oracle.py) is a correct proportional sampler, and the ctypes
mirror of the pbn_per struct matches include/pbn_b200.h."""
import ctypes as C

import numpy as np
import pytest

from oracle import per_oracle as P


def test_descent_matches_cumsum_search():
    rng = np.random.default_rng(0)
    for cap in (1, 2, 5, 100, 1000):
        L = P.pow2_at_least(cap)
        leaves = rng.random(cap).astype(np.float32) + np.float32(0.01)
        s, m = P.build_trees(leaves, leaves, L)
        P.rebuild(s, m, L)
        assert m[1] == leaves.min()
        edges = np.cumsum(leaves.astype(np.float64))
        mass = rng.random(2000) * s[1]
        # masses away from the segment boundaries (rounding of the partial sums decides exactly at a boundary)
        gap = np.min(np.abs(mass[:, None] - edges[None, :]), axis=1)
        mass = mass[gap > 1e-3 * s[1]].astype(np.float32)
        want = np.searchsorted(edges, mass.astype(np.float64), side="right")
        assert np.array_equal(P.descend(s, L, mass), want), cap


def test_last_occurrence_wins_and_clamp():
    per = P.OraclePER(10, alpha=1.0)
    per.update([3, 3, 3, 12, -1], [1.0, 2.0, 0.5, 9.0, 9.0], eps=0.0625)
    assert per.leaves()[3] == np.float32(0.5625)   # last in batch order; 12 and -1 are ignored
    assert per.max_p == np.float32(2.0625)          # every valid entry folds into max_p
    raw = P.clamp_raw([np.nan, np.inf, -np.inf, -2.0, 0.0], 1e-6)
    assert raw.dtype == np.float32
    assert raw.tolist() == [np.float32(1e-6), np.float32(1e30), np.float32(1e30), np.float32(2.0) + np.float32(1e-6),
                            np.float32(1e-6)]
    per.update([4], [np.nan], eps=0.25)
    assert np.isfinite(per.s).all() and per.leaves()[4] == np.float32(0.25)


def test_push_enters_at_max_priority_and_weights():
    per = P.OraclePER(6, alpha=0.5)
    per.push(4, 4)                                  # wraps: slots 4, 5, 0, 1
    assert per.leaves().tolist() == [1.0, 1.0, 0.0, 0.0, 1.0, 1.0]
    per.update([0], [3.0], eps=1.0)                 # raw 4 -> p 2, max_p 4
    per.push(2, 1)
    assert per.leaves()[2] == np.float32(2.0) and per.s[1] == np.float32(7.0) and per.m[1] == np.float32(1.0)
    idx, w = per.sample(np.array([0.0, 0.5, 0.999], dtype=np.float32), beta=1.0)
    assert np.all((idx >= 0) & (idx < 6)) and np.all(per.leaves()[idx] > 0)
    assert np.allclose(w, per.m[1] / per.leaves()[idx].astype(np.float64)) and w.max() <= 1.0


def test_mass_rounded_up_to_total_lands_on_a_written_slot():
    per = P.OraclePER(13, alpha=1.0)
    per.push(0, 7)                                  # slots 7..12 and the padding leaves stay empty
    u = np.array([np.nextafter(np.float32(1), np.float32(0))] * 3, dtype=np.float32)
    idx, _ = per.sample(u, beta=0.4)
    assert idx.max() < 7


def test_sampled_frequencies_are_proportional_to_priorities():
    from scipy.stats import chisquare
    rng = np.random.default_rng(7)
    cap, alpha = 50, 0.6
    per = P.OraclePER(cap, alpha)
    per.push(0, cap)
    per.update(np.arange(cap), rng.exponential(1.0, cap).astype(np.float32), eps=1e-6)
    counts = np.zeros(cap)
    for _ in range(200):
        idx, _ = per.sample(rng.random(256, dtype=np.float32), beta=0.4)
        counts += np.bincount(idx, minlength=cap)
    p = per.leaves().astype(np.float64)
    expected = counts.sum() * p / p.sum()
    assert chisquare(counts, expected).pvalue > 1e-3


def test_per_struct_layout_matches_the_header(tmp_path):
    import subprocess
    from pathlib import Path

    from pbn_rl_b200 import _cabi
    root = Path(__file__).resolve().parent.parent
    cls = _cabi.Per
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "pbn_b200.h"', "int main(void) {",
             'printf("size %zu\\n", sizeof(pbn_per));']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(pbn_per, %s));' % (fname, fname))
    lines += ["return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-I", str(root / "include"), "-o", str(exe), str(src)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(cls)
    for fname, _ in cls._fields_:
        assert int(got[fname]) == getattr(cls, fname).offset, fname


def test_tree_floats_and_argument_checks_without_a_device():
    from pbn_rl_b200 import _cabi
    lib = _cabi.load_library()
    assert lib.pbn_per_tree_floats(1) == 5 and lib.pbn_per_tree_floats(1000) == 5 * 1024
    assert lib.pbn_per_tree_floats(0) < 0 and lib.pbn_per_tree_floats((1 << 30) + 1) < 0
    p = _cabi.Per()
    assert lib.pbn_per_init(None, C.byref(p), None) < 0
    assert b"PER" in lib.pbn_last_error()
