"""Numpy restatement of the steady-state record contract (include/pbn_b200.h, pbn_rollout_record /
pbn_record_states): per-gene ON counts and the histogram of the states projected onto up to 12 genes."""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np


def record_states(states_u64: np.ndarray, n_genes: int, genes: Optional[Sequence[int]]) -> Tuple[np.ndarray, Optional[np.ndarray]]:
    """``(gene_on [n_genes] uint64, hist [2^k] uint64)`` of one record of ``states_u64`` ([E, W] packed words, bit g of
    word g // 64 = gene g).  ``gene_on[g]`` = number of states with gene g ON; bin ``b = sum_j bit(genes[j]) << j``;
    ``genes=None`` gives ``hist = None``, ``genes=[]`` one bin holding E."""
    st = np.asarray(states_u64, dtype=np.uint64)
    st = st.reshape(st.shape[0], -1)
    if genes is not None:
        genes = [int(g) for g in genes]
        if len(genes) > 12 or len(set(genes)) != len(genes) or any(g < 0 or g >= n_genes for g in genes):
            raise ValueError("at most 12 distinct projection genes in [0, n_genes)")
    bits = [(st[:, g >> 6] >> np.uint64(g & 63)) & np.uint64(1) for g in range(n_genes)]
    gene_on = np.array([int(b.sum()) for b in bits], dtype=np.uint64)
    if genes is None:
        return gene_on, None
    idx = np.zeros(st.shape[0], dtype=np.int64)
    for j, g in enumerate(genes):
        idx |= bits[g].astype(np.int64) << j
    hist = np.bincount(idx, minlength=1 << len(genes)).astype(np.uint64)
    return gene_on, hist
