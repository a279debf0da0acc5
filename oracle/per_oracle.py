"""TEST INFRASTRUCTURE -- float32 numpy restatement of the prioritised-replay contract of include/pbn_b200.h
("Prioritised replay"; only tests/ may import this, the product never does).

Proportional PER over a sum / min segment tree (Schaul et al.), in the form of OpenAI baselines that SURVEY.md
section 2 rows 13-14 describes for the reference's data_structures.py: stratified masses, a min tree for the
weight normaliser, new transitions at the running maximum priority.  The reference's own PER tests are stale
(SURVEY.md section 4), so parity is unpinned; this file states the project's semantics:

  trees     heap arrays of 2L float32 (node k -> 2k, 2k+1; root 1; leaf of slot i at L + i), sum: one fp32 add per
            node, min: fmin; unwritten leaves 0 (sum) / +inf (min); max_p = 1.0 initially
  push      slots (head + e) % capacity <- float32 max_p ** alpha
  update    raw = fmin(fmax(|td|, 0) + eps, 1e30) (NaN -> eps, inf -> 1e30); leaf <- raw ** alpha, in batch order
            (the last occurrence of a slot wins); max_p = max(max_p, raw); indices outside [0, capacity) ignored
  sample    seg = total / B, mass_b = fl(fl(u_b seg) + fl(b seg)); descend: left if left > mass or right == 0, else
            mass = fl(mass - left), right; weight = (pmin / p) ** beta (float64 here)
"""
import numpy as np

F32 = np.float32


def pow2_at_least(capacity: int) -> int:
    n = 1
    while n < capacity:
        n *= 2
    return n


def clamp_raw(td, eps) -> np.ndarray:
    """raw priority of TD errors: NaN -> eps, +-inf -> 1e30 (np.fmax / np.fmin drop the NaN)."""
    td = np.asarray(td, dtype=F32)
    with np.errstate(invalid="ignore"):
        return np.fmin(np.fmax(np.abs(td), F32(0)) + F32(eps), F32(1e30)).astype(F32)


def build_trees(sum_leaves: np.ndarray, min_leaves: np.ndarray, L: int):
    """Sum and min heaps with the given leaf rows (float32; leaves past the rows 0 / +inf).  The rows differ where a
    slot is unwritten: 0 in the sum tree, +inf in the min tree.  Internal nodes are left for rebuild()."""
    s = np.zeros(2 * L, dtype=F32)
    m = np.full(2 * L, np.inf, dtype=F32)
    s[L:L + len(sum_leaves)] = sum_leaves
    m[L:L + len(min_leaves)] = min_leaves
    return s, m


def rebuild(s: np.ndarray, m: np.ndarray, L: int) -> None:
    """Every internal node from the leaves, level by level (the fixed pairwise order of the contract)."""
    n = L // 2
    while n >= 1:
        s[n:2 * n] = s[2 * n:4 * n:2] + s[2 * n + 1:4 * n:2]
        m[n:2 * n] = np.fmin(m[2 * n:4 * n:2], m[2 * n + 1:4 * n:2])
        n //= 2


def descend(s: np.ndarray, L: int, mass: np.ndarray) -> np.ndarray:
    """The guarded descent for float32 masses; returns slot indices."""
    mass = np.asarray(mass, dtype=F32).copy()
    node = np.ones(mass.shape, dtype=np.int64)
    for _ in range(L.bit_length() - 1):
        left, right = s[2 * node], s[2 * node + 1]
        go_left = (left > mass) | (right == 0)
        mass = np.where(go_left, mass, (mass - left).astype(F32)).astype(F32)
        node = 2 * node + (~go_left)
    return node - L


def stratified_masses(total, u) -> np.ndarray:
    u = np.asarray(u, dtype=F32)
    seg = F32(total) / F32(len(u))
    return (u * seg).astype(F32) + (np.arange(len(u), dtype=F32) * seg).astype(F32)


def sample(s: np.ndarray, m: np.ndarray, L: int, u, beta):
    """index (int64) and float64 weights of a stratified sample from the trees."""
    index = descend(s, L, stratified_masses(s[1], u))
    weight = (np.float64(m[1]) / s[L + index].astype(np.float64)) ** beta
    return index, weight


class OraclePER:
    def __init__(self, capacity: int, alpha: float):
        self.capacity, self.alpha = capacity, F32(alpha)
        self.L = pow2_at_least(capacity)
        self.s, self.m = build_trees(np.zeros(0, dtype=F32), np.zeros(0, dtype=F32), self.L)
        self.max_p = F32(1.0)

    def leaves(self) -> np.ndarray:
        return self.s[self.L:self.L + self.capacity]

    def push(self, head: int, n: int) -> None:
        slots = (head + np.arange(n)) % self.capacity
        p = np.power(self.max_p, self.alpha, dtype=F32)
        self.s[self.L + slots] = p
        self.m[self.L + slots] = p
        rebuild(self.s, self.m, self.L)

    def update(self, index, td, eps) -> None:
        raw = clamp_raw(td, eps)
        for i, r in zip(np.asarray(index, dtype=np.int64), raw):   # batch order: the last occurrence wins
            if 0 <= i < self.capacity:
                p = np.power(r, self.alpha, dtype=F32)
                self.s[self.L + i] = p
                self.m[self.L + i] = p
                self.max_p = max(self.max_p, r)
        rebuild(self.s, self.m, self.L)

    def sample(self, u, beta):
        return sample(self.s, self.m, self.L, u, beta)
