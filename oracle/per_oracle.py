"""TEST INFRASTRUCTURE, NOT PRODUCT CODE: sequential numpy restatement of the proportional prioritized replay of
include/madigan_b200.h ("Proportional prioritized replay"), one record and one sample at a time.

``PerOracle`` keeps the leaves and replays ingest and update_priorities as a loop would; ``sample`` descends a given
sum tree (the oracle's own, or one read back from the GPU) with the Philox draws of ``orc_philox4x32_10``."""
import ctypes as C

import numpy as np

from oracle.oracle import lib

SUB_LEAVES = 1024
DRAW_TAG = 0x80000000  # bit 31 of the second Philox counter word
MAX_ATTEMPTS = 64
INT64_MIN = -2 ** 63
_M32 = 0xFFFFFFFF


def tree_size(capacity):
    """Leaves of the trees: a power of two >= max(capacity, 1024)."""
    return max(SUB_LEAVES, 1 << (int(capacity) - 1).bit_length())


def build_tree(leaves, op):
    """Heap array [2T] over T leaves: node 1 is the root, node j = op(node 2j, node 2j+1); node 0 is unused (0)."""
    T = len(leaves)
    t = np.zeros(2 * T, dtype=np.float64)
    t[T:] = leaves
    n = T
    while n > 1:
        t[n // 2:n] = op(t[n:2 * n:2], t[n + 1:2 * n:2])
        n //= 2
    return t


def draw_uniform(seed, draw, b, attempt):
    """u in [0, 1) of sample b, attempt `attempt`: Philox counter (b lo, (b hi) ^ (attempt << 8) ^ tag, draw lo,
    draw hi), key seed, u = (x0 >> 11) 2^-53."""
    ctr = (C.c_uint32 * 4)(b & _M32, ((b >> 32) ^ (attempt << 8) ^ DRAW_TAG) & _M32, draw & _M32, (draw >> 32) & _M32)
    key = (C.c_uint32 * 2)(seed & _M32, (seed >> 32) & _M32)
    out = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(ctr, key, out)
    x0 = (out[1] << 32) | out[0]
    return (x0 >> 11) * 2.0 ** -53


def descend(sum_tree, mass):
    """Leaf index reached from the root: go left if the left child > mass, else subtract it and go right."""
    T = len(sum_tree) // 2
    node = 1
    while node < T:
        left = float(sum_tree[2 * node])
        if left > mass:
            node = 2 * node
        else:
            mass = mass - left
            node = 2 * node + 1
    return node - T


def sample(sum_tree, min_tree, leaf_pos, state_step, filled, cur_step, depth, batch, beta, seed, draw):
    """(idx, pos, weights) of one sample call.  leaf_pos [capacity]: append position per slot (-1 unfilled);
    state_step [capacity]: MdgReplay.t_state_step; filled = min(cursor, capacity)."""
    capacity = len(leaf_pos)
    T = len(sum_tree) // 2
    total = float(sum_tree[1])
    seg = total / float(batch)
    idx = np.full(batch, -1, dtype=np.int64)
    pos = np.full(batch, -1, dtype=np.int64)
    w = np.zeros(batch, dtype=np.float64)
    for b in range(batch):
        attempt = 0
        while attempt < MAX_ATTEMPTS and filled > 0 and total > 0.:
            u = draw_uniform(seed, draw, b, attempt)
            mass = u * seg + float(b) * seg if attempt == 0 else u * total
            attempt += 1
            leaf = descend(sum_tree, mass)
            if leaf >= capacity or leaf_pos[leaf] < 0 or not float(sum_tree[T + leaf]) > 0.:
                continue
            ss = int(state_step[leaf])
            if ss != INT64_MIN and ss > cur_step - depth:
                idx[b] = leaf
                break
        if idx[b] < 0:
            continue
        pos[b] = leaf_pos[idx[b]]
        n = float(filled)
        with np.errstate(divide="ignore"):  # C's pow: a p_min of 0 (an underflowed leaf) gives weight 0
            w[b] = np.float64(float(sum_tree[T + idx[b]]) / total * n) ** -beta / \
                np.float64(float(min_tree[1]) / total * n) ** -beta
    return idx, pos, w


class PerOracle:
    """Leaves, append positions, max_priority and the rejected count of one buffer of `capacity` slots."""

    def __init__(self, capacity, alpha):
        self.capacity, self.alpha = int(capacity), float(alpha)
        self.T = tree_size(capacity)
        self.sum_leaves = np.zeros(self.T)
        self.min_leaves = np.full(self.T, np.inf)
        self.leaf_pos = np.full(self.capacity, -1, dtype=np.int64)
        self.max_priority = 1.0
        self.seen = 0
        self.n_rejected = 0

    def ingest(self, cursor):
        """The records appended up to `cursor` (MdgReplay.cursor) enter at max_priority ** alpha."""
        for p in range(max(self.seen, cursor - self.capacity), cursor):
            slot = p % self.capacity
            self.sum_leaves[slot] = self.min_leaves[slot] = self.max_priority ** self.alpha
            self.leaf_pos[slot] = p
        self.seen = cursor

    def update(self, idx, pos, priorities):
        """update_priorities for a sampled batch (idx, pos as sample returned them), in batch order."""
        for i, p, q in zip(idx, pos, priorities):
            i, q = int(i), float(q)
            if i < 0 or self.leaf_pos[i] != p:
                continue
            if not (np.isfinite(q) and q > 0.):
                self.n_rejected += 1
                continue
            self.sum_leaves[i] = self.min_leaves[i] = q ** self.alpha
            self.max_priority = max(self.max_priority, q)

    def trees(self):
        return build_tree(self.sum_leaves, np.add), build_tree(self.min_leaves, np.minimum)
