"""numpy restatement of the segmented draw of ``csrc/nprng.cu`` (``invpref_mt_randint``): numpy's legacy
``np.random.randint(0, high, n)`` (MT19937, 1 <= high <= 2^32) computed segment by segment, with segment start states
from GF(2) jumps, per-segment acceptance counts, a prefix sum, compaction and the final state.

The key is a 19 968-bit row vector s (bit k = bit k % 32 of word k // 32); one twist is s -> s A with row k of A the
twist of unit vector e_k.  The library squares A into jump matrices; here a jump of S blocks is S products with A
(squaring a 19 968 x 19 968 matrix is out of reach for numpy), which checks the same linear-map view of the twist."""
from __future__ import annotations

import numpy as np

N, M = 624, 397
MATRIX_A, UPPER, LOWER = np.uint32(0x9908b0df), np.uint32(0x80000000), np.uint32(0x7fffffff)
BITS = N * 32


def _mag(a, b):
    y = (a & UPPER) | (b & LOWER)
    return (y >> np.uint32(1)) ^ np.where((y & np.uint32(1)) != 0, MATRIX_A, np.uint32(0))


def twist(key: np.ndarray) -> np.ndarray:
    """numpy's mt19937_gen on one key [624] or a batch [..., 624] (uint32), in its three dependent sub-ranges."""
    cur = np.asarray(key, dtype=np.uint32)
    nxt = np.empty_like(cur)
    a = N - M                                                    # 227
    nxt[..., :a] = cur[..., M:] ^ _mag(cur[..., :a], cur[..., 1:a + 1])
    nxt[..., a:2 * a] = nxt[..., :a] ^ _mag(cur[..., a:2 * a], cur[..., a + 1:2 * a + 1])
    nxt[..., 2 * a:N - 1] = nxt[..., a:N - 1 - a] ^ _mag(cur[..., 2 * a:N - 1], cur[..., 2 * a + 1:N])
    nxt[..., N - 1] = nxt[..., M - 1] ^ _mag(cur[..., N - 1], nxt[..., 0])
    return nxt


def temper(y: np.ndarray) -> np.ndarray:
    y = np.asarray(y, dtype=np.uint32)
    y = y ^ (y >> np.uint32(11))
    y = y ^ ((y << np.uint32(7)) & np.uint32(0x9d2c5680))
    y = y ^ ((y << np.uint32(15)) & np.uint32(0xefc60000))
    return y ^ (y >> np.uint32(18))


def twist_matrix() -> np.ndarray:
    """A [19968, 624] uint32: row k = twist(e_k), built from unit vectors (the library's mt_unit_twist_kernel)."""
    units = np.zeros((BITS, N), dtype=np.uint32)
    k = np.arange(BITS)
    units[k, k >> 5] = np.uint32(1) << (k & 31).astype(np.uint32)
    return twist(units)


def apply(A: np.ndarray, key: np.ndarray) -> np.ndarray:
    """key A over GF(2): XOR of the rows of A at the set bits of key."""
    bits = np.unpackbits(np.asarray(key, dtype="<u4").view(np.uint8), bitorder="little").astype(bool)
    return np.bitwise_xor.reduce(A[bits], axis=0) if bits.any() else np.zeros(N, dtype=np.uint32)


def _mask(rng: int) -> int:
    return (1 << rng.bit_length()) - 1


def randint(state, high: int, n: int, A: np.ndarray, S: int = 2, G: int = 3):
    """(values int64 [n], new state tuple) of np.random.randint(0, high, n) from ``state`` (np.random.get_state()), as
    the library computes it: rounds of G segments of S blocks with start states by jumps, counts, ranks, compaction;
    whatever is missing after the rounds comes from a sequential tail.  ``A``: twist_matrix()."""
    name, key, pos, has_gauss, gauss = state
    key, pos, high, n = np.asarray(key, dtype=np.uint32), int(pos), int(high), int(n)
    if not 1 <= high <= 1 << 32:
        raise ValueError("high must be in [1, 2^32]")
    out = np.zeros(n, dtype=np.int64)
    if n == 0 or high == 1:
        return out, (name, key.copy(), pos, has_gauss, gauss)
    rng = high - 1
    mask = _mask(rng)
    p = (rng + 1) / (mask + 1)
    final = None

    def block_values(blk, off):
        v = temper(blk).astype(np.int64) & mask
        acc = (v <= rng) & (np.arange(N) >= off)
        return v, acc

    def consume(blk, off, rank):
        """writes the acceptances of one block from rank on; returns (new rank, final state if value n-1 is here)."""
        v, acc = block_values(blk, off)
        idx = np.nonzero(acc)[0]
        take = idx[:max(0, n - rank)]
        out[rank:rank + take.size] = v[take]
        if rank < n <= rank + idx.size:
            return rank + idx.size, (blk.copy(), int(idx[n - rank - 1]) + 1)
        return rank + idx.size, None

    done, base, off = 0, key, pos
    left = int(np.ceil((n / p - (N - pos)) / N))
    while left >= 2 * S:                                         # rounds
        starts = [base]
        for _ in range(G):                                       # s_{g+1} = s_g A^S
            s = starts[-1]
            for _ in range(S):
                s = apply(A, s)
            starts.append(s)
        counts = []
        for g in range(G):                                       # count pass
            blk, o, c = starts[g], off if g == 0 else N, 0
            for b in range(S + 1):
                c += int(block_values(blk, o)[1].sum())
                blk, o = twist(blk), 0
            counts.append(c)
        first = done + np.concatenate([[0], np.cumsum(counts)[:-1]])
        for g in range(G):                                       # write pass
            rank, blk, o = int(first[g]), starts[g], off if g == 0 else N
            for b in range(S + 1):
                if rank >= n:
                    break
                rank, f = consume(blk, o, rank)
                final = f or final
                blk, o = twist(blk), 0
        done += sum(counts)
        base, off = starts[G], N
        left -= G * S
    blk, o, rank = base, off, done                               # sequential tail
    while rank < n:
        rank, f = consume(blk, o, rank)
        final = f or final
        blk, o = twist(blk), 0
    return out, (name, final[0], final[1], has_gauss, gauss)
