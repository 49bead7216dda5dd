"""CPU RESTATEMENT OF THE DEVICE-SIDE NUMERICAL SCHEMES -- TEST INFRASTRUCTURE ONLY.  NOT A PRODUCT PATH.

Nothing here follows a reference file: the reference (Stheno.jl) calls LAPACK `dpotrf` / `dtrsm`
(SURVEY.md App. A) and has no counterpart for *how* the B200 library reaches the same numbers.  These are
plain NumPy statements of three device algorithms, so that their mathematics is pinned on the CPU against
LAPACK / exact arithmetic and the CUDA sources can cite a runnable specification:

  * `oz_slice`, `oz_product`      -- the int8 digit-plane ("Ozaki") product of stheno.jl_b200/csrc/ozaki.cu
                                     (oz_rowscale_kernel, oz_slice_kernel, the 7 grouped int32 accumulators);
  * `oz_groups`, `oz_epilogue_acc`, `oz_update`, `oz_store`, `oz_syrk_tiles`, the packed-layout helpers
                                  -- the same product restated bit for bit as the tcgen05 kernel computes it
                                     (accumulators, epilogue rounding order, the tiles a launch covers), so that
                                     tests/test_gpu_ozaki_exact.py can demand equality of every output bit;
  * `wide_panel_factor`           -- the wide panel phase of api.cu (wide_diag_phase + launch_panel_solve_ozaki):
                                     512 x 512 diagonal block stacked over an identity, right-looking 128-block
                                     elimination, X = A inv(L_512)^T for the rows below;
  * `P2PExchangeModel`            -- the ready / ack / slot-guard protocol of the peer-to-peer column exchange
                                     (api.cu "P2P panel exchange"), as a discrete-event model that can be driven
                                     with arbitrary interleavings.

Only tests/ may import this module.
"""
from __future__ import annotations

import math

import numpy as np

OZ_S = 7            # digit planes
NB = 128


# ---------------------------------------------------------------------------------------------------------
# int8 digit planes
# ---------------------------------------------------------------------------------------------------------
OZ_NO_EXPO = 0x7fffffff   # exponent the slicer stores for a row it maps to zero digits


def oz_row_exponents(P: np.ndarray) -> np.ndarray:
    """Row exponents e_i = ilogb(max|P[i, :]|) + 2 as oz_rowscale_kernel stores them: OZ_NO_EXPO for a row whose
    max is not inside (1e-280, 1e280) (all zero, tiny or huge rows get zero digits and scale 0)."""
    mx = np.max(np.abs(np.asarray(P, dtype=np.float64)), axis=1)
    ok = (mx > 1e-280) & (mx < 1e280)
    return np.where(ok, np.frexp(np.where(ok, mx, 1.0))[1] - 1 + 2, OZ_NO_EXPO).astype(np.int32)


def oz_slice(P: np.ndarray):
    """Digit planes of the rows of P (m x K).  Returns (digits[7, m, K] int8, scale[m] float64).

    Row i is scaled by 2^-e_i with e_i = ilogb(max|P[i, :]|) + 2 (so |x| 2^-e < 0.5), rounded to a 56-bit
    two's-complement fixed-point integer Z = rint(x 2^(55 - e)), and cut into bytes.  Adding the bias
    0x0000808080808080 before cutting re-centres the six low bytes to [-128, 127] (the carry of each ripples
    into the next), so that  Z = sum_p d_p 256^(6 - p)  with every d_p a signed byte.
    scale[i] = 2^(e_i - 31):  x ~= scale * 2^-24 * sum_p d_p 256^(6 - p)  (see oz_product for the pairing).
    """
    P = np.asarray(P, dtype=np.float64)
    m, K = P.shape
    expo = oz_row_exponents(P)
    ok = expo != OZ_NO_EXPO
    e = np.where(ok, expo, 0)
    scale = np.where(ok, np.ldexp(1.0, e - 31), 0.0)
    Z = np.zeros((m, K), dtype=np.int64)
    Z[ok] = np.rint(np.ldexp(P[ok], (55 - e[ok])[:, None])).astype(np.int64)
    Zb = Z + np.int64(0x0000808080808080)
    digits = np.empty((OZ_S, m, K), dtype=np.int8)
    digits[0] = (Zb >> 48).astype(np.int8)
    for p in range(1, OZ_S):
        byte = (Zb >> (8 * (OZ_S - 1 - p))) & 0xFF
        digits[p] = (byte ^ 0x80).astype(np.uint8).view(np.int8)
    return digits, scale


def oz_reconstruct(digits: np.ndarray, scale: np.ndarray) -> np.ndarray:
    """x = scale 2^-24 sum_p d_p 256^(6-p): exact inverse of oz_slice up to the 56-bit rounding."""
    Z = np.zeros(digits.shape[1:], dtype=np.int64)
    for p in range(OZ_S):
        Z += digits[p].astype(np.int64) << (8 * (OZ_S - 1 - p))
    return np.ldexp(Z.astype(np.float64) * scale[:, None], -24)


def oz_product(dA, sA, dB, sB, max_group: int = OZ_S - 1):
    """A B^T from digit planes, as the kernel does it: int32 accumulators G_g = sum_{p+q=g} d_p(A) d_q(B)^T
    for g = 0..6 (pairs with p + q > 6 are dropped), weights 256^(6 - g), then s_i s_j.  Also returns
    max|G_g| so a test can assert the int32 head-room."""
    m, n = dA.shape[1], dB.shape[1]
    acc = np.zeros((m, n), dtype=np.float64)
    gmax = 0
    for g in range(max_group + 1):
        G = np.zeros((m, n), dtype=np.int64)
        for p in range(g + 1):
            q = g - p
            if p < OZ_S and q < OZ_S:
                G += dA[p].astype(np.int64) @ dB[q].astype(np.int64).T
        gmax = max(gmax, int(np.max(np.abs(G))))
        acc += G.astype(np.float64) * math.ldexp(1.0, 8 * (OZ_S - 1 - g))
    # x = s 2^-24 sum d_p 256^(6-p)  ->  x_i x_j = s_i s_j 2^-48 sum_g 256^(12-g) G_g; the kernel's s already
    # absorbs 2^-24 * 256^3 per operand (s = 2^(e-31) = 2^(e-55) 256^3), leaving 256^(6-g)
    return acc * sA[:, None] * sB[None, :], gmax


# ---------------------------------------------------------------------------------------------------------
# the tcgen05 kernel, bit for bit
# ---------------------------------------------------------------------------------------------------------
def oz_groups(dA: np.ndarray, dB: np.ndarray) -> list:
    """The seven int32 accumulators G_g = sum_{p+q=g} d_p(A) d_q(B)^T, g = 0..6, as float64 arrays of exact
    integers.  One float64 BLAS product per group on the int8-valued digits (the pairs of a group are concatenated
    along K): every partial sum is an integer of magnitude below 7 * 512 * 2^14 < 2^53, so the result is exact
    whatever order the BLAS sums in."""
    A = dA.astype(np.float64)
    B = dB.astype(np.float64)
    return [np.concatenate([A[p] for p in range(g + 1)], axis=1) @
            np.concatenate([B[g - p] for p in range(g + 1)], axis=1).T for g in range(OZ_S)]


def oz_epilogue_acc(G: list) -> np.ndarray:
    """The epilogue's fp64 sum: acc = fma((double)G_g, 2^(8(6 - g)), acc) for g = 0..6 in this order.  The product
    is exact, so each step is one rounding of acc + G_g 2^(8(6 - g)), which is what NumPy's addition does."""
    acc = np.zeros_like(G[0])
    for g in range(OZ_S):
        acc = acc + G[g] * math.ldexp(1.0, 8 * (OZ_S - 1 - g))
    return acc


def oz_update(old: np.ndarray, sA: np.ndarray, sB: np.ndarray, acc: np.ndarray) -> np.ndarray:
    """SYRK / plain mode: C = fma(-(s_i s_j), acc, C), with s_i s_j formed first.  s_i s_j is a power of two (or 0),
    so the product with acc is exact and old - s_i s_j acc rounds once like the fma, as long as the product stays
    in the normal range (asserted: below it the fma's single rounding is not what NumPy computes)."""
    s = sA[:, None] * sB[None, :]
    p = s * acc
    assert not np.any((np.abs(p) < np.finfo(np.float64).tiny) & (s != 0) & (acc != 0)), "product below the normal range"
    return old - p


def oz_store(sA: np.ndarray, sB: np.ndarray, acc: np.ndarray) -> np.ndarray:
    """STORE mode (panel solve): X = (s_i s_j) acc."""
    return (sA[:, None] * sB[None, :]) * acc


def packed_offset(Np: int, J: int) -> int:
    """Element offset of block column J in the packed lower layout (sb_common.cuh `Packed`)."""
    return NB * (J * Np - NB * (J * (J - 1) // 2))


def packed_size(Np: int) -> int:
    return packed_offset(Np, Np // NB)


def packed_column(buf: np.ndarray, Np: int, J: int) -> np.ndarray:
    """Writable (Np - J NB) x NB view of block column J (rows J NB .. Np - 1) of a packed buffer."""
    ld = Np - J * NB
    o = packed_offset(Np, J)
    return buf[o:o + NB * ld].reshape(NB, ld).T


def tiled_offset(rb: int, k: int, r: int) -> int:
    """Element (row block rb, column k, row r) of a TILED panel buffer: [row block][128 columns][132 padded rows]."""
    return (rb * NB + k) * (NB + 4) + r


def oz_syrk_tiles(nblk: int, k: int, jlo: int, jhi: int, rank: int = 0, world: int = 1,
                  tile_lo: int = 0, tile_hi: int = 0) -> list:
    """(I, J, h) of the 128 x 64 tiles launch_syrk_ozaki updates, in the kernel's tile order (OzCursor): owned block
    columns J = J0, J0 + world, ... in [max(jlo, k + 1), jhi) with J % world == rank, in each the row blocks I >= J,
    in each both 64-column halves h.  tile_lo / tile_hi select a sub-range of the list; tile_hi <= 0 means its end."""
    jlo, jhi = max(jlo, k + 1), min(jhi, nblk)
    J0 = jlo + (rank - jlo) % world
    tiles = [(I, J, h) for J in range(J0, jhi, world) for I in range(J, nblk) for h in (0, 1)]
    if tile_hi <= 0 or tile_hi > len(tiles):
        tile_hi = len(tiles)
    return tiles[max(tile_lo, 0):tile_hi]


def oz_syrk_update(packed: np.ndarray, Np: int, digits: np.ndarray, scale: np.ndarray) -> np.ndarray:
    """The packed matrix with EVERY block (I >= J) updated as the SYRK instance updates a tile of it:
    C -= P P^T from the digit planes digits[7][Np][K] and scales[Np] of the rows (plane row == matrix row), the
    strictly upper part of the diagonal blocks included.  Combine with oz_apply_tiles for what one launch writes."""
    out = packed.copy()
    for J in range(Np // NB):
        r0 = J * NB
        acc = oz_epilogue_acc(oz_groups(digits[:, r0:], digits[:, r0:r0 + NB]))
        V = packed_column(out, Np, J)
        V[...] = oz_update(V, scale[r0:], scale[r0:r0 + NB], acc)
    return out


def oz_apply_tiles(old: np.ndarray, new: np.ndarray, Np: int, tiles) -> np.ndarray:
    """`old` with the tiles (I, J, h) taken from `new`."""
    out = old.copy()
    for I, J, h in tiles:
        rows, cols = slice((I - J) * NB, (I - J + 1) * NB), slice(h * 64, h * 64 + 64)
        packed_column(out, Np, J)[rows, cols] = packed_column(new, Np, J)[rows, cols]
    return out


# ---------------------------------------------------------------------------------------------------------
# wide panel phase
# ---------------------------------------------------------------------------------------------------------
def wide_panel_factor(Acol: np.ndarray, nq: int = 4, nb: int = NB, product=None):
    """Acol: (m x nq*nb) -- the (already updated) block columns of one outer step, rows from the step's diagonal
    block down.  Returns the same shape holding the Cholesky panel: the lower triangle of the nq*nb diagonal
    block factored, the rows below solved against it.

    Mirrors the device path: the diagonal block is stacked over an identity; for q = 0..nq-1: potrf of block
    (q, q), the rows below (including the identity rows) times inv(L_qq)^T, then the rank-nb updates of the
    later columns.  The identity rows end up holding inv(L_w)^T, and everything below the diagonal block is ONE
    product X = A inv(L_w)^T (`product(A, W)` -> A @ W.T; the device uses int8 digit planes there)."""
    w = nq * nb
    m = Acol.shape[0]
    D = np.zeros((2 * w, w))
    D[:w] = np.tril(Acol[:w])
    for q in range(nq):                       # blocks above the block diagonal are never read
        D[: q * nb, q * nb:(q + 1) * nb] = 0.0
    D[w:] = np.eye(w)
    X = np.zeros_like(D)
    Ld = np.zeros((w, w))
    for q in range(nq):
        c = slice(q * nb, (q + 1) * nb)
        Lqq = np.linalg.cholesky(np.tril(D[c, c]) + np.tril(D[c, c], -1).T)
        inv = np.linalg.solve(Lqq, np.eye(nb))             # explicit inverse, as potrf_inv_kernel
        Ld[c, c] = Lqq
        r = slice((q + 1) * nb, 2 * w)
        X[r, c] = D[r, c] @ inv.T
        for q2 in range(q + 1, nq):
            c2 = slice(q2 * nb, (q2 + 1) * nb)
            r2 = slice(q2 * nb, 2 * w)
            D[r2, c2] -= X[r2, c] @ X[c2, c].T
    for q in range(nq):
        c = slice(q * nb, (q + 1) * nb)
        Ld[(q + 1) * nb:, c] = X[(q + 1) * nb:w, c]
    W = X[w:].T.copy()                                      # inv(L_w), block lower triangular
    out = np.zeros_like(Acol)
    out[:w] = Ld
    if m > w:
        out[w:] = (product or (lambda A, Wm: A @ Wm.T))(Acol[w:], W)
    return out, W


# ---------------------------------------------------------------------------------------------------------
# peer-to-peer column exchange: protocol model
# ---------------------------------------------------------------------------------------------------------
class P2PExchangeModel:
    """Each rank r has an arena: ready[owner], ack[peer] counters and `slots` column slots.  Column k (owner
    k % world) is published into slot k % slots of the owner's arena and pulled by every peer.

    Mirrors the stream structure of the device code (wide_diag_phase): the columns of one outer step (4) are
    exchanged on one stream per owner (owner % 4), concurrently; all of a step's exchanges are joined before
    the next step starts.  The model runs these per-rank, per-stream programs under an arbitrary scheduler and
    asserts the two safety properties the device code relies on:
      (1) a peer only ever reads a slot that holds the column it expects;
      (2) the owner never overwrites a slot before every peer has read its previous occupant.
    Liveness (no deadlock) is asserted by the scheduler finding a runnable operation until all programs end."""

    def __init__(self, world: int, ncols: int, slots: int = 8, base=None, outer: int = 4, guard: bool = True):
        self.world, self.ncols, self.slots, self.outer = world, ncols, slots, outer
        self.ready = [[0] * world for _ in range(world)]      # ready[r][owner]: as seen in r's arena
        self.ack = [[0] * world for _ in range(world)]        # ack[owner][peer]
        self.slot = [[None] * slots for _ in range(world)]    # content: column index
        self.readers_pending = [[set() for _ in range(slots)] for _ in range(world)]
        self.pub = list(base) if base is not None else [0] * world
        if base is not None:                                  # counters of the earlier factorisations are in place
            for r in range(world):
                for p in range(world):
                    self.ack[r][p] = base[r]
                    self.ready[p][r] = base[r]
        self.ord = []
        for k in range(ncols):
            self.pub[k % world] += 1
            self.ord.append(self.pub[k % world])
        self.nsteps = (ncols + outer - 1) // outer
        # prog[r][step] = {stream: [ops]}
        self.prog = [[self._step_program(r, s, guard) for s in range(self.nsteps)] for r in range(world)]
        self.step_of = [0] * world
        self.pc = [dict((xi, 0) for xi in self.prog[r][0]) if self.nsteps else {} for r in range(world)]
        self.got = [[] for _ in range(world)]

    def _step_program(self, r, s, guard):
        streams = {}
        for k in range(s * self.outer, min(self.ncols, (s + 1) * self.outer)):
            owner = k % self.world
            ops = streams.setdefault(owner % 4, [])
            if owner == r:
                kp = k - self.slots
                while kp >= 0 and kp % self.world != r:
                    kp -= self.slots
                if kp >= 0 and guard:
                    ops.append(("guard", self.ord[kp]))
                ops.append(("publish", k))
            else:
                ops.append(("wait", owner, self.ord[k]))
                ops.append(("pull", owner, k))
        return streams

    def _op_ready(self, r, op):
        if op[0] == "guard":
            return all(self.ack[r][p] >= op[1] for p in range(self.world) if p != r)
        if op[0] == "wait":
            return self.ready[r][op[1]] >= op[2]
        return True

    def _pending(self, r):
        """(stream, op) pairs that could execute next on rank r"""
        if self.step_of[r] >= self.nsteps:
            return []
        prog = self.prog[r][self.step_of[r]]
        return [(xi, ops[self.pc[r][xi]]) for xi, ops in prog.items() if self.pc[r][xi] < len(ops)]

    def _execute(self, r, xi, op):
        self.pc[r][xi] += 1
        if op[0] == "publish":
            k = op[1]
            s = k % self.slots
            assert not self.readers_pending[r][s], (
                f"rank {r} overwrites slot {s} (column {self.slot[r][s]}) before {self.readers_pending[r][s]} pulled it")
            self.slot[r][s] = k
            self.readers_pending[r][s] = {p for p in range(self.world) if p != r}
            for p in range(self.world):
                if p != r:
                    self.ready[p][r] = self.ord[k]
        elif op[0] == "pull":
            owner, k = op[1], op[2]
            s = k % self.slots
            assert self.slot[owner][s] == k, f"rank {r} expected column {k} in slot {s} of rank {owner}, found {self.slot[owner][s]}"
            self.readers_pending[owner][s].discard(r)
            self.got[r].append(k)
            self.ack[owner][r] = self.ord[k]
        # join: the next step starts when every stream of this one has drained
        prog = self.prog[r][self.step_of[r]]
        if all(self.pc[r][x] >= len(ops) for x, ops in prog.items()):
            self.step_of[r] += 1
            if self.step_of[r] < self.nsteps:
                self.pc[r] = dict((x, 0) for x in self.prog[r][self.step_of[r]])

    def run(self, rng, bias=None):
        """bias: optional per-rank weights (a small weight makes a rank slow)"""
        while True:
            cand = []
            alive = False
            for r in range(self.world):
                pend = self._pending(r)
                alive = alive or bool(pend)
                cand += [(r, xi, op) for xi, op in pend if self._op_ready(r, op)]
            if not alive:
                return
            assert cand, f"deadlock: steps {self.step_of}"
            if bias is None:
                r, xi, op = cand[rng.integers(len(cand))]
            else:
                w = np.array([bias[c[0]] for c in cand], dtype=float)
                r, xi, op = cand[rng.choice(len(cand), p=w / w.sum())]
            self._execute(r, xi, op)
