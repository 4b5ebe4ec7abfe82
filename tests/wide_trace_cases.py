"""Planted pairs for the wide traceback (swb_wide.cu, wide_trace_kernel) and the host and device rules that place them.

Every case is a read cut from a seeded random reference (one per case group), with a gap, a path end or a max cell put
on a tile, lane-row, band or round edge on purpose.  A case carries a geometry claim, checked on the oracle's own path
before any comparison, so that a builder that misses its seam fails as wrong geometry rather than passing quietly.

Mirrors of the rules the cases rely on:
  pick_kl          swb_wide_host.cu  rows per lane of a read (closed form of the cost rule)
  tile             swb_wide.cu       tile coordinates of a cell: lane-row T, lane t, band, step, block, tile row / column
  grouping         swb_wide.cu       launch_trace_kl: cluster / warp / thread from the max-cell count of a launch
  cluster_c        swb_wide.cu       launch_trace_pipe: CTAs per cell, 3 / 2 / 1 while every cluster is resident
  wide_shape, hsr  swb_wide.cu       the CTA-wide corridor shape (16 x 8 for low score density) and its round length
  tile_trace_ok    swb_trace_tile.cu byte tiles, or int32 tiles for large scores
"""
import random

from tests.helpers import OP_ALIGN, OP_DEL, OP_INS

WL = WCB = 32                                       # lanes per band, steps per block
KL_READS = {8: (60, 256), 16: (1025, 1536), 32: (1537, 2100)}   # read lengths of each class used by the gap cases
FILLER = "Z"                                        # symbol of the filler tie set: in no planted sequence
JUNK = "N"                                          # inserted / leading read bases: in no reference
GAP_REF = "X"                                       # deleted reference bases: in no read


# ---- mirrors -----------------------------------------------------------------------------------------------------

def pick_kl(m):
    """Rows per lane of a read of m rows: 8 up to 256 rows, 16 for 257-512 and 1025-1536, 32 otherwise."""
    if m <= 256:
        return 8
    return 16 if 257 <= m <= 512 or 1025 <= m <= 1536 else 32


def pick_kl_cost(m):
    """The cost rule of swb_wide_host.cu itself: bands times (3 KL + 25), the larger KL on a tie."""
    best = best_cost = 0
    for kl in (8, 16, 32):
        cost = -(-m // (WL * kl)) * (3 * kl + 25)
        if not best or cost <= best_cost:
            best, best_cost = kl, cost
    return best


def tile(i, j, kl):
    """Tile coordinates of cell (i, j) (1-based): lane-row T, lane t, band, step, block, tile row r, tile column c."""
    T = (i - 1) // kl
    t = T % WL
    step = j - 1 + t
    return {"T": T, "t": t, "band": T // WL, "step": step, "block": step // WCB, "r": i - T * kl, "c": step % WCB + 1}


def cell_at(kl, T, r, block, c):
    """The cell at tile row r, tile column c of the tile (lane-row T, block)."""
    return T * kl + r, block * WCB + c - T % WL


def grouping(n_cells, sm):
    return "cluster" if n_cells <= sm else ("warp" if n_cells < 256 * sm else "thread")


def cluster_c(n_cells, sm):
    c = 3
    while c > 1 and n_cells * c > sm:
        c -= 1
    return c


def tile_trace_ok(match, mismatch, gap):
    if gap >= 0:
        return False
    return 2 * (max(match, mismatch, 0) - gap) + max(abs(match), abs(mismatch)) < 250


def wide_shape(h0, match, i0, j0):
    return 2 * h0 < max(match, 1) * min(i0, j0)


def hsr(h0, match, i0, j0):
    """Lane-rows per round of the CTA-wide traceback."""
    return 16 if wide_shape(h0, match, i0, j0) else 32


def trace_kernel(kl, group, byte):
    """The wide_trace_kernel<KL, NT, G, BYTE> a launch of this grouping runs (the int32 tiles have no cluster mode)."""
    if not byte:
        return rf"\bwide_trace_kernel<{kl}, 32, {1 if group == 'thread' else 32}, false>"
    if group == "cluster":
        return rf"\bwide_trace_kernel<{kl}, 256, 256, true>"
    return rf"\bwide_trace_kernel<{kl}, {64 if kl >= 32 else 128}, {32 if group == 'warp' else 1}, true>"


# ---- the oracle's path --------------------------------------------------------------------------------------------

class Path:
    """The walk of max cell k of an oracle_arrays result, in walk order (from the max cell back to the beginning):
    moves [(i, j, op, hcur)] -- the cell the walker stands on, the move it takes there and that cell's score -- and
    the cell it stops on."""

    def __init__(self, exp, scores, read, ref, k=0):
        match, mismatch, gap = scores
        i, j = (int(v) for v in exp["cells"][k])
        a, b = int(exp["aln_off"][k]), int(exp["aln_off"][k + 1])
        self.i0, self.j0, self.h0 = i, j, exp["score"]
        self.moves = []
        h = self.h0
        for op in exp["ops"][a:b][::-1]:
            self.moves.append((i, j, int(op), h))
            if op == OP_ALIGN:
                h -= match if read[i - 1] == ref[j - 1] else mismatch
                i, j = i - 1, j - 1
            else:
                h -= gap
                i, j = (i - 1, j) if op == OP_INS else (i, j - 1)
        self.end = (i, j, h)

    def gap_runs(self):
        """(op, i, j, length) of each run of one gap op, at the run's first move in walk order."""
        runs = []
        for k, (i, j, op, _) in enumerate(self.moves):
            if op == OP_ALIGN:
                continue
            if runs and k > 0 and self.moves[k - 1][2] == op and runs[-1][4] == k - 1:
                runs[-1][3] += 1
                runs[-1][4] = k
            else:
                runs.append([op, i, j, 1, k])
        return [tuple(r[:4]) for r in runs]

    def diag_runs(self):
        """(i, j, length, hcur) of each run of alignment moves, at its first move in walk order."""
        runs, k = [], 0
        while k < len(self.moves):
            if self.moves[k][2] != OP_ALIGN:
                k += 1
                continue
            s = k
            while k < len(self.moves) and self.moves[k][2] == OP_ALIGN:
                k += 1
            i, j, _, h = self.moves[s]
            runs.append((i, j, k - s, h))
        return runs

    def round_of(self, i, kl, match):
        """Round of the CTA-wide traceback that walks the cells of row i."""
        T00 = (self.i0 - 1) // kl
        return (T00 - (i - 1) // kl) // hsr(self.h0, match, self.i0, self.j0)


class WrongGeometry(AssertionError):
    pass


def claim(ok, case, what):
    if not ok:
        raise WrongGeometry(f"wrong geometry: {case.name}: {what}")


# ---- cases --------------------------------------------------------------------------------------------------------

class Case:
    def __init__(self, name, read, check):
        self.name, self.read, self.check = name, read, check

    def assert_geometry(self, exp, scores, ref, kl):
        claim(exp["score"] > 0 and exp["count"] >= 1, self, f"score {exp['score']}")
        claim(pick_kl(len(self.read)) == kl, self, f"read of {len(self.read)} rows is not in class KL = {kl}")
        for k in range(exp["count"]):
            self.check(self, Path(exp, scores, self.read, ref, k), exp, k)


def flank(L, scores):
    """Bases of a flank that out-scores a gap of L."""
    match, _, gap = scores
    return -(-(-gap * L + 1) // match) + 64              # and out-scores a random gapped alignment


class Group:
    """Planted reads against one seeded reference of n bases (n % 32 != 31: the last block is partial)."""

    def __init__(self, name, kl, n, scores, seed):
        self.name, self.kl, self.scores = name, kl, scores
        self.rng = random.Random(seed)
        self.ref = "".join(self.rng.choice("ACGT") for _ in range(n))
        self.n0 = n
        self.cases = []

    def add(self, name, read, check):
        self.cases.append(Case(f"{self.name}/{name}", read, check))

    # a single gap whose first move (walk order) is at cell (gi, gj): k junk rows, a flank, the gap, a flank, junk rows.
    # Inserted read bases are JUNK; deleted reference bases are a stretch of GAP_REF, appended to the reference for
    # this case -- neither can be aligned to anything, so the gap can neither slide nor be broken up.
    def gap(self, name, op, L, gi, gm, m, fl=None, extra=None):
        """gm: the wanted first-move column modulo 32; fl: the flank length (default flank(L)); extra: a further
        claim on the path.  Returns the case's column."""
        fl = fl or flank(L, self.scores)
        x0 = fl
        k = gi - x0 - (L if op == OP_INS else 0)
        tail = m - k - x0 - fl - (L if op == OP_INS else 0)
        if k < 0 or tail < 0:
            return None
        ref = self.ref
        if op == OP_INS:                                    # from the reference's leading random bases
            gj = x0 + 8
            gj += (gm - gj) % WCB
            assert gj + fl <= self.n0
            s = gj - x0
            read = JUNK * k + ref[s:gj] + JUNK * L + ref[gj:gj + fl] + JUNK * tail
            end = (gi + fl, gj + fl)
        else:
            gj = len(ref) + x0 + 8 + L
            gj += (gm - gj) % WCB
            pre = "".join(self.rng.choice("ACGT") for _ in range(gj - L - len(ref)))
            ref += pre + GAP_REF * L + "".join(self.rng.choice("ACGT") for _ in range(fl + 8))
            read = JUNK * k + ref[gj - L - x0:gj - L] + ref[gj:gj + fl] + JUNK * tail
            end = (gi + fl, gj + fl)
        self.ref = ref
        assert len(read) == m

        def check(case, p, exp, kk):
            runs = p.gap_runs()
            claim(runs == [(op, gi, gj, L)], case, f"gap runs {runs[:4]}, planted {(op, gi, gj, L)}")
            claim((p.i0, p.j0) == end and p.end[2] == 0, case, f"max cell {(p.i0, p.j0)}, end {p.end}")
            if extra:
                extra(case, p)
        self.add(name, read, check)
        return gj


def _tile_positions(kl):
    """(name, r, c) of a gap's first move inside its tile."""
    return [("r1c1", 1, 1), ("r1c32", 1, 32), (f"r{kl}c1", kl, 1), (f"r{kl}c32", kl, 32), ("interior", kl // 2 + 1, 17)]


GAP_LENGTHS = lambda kl: sorted({1, 2, kl - 1, kl, kl + 1, 31, 32, 33, 64, 65, 127, 128, 129, 257})


def gap_group(kl, scores, seed=0):
    """Single insertions and deletions of every length, their first move at a tile corner, inside a tile, on the lane
    31 -> lane 0 jump of a band seam, or one row either side of it.  Lengths rotate through the positions, so every
    length and every position is planted for both ops (KL = 8 reads are one band: no seam)."""
    m_lo, m_hi = KL_READS[kl]
    g = Group(f"gaps-kl{kl}-{scores}", kl, 2 * flank(32 * kl + 1, scores) + 69, scores, seed + kl)   # insertions' bases
    bh, rng = WL * kl, g.rng
    positions = [(nm, r, c, None) for nm, r, c in _tile_positions(kl)]
    if kl > 8:
        positions += [("seam-jump", 1, 32, 0), ("seam-above", kl, 16, -1), ("seam-below", 2, 16, 0)]
    for op, ev in ((OP_INS, "ins"), (OP_DEL, "del")):
        for idx, L in enumerate(GAP_LENGTHS(kl)):
            fl = flank(L, scores)
            need = 2 * fl + (L if op == OP_INS else 0)
            if need > m_hi:
                continue                                    # no read of this class holds the gap and its flanks
            for attempt in range(len(positions)):
                nm, r, c, seam = positions[(idx + 3 * (op == OP_DEL) + attempt) % len(positions)]
                m = rng.randint(max(m_lo, need), m_hi)
                lo, hi = fl + (L if op == OP_INS else 0), m - fl
                if seam is None:
                    Ts = [T for T in range(m // kl + 1) if lo <= T * kl + r <= hi]
                else:
                    Ts = [B * WL + seam for B in range(1, -(-m // bh)) if lo <= (B * WL + seam) * kl + r <= hi]
                if not Ts:
                    continue
                T = rng.choice(Ts)
                g.gap(f"{ev}{L}@{nm}", op, L, T * kl + r, (c - T % WL) % WCB, m)
                break
    match = scores[0]

    # an insertion longer than a round of the CTA-wide traceback (HSr lane-rows): the round changes inside the gap
    L = 16 * kl + 1 if kl == 8 else 32 * kl + 1
    if 2 * flank(L, scores) + L <= m_hi:
        def crosses(case, p, L=L):
            _, gi, _, _ = p.gap_runs()[0]
            claim(p.round_of(gi, kl, match) != p.round_of(gi - L, kl, match), case, "the insertion stays in one round")
        g.gap(f"ins{L}@round-edge", OP_INS, L, m_hi - flank(L, scores) - 3, 5, m_hi, extra=crosses)

    # deletions wider than the 4-block corridor (128 columns) near the top of a long read: few rows above the max
    # cell keep min(i0, j0) small, so the path takes the 32 x 4 shape (at KL = 16 and 32 the leading junk rows of the
    # other gap cases make it 16 x 8)
    if kl > 8:
        for L in (129, 257):
            fl = flank(L, scores) + 96

            def narrow(case, p, L=L):
                claim(not wide_shape(p.h0, match, p.i0, p.j0) and L > 4 * WCB, case, "the 16 x 8 corridor")
            g.gap(f"del{L}@narrow", OP_DEL, L, fl + kl // 2, 17, m_hi, fl=fl, extra=narrow)
    return g


def _substring(g, name, m, s, k=0, check=None):
    """Read = k junk bases + ref[s : s + m - k]: a pure diagonal from (m, s + m - k) back to (k + 1, s + 1)."""
    read = JUNK * k + g.ref[s:s + m - k]

    def base_check(case, p, exp, kk):
        claim((p.i0, p.j0) == (m, s + m - k), case, f"max cell {(p.i0, p.j0)}")
        claim(not p.gap_runs() and p.end[:2] == (k, s), case, f"path end {p.end}, gaps {p.gap_runs()[:3]}")
        if check:
            check(case, p, exp, kk)
    g.add(name, read, base_check)


def ends_group(kl, scores, seed=0):
    """Path ends, max cells, rounds, ties and drift of one class."""
    m_lo, m_hi = KL_READS[kl]
    match, _, gap = scores
    g = Group(f"ends-kl{kl}-{scores}", kl, {8: 805, 16: 1829, 32: 2597}[kl], scores, seed + 100 + kl)
    n, rng, bh = len(g.ref), g.rng, WL * kl
    big = max(abs(match), abs(scores[1]))
    mid = (m_lo + m_hi) // 2

    # path ends: the beginning on column 1 / row 1 (the exits toward row 0 / column 0), a score of 0 inside a tile and
    # on its boundary row
    _substring(g, "begin-r1c1", mid, 0)
    _substring(g, "begin-row1", mid + 3, 37)
    _substring(g, "begin-col1", mid - 1, 0, k=45)
    T = 3
    for nm, r, c in (("zero-interior", kl // 2, 9), ("zero-edge", 1, 9), ("zero-c1", kl // 2, 1)):
        k = T * kl + r - 1                                  # first aligned row T kl + r, column at tile column c
        s = cell_at(kl, T, r, 2, c)[1] - 1

        def chk(case, p, exp, kk, r=r, c=c):
            ti = tile(p.moves[-1][0], p.moves[-1][1], kl)
            claim((ti["r"], ti["c"]) == (r, c) and p.end[2] == 0, case, f"last cell {ti}, end {p.end}")
        _substring(g, nm, mid, s, k=k, check=chk)

    # the path begins right after a mismatch cell of score 0 whose diagonal predecessor scores |mismatch| (a match, then
    # a mismatch: match = -2 mismatch), and its first cell is the first of a tile the thread walker enters, so its run
    # of up to four diagonal moves starts there: only the walker's check that the next cell is positive ends the path
    if match == -2 * scores[1]:
        T = 5
        k = T * kl + kl - 4                                 # rows k + 1 .. k + 3: match, junk, junk; row k + 4 = T kl + kl
        s = cell_at(kl, T, kl, 3, 9)[1] - 1                 # the first aligned cell (k + 4, s + 1): tile row KL, column 9
        read = JUNK * k + g.ref[s - 3] + JUNK * 2 + g.ref[s:s + mid - k - 3]

        def chk(case, p, exp, kk, k=k, s=s):
            ti = tile(k + 4, s + 1, kl)
            claim(p.end == (k + 3, s, 0) and (ti["r"], ti["c"]) == (kl, 9), case, f"path end {p.end}, first cell {ti}")
        g.add("begin-after-mismatch", read, chk)

    # the last diagonal run (walk order) of R matches begins at hcur = R * match, on both sides of 32 * big
    for R in (31, 32, 33):
        s, k = rng.randint(40, 300), 24
        read = JUNK * k + g.ref[s:s + R] + JUNK * 2 + g.ref[s + R:s + mid - k - 2]

        def chk(case, p, exp, kk, R=R):
            last = p.diag_runs()[-1]
            claim(last[2] == R and last[3] == R * match and p.end[2] == 0, case, f"last run {last}, end {p.end}")
            claim((last[3] > 32 * big) == (R > 32 and match == big), case, "hcur against 32 * big")
        g.add(f"last-run{R}", read, chk)

    # max cells: in block 0 with j <= 32; rows with m % KL = 0, 1, KL - 1; column n (partial last block); a band's
    # first and last row
    m0 = next(x for x in range(m_lo, m_hi + 1) if ((x - 1) // kl) % WL <= 8)
    j = 32 - ((m0 - 1) // kl) % WL                          # step j - 1 + t = 31: the last column of block 0
    read = JUNK * (m0 - j) + g.ref[:j]

    def chk(case, p, exp, kk, j=j):
        ti = tile(p.i0, p.j0, kl)
        claim(ti["block"] == 0 and p.j0 == j <= 32 and p.end[:2] == (m0 - j, 0), case, f"max cell tile {ti}, end {p.end}")
    g.add("block0", read, chk)
    for rm in (0, 1, kl - 1):
        m = next(x for x in range(mid, m_hi + 1) if x % kl == rm)
        _substring(g, f"m%kl={rm}", m, 11, check=lambda case, p, e, kk, rm=rm: claim(p.i0 % kl == rm, case, "row"))
    assert (n + WL - 1) % WCB != 0
    _substring(g, "col-n", mid + 5, n - (mid + 5), check=lambda case, p, e, kk: claim(p.j0 == n, case, "column n"))
    for B in range(1, -(-m_hi // bh)):
        for nm, m in (("band-last-row", B * bh), ("band-first-row", B * bh + 1)):
            if m_lo <= m <= m_hi:
                _substring(g, f"{nm}{B}", m, 23, check=lambda case, p, e, kk, m=m: claim(p.i0 == m, case, "max row"))
    if kl == 8:
        _substring(g, "band-last-row0", 256, 23)

    # rounds: pure diagonals whose last cell lies in round R, on its first and on its last lane-row
    T00 = (m_hi - 1) // kl
    for R in range(0, 5):
        for nm, Tend in (("mid", T00 - 32 * R - 16), ("first", T00 - 32 * R), ("last", T00 - 32 * R - 31)):
            k = Tend * kl + 3
            if Tend < 0 or m_hi - k < 40:                   # too few aligned rows to be the pair's best
                continue

            def chk(case, p, exp, kk, R=R, Tend=Tend):
                T = (p.moves[-1][0] - 1) // kl
                claim(T == Tend and p.round_of(p.moves[-1][0], kl, match) == R, case, f"ends on lane-row {T}")
            _substring(g, f"round{R}-{nm}", m_hi, 5, k=k, check=chk)

    # rounds 3 and 4 within the class's read lengths: a read whose every other base is junk has a low score density,
    # takes the 16 x 8 corridor and so rounds of 16 lane-rows
    if kl > 8:
        for R in (3, 4):
            for nm, Tend in (("mid", T00 - 16 * R - 8), ("first", T00 - 16 * R), ("last", T00 - 16 * R - 15)):
                k = Tend * kl + 3
                if Tend < 0:
                    continue
                a = m_hi - k - (1 - (m_hi - k) % 2)                # an odd count: the aligned part starts and ends on a base
                read = JUNK * k + "".join(ch if x % 2 == 0 else JUNK for x, ch in enumerate(g.ref[5:5 + a]))
                read += JUNK * (m_hi - len(read))

                def chk(case, p, exp, kk, R=R, Tend=Tend):
                    T = (p.moves[-1][0] - 1) // kl
                    claim(hsr(p.h0, match, p.i0, p.j0) == 16, case, "the 32 x 4 corridor")
                    claim(T == Tend and p.round_of(p.moves[-1][0], kl, match) == R, case, f"ends on lane-row {T}")
                g.add(f"round{R}-{nm}-sparse", read, chk)

    # ties: a run of copies of the base before an insertion, so that the copies can be aligned at any of its places;
    # the run straddles a band seam (a lane-row edge for KL = 8)
    seam_row = bh if kl > 8 else 12 * kl
    for L in (1, 3, 9):
        x, s = 60, rng.randint(5, 300)
        k = seam_row - 1 - x                                # inserted rows seam_row .. seam_row + L - 1
        hp = g.ref[s + x - 1]
        read = JUNK * k + g.ref[s:s + x] + hp * L + g.ref[s + x:s + x + 60]
        read += JUNK * (mid - len(read))

        def chk(case, p, exp, kk, L=L):
            runs = p.gap_runs()
            claim(len(runs) == 1 and runs[0][0] == OP_INS and runs[0][3] == L, case, f"gaps {runs}")
            top = runs[0][1] - L                            # the inserted rows are top + 1 .. top + L
            claim(abs(top + 1 - seam_row) <= 8, case, f"insertion rows {top + 1}..{top + L}, seam row {seam_row}")
        g.add(f"tie-hp{L}", read, chk)

    # drift: a train of 1-3-base indels every 10-40 bases; a staircase of 16-40-base insertions and deletions
    def indels(lo_len, hi_len, lo_gap, hi_gap, m, alternate):
        s = rng.randint(5, 40)
        out, pos, ins = [], s, True
        while len(out) < m and pos < n:
            seg = rng.randint(lo_gap, hi_gap)
            out.append(g.ref[pos:pos + seg])
            pos += seg
            L = rng.randint(lo_len, hi_len)
            ins = (not ins) if alternate else rng.random() < 0.5
            if ins:
                out.append(JUNK * L)
            else:
                pos += L
        return "".join(out)[:m]

    def min_runs(count, min_len, shape):
        def chk(case, p, exp, kk):
            runs = [r for r in p.gap_runs() if r[3] >= min_len and (min_len == 1 or r[0] == OP_INS)]
            claim(len(runs) >= count, case, f"{len(runs)} gap runs of {min_len}+")
            claim(shape is None or wide_shape(p.h0, match, p.i0, p.j0) == shape, case, f"wide_shape {not shape}")
        return chk
    g.add("indel-train", indels(1, 3, 10, 40, m_hi, False), min_runs(m_hi // 60, 1, False))
    g.add("staircase", indels(16, 40, 30, 60, m_hi, True), min_runs(m_hi // 200, 16, None))
    # low score density: every other base replaced by junk takes the 16 x 8 corridor
    s = 17
    g.add("wide-shape", "".join(ch if x % 2 == 0 else JUNK for x, ch in enumerate(g.ref[s:s + mid])), min_runs(0, 1, True))
    return g


# score sets and the groups each runs: the whole catalogue with cheap gaps (long gaps stay optimal), a part of it with
# the others -- about 1.5e9 oracle cells in all, both tie rules
SCORE_SETS = {(5, -3, -1): (8, 16, 32), (5, -3, -4): (8,), (2, -1, -2): (8,), (60, -30, -40): (8,)}


def groups(kl, scores):
    return [gap_group(kl, scores), ends_group(kl, scores)]


def all_groups():
    return [g for scores, kls in SCORE_SETS.items() for kl in kls for g in groups(kl, scores)]
