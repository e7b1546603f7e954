"""Deterministic generators for the two large code files BASELINE.json configs 3/4 are quoted on.

Neither the 3GPP TS 38.212 BG1 shift table nor the EN 302 307 Annex B address table exists anywhere in
this image or in the reference repository (SURVEY.md §7 "hard parts"), and there is no network.  What is
generated here is therefore STRUCTURE-MATCHED, not standard-exact:

* ``nr_bg1_like(Z=384)``: a quasi-cyclic code on a 46 x 68 base graph with BG1's block structure —
  4 core rows of weight 19 over 22 information columns + a dual-diagonal 4 x 4 parity core, 42 extension
  rows (weights 3..10, BG1's histogram) each closed by one identity block, 316 blocks in total, the first
  two (high-degree) block columns punctured.  H is 17664 x 26112, nnz 121344, nct 25344 — the sizes
  SURVEY.md §8 lists.  The circulant shifts are seeded-random (4-cycles between block pairs avoided), not
  the 3GPP values.
* ``dvbs2_like_r12()``: an IRA code with DVB-S2's rate-1/2 n=64800 structure — q=90, 36 groups of 360
  degree-8 information columns + 54 groups of degree-3 columns, addresses expanded as
  ``(x + (m mod 360)*q) mod 32400``, staircase parity part.  H is 32400 x 64800, nnz 226799, every check of
  degree 7 (check 0: 6).  The address table is seeded-random with balanced residues, not Annex B's.

Throughput and the roofline depend only on the degree structure; decoder parity is always measured against
the oracle / reference on the SAME file (tests/test_gpu_large_codes.py).  The edge list is written
row-major (row, then column), like the reference's sample file.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
BG1_FILE = os.path.join(HERE, "nr_bg1_like_z384.txt")
DVBS2_FILE = os.path.join(HERE, "dvbs2_like_r12_n64800.txt")

# extension-row weights of the BG1-shaped base graph (42 rows, sum 240 -> 76 + 240 = 316 blocks)
_BG1_EXT_WEIGHTS = [3, 8, 9, 7, 10, 9, 7, 8, 7, 6, 7, 7, 6, 6, 6, 6, 6, 6, 6, 5, 6, 5, 5, 5, 5, 6, 5, 4, 5, 5, 5, 5,
                    4, 5, 5, 5, 4, 4, 4, 3, 6, 4]


def _write(path, n_rows, n_cols, rows, cols, puncture=()):
    order = np.lexsort((cols, rows))
    rows, cols = rows[order], cols[order]
    with open(path, "w") as f:
        if len(puncture):
            f.write("puncture [%d]: %s \n" % (len(puncture), " ".join(str(int(p)) for p in puncture)))
        f.write("\n".join("%d %d" % (r, c) for r, c in zip(rows.tolist(), cols.tolist())))
        f.write("\n")
    return path


def nr_bg1_like(path=BG1_FILE, Z=384, seed=38212):
    rng = np.random.default_rng(seed)
    nb_rows, nb_cols, k_cols = 46, 68, 22
    assert sum(_BG1_EXT_WEIGHTS) + 4 * 19 == 316 and len(_BG1_EXT_WEIGHTS) == 42
    base = {}  # (block row, block col) -> shift
    # core: columns 0 and 1 in every core row (they are the punctured, high-degree columns), 13 more
    # information columns per row chosen so that every information column is covered, dual-diagonal parity
    core_parity = {0: [(22, 1), (23, 0)], 1: [(22, 0), (23, 0), (24, 0)], 2: [(24, 0), (25, 0)], 3: [(22, 1), (25, 0)]}
    for r in range(4):
        n_par = len(core_parity[r])
        n_info = 19 - n_par
        others = list(range(2, k_cols))
        rng.shuffle(others)
        pick = sorted([0, 1] + others[: n_info - 2])
        for c in pick:
            base[(r, c)] = int(rng.integers(0, Z))
        for c, s in core_parity[r]:
            base[(r, c)] = s
    # extension rows: weight-1 identity in column 26 + (r - 4); the rest from the first 26 columns with a
    # bias to columns 0/1 (BG1: column 0 has weight 30, column 1 weight 28)
    for i, w in enumerate(_BG1_EXT_WEIGHTS):
        r = 4 + i
        base[(r, 26 + i)] = 0
        cand = []
        if rng.random() < 0.62:
            cand.append(0)
        if rng.random() < 0.57:
            cand.append(1)
        if not cand:
            cand.append(int(rng.integers(0, 2)))
        rest = [c for c in range(2, 26)]
        rng.shuffle(rest)
        cand = (cand + rest)[: w - 1]
        for c in cand:
            base[(r, c)] = int(rng.integers(0, Z))
    assert len(base) == 316, len(base)

    # remove length-4 cycles between block pairs: rows r1, r2 sharing columns c1, c2 must not satisfy
    # s(r1,c1) - s(r1,c2) + s(r2,c2) - s(r2,c1) == 0 (mod Z); re-draw a free (non-structural) shift otherwise
    structural = {(r, c) for r in range(4) for c, _ in core_parity[r]} | {(4 + i, 26 + i) for i in range(42)}
    by_row = {}
    for (r, c) in base:
        by_row.setdefault(r, []).append(c)
    for _ in range(200):
        bad = 0
        rows_l = sorted(by_row)
        for a in range(len(rows_l)):
            for b in range(a + 1, len(rows_l)):
                r1, r2 = rows_l[a], rows_l[b]
                common = sorted(set(by_row[r1]) & set(by_row[r2]))
                for x in range(len(common)):
                    for y in range(x + 1, len(common)):
                        c1, c2 = common[x], common[y]
                        if (base[(r1, c1)] - base[(r1, c2)] + base[(r2, c2)] - base[(r2, c1)]) % Z == 0:
                            free = [e for e in ((r2, c2), (r2, c1), (r1, c1), (r1, c2)) if e not in structural]
                            if free:
                                base[free[0]] = int(rng.integers(0, Z))
                                bad += 1
        if bad == 0:
            break

    rows, cols = [], []
    z = np.arange(Z)
    for (r, c), s in base.items():
        rows.append(r * Z + z)
        cols.append(c * Z + (z + s) % Z)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    assert rows.size == 121344
    return _write(path, nb_rows * Z, nb_cols * Z, rows, cols, puncture=np.arange(2 * Z))


def dvbs2_like_r12(path=DVBS2_FILE, seed=302307):
    rng = np.random.default_rng(seed)
    n, k, q, M = 64800, 32400, 90, 360
    m = n - k
    degs = [8] * 36 + [3] * 54
    # 450 table entries, every residue mod q exactly 5 times -> every check gets exactly 5 information edges
    residues = np.repeat(np.arange(q), 5)
    for _ in range(1000):
        rng.shuffle(residues)
        ok = True
        hi = rng.integers(0, M, size=residues.size)
        table, p = [], 0  # the addresses of one table row must hit distinct checks
        for d in degs:
            ent = sorted(set(int(residues[p + j] + q * hi[p + j]) for j in range(d)))
            if len(ent) != d:
                ok = False
                break
            table.append(ent)
            p += d
        if ok:
            break
    assert ok
    rows, cols = [], []
    mm = np.arange(M)
    for g, ent in enumerate(table):
        for x in ent:
            rows.append((x + mm * q) % m)
            cols.append(g * M + mm)
    # staircase parity: check j involves parity bits j and j-1
    j = np.arange(m)
    rows.append(j); cols.append(k + j)
    rows.append(j[1:]); cols.append(k + j[1:] - 1)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    assert rows.size == 226799, rows.size
    return _write(path, m, n, rows, cols)


def ensure(which=("bg1", "dvbs2"), directory=HERE):
    """Paths of the code files in `directory`; the missing ones are generated there."""
    out = {}
    for name, default, make in (("bg1", BG1_FILE, nr_bg1_like), ("dvbs2", DVBS2_FILE, dvbs2_like_r12)):
        if name in which:
            path = os.path.join(directory, os.path.basename(default))
            out[name] = path if os.path.exists(path) else make(path)
    return out


if __name__ == "__main__":
    for name, path in ensure(sys.argv[1:] or ("bg1", "dvbs2")).items():
        print(name, path, os.path.getsize(path))
