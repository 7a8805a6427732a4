"""Shared-memory wavefronts per warp-row of pair16_kernel (csrc/pair16.cuh) on the benchmark's resident round, for the
substitution-table layout before and after the bank-conflict-free one (CPU only; DESIGN 4.2).

The reads, their windows and their pair classes are those of `bench.py`'s resident round (bench.make_workload, seed 1000,
bench.windows over the wrapped circular reference).  Reads of one (class, length) are paired in index order, two pairs to a
work item, as the layout kernel does; one warp-row is one DP row of one work item.  Per warp-row the kernel issues

  table  K LDS.64 of the (a, b) entries, one per column of a lane;
  build  4 profile loads (LDS.S16 / LDS.U16) and 2 STS.64 of the next row's table;
  rowoff the profile-row offsets of the next row: 2 LDS.U16 (old), 1 LDS.32 (new);
  shfl   8 SHFL.UP (listed apart: whether the shared-memory counter includes them is not known).

Counting rules: a 64-bit access is served per half-warp (16 lanes); an access of at most 32 bits per warp; either costs the
largest number of distinct 32-bit words (64-bit: bank pairs) that one bank (bank pair) is asked for.

    python scripts/p16_smem_model.py [--reads N]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

G = 16                                        # lanes per pair (P16_G)
MAXL = 256                                    # P16_MAXL
NMAT, PROF_ROW = 31, 8                        # 2 * PSSM_DEPTH + 1 depths; int16 per profile row
PSSM_DEPTH = 15
CLASS_K = [8, 9, 10, 11, 12, 13, 14, 16]      # K of the wide pair classes (128 .. 256 columns)
CLASS_TOP = [128, 144, 160, 176, 192, 208, 224, 256]
CAPTURE_K11 = 366.8e6 / 5.79e6                # profiles/r02j_ncu_pair16_full.md: shared wavefronts / warp-rows of the K = 11 launch


def tab_old(a, b):
    return a * 5 + b


def tab_new(a, b):                            # p16_tab_entry
    return np.where((a < 4) & (b < 4), a * 4 + b, np.where(a == 4, 16 + b, 21 + a))


def inv_old(e):
    return e // 5, e % 5


def inv_new(e):                               # p16_tab_a, p16_tab_b
    e = np.asarray(e)
    return (np.where(e < 16, e >> 2, np.where(e < 21, 4, e - 21)),
            np.where(e < 16, e & 3, np.where(e < 21, e - 16, 4)))


# entry map, its inverse, code of a padding column, wavefronts of the row offsets (old: two LDS.U16 whose pairs hit one bank)
LAYOUTS = {"old": (tab_old, inv_old, 4, 4.0), "new": (tab_new, inv_new, 0, 1.0)}


def p16_class(len1):
    c = np.searchsorted(np.array(CLASS_TOP), len1)
    return np.where(len1 <= 256, c, -1)


def sm_depth(r, L):                           # pssm.c:36-46
    fe = L - (r + 1)
    return np.where(r < PSSM_DEPTH, r, np.where(fe < PSSM_DEPTH, 2 * PSSM_DEPTH - fe, PSSM_DEPTH))


def table_wavefronts(ea):
    """ea: [..., 16] entries of one half-warp's LDS.64 -> wavefronts (distinct entries on the busiest bank pair)"""
    has = np.zeros(ea.shape[:-1] + (32,), bool)
    np.put_along_axis(has, ea, True, axis=-1)
    return (has[..., :16].astype(int) + has[..., 16:]).max(-1)


def workload(n):
    import bench
    ref, bases, off, rc, as_, ae = bench.make_workload(n, seed=1000)
    wrap = ref + ref[:min(len(ref), MAXL)]
    lut = np.full(256, 4, np.int64)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
        lut[ch + 32] = i
    codes = lut[np.frombuffer(wrap.encode(), np.uint8)]
    ws, wl = bench.windows(off, as_, ae, len(wrap))
    return codes, lut[bases], off, rc.astype(np.int64), ws.astype(np.int64), wl.astype(np.int64)


def items_of(L, cls):
    """work items of one class: [n_items, 2 pairs, 2 reads] read ids; reads of one length paired in index order, an empty
    pair slot recomputes the item's first pair, a missing B read rides along as a copy of A"""
    out = []
    for length in np.unique(L[cls]):
        rd = np.flatnonzero(cls & (L == length))
        rd = np.concatenate([rd, rd[-1:]]) if len(rd) % 2 else rd
        pairs = rd.reshape(-1, 2)
        if len(pairs) % 2:
            pairs = np.concatenate([pairs, pairs[-2:-1] if len(pairs) > 1 else pairs])
        out.append(pairs.reshape(-1, 2, 2))
    return np.concatenate(out) if out else np.zeros((0, 2, 2), np.int64)


def model(n):
    codes, rcodes, off, rc, ws, wl = workload(n)
    L = np.diff(off)
    klass = p16_class(wl)
    res = {}
    for ci, K in enumerate(CLASS_K):
        it = items_of(L, klass == ci)
        if len(it) == 0:
            continue
        rows = L[it[:, 0, 0]]                                     # warp-rows of each item
        c = np.arange(G * K).reshape(G, K).T                      # [K, 16]: column of lane l, step j
        row = {}
        for name, (tab, inv, pad, rowoff) in LAYOUTS.items():
            # table loads: per pair, per step j, the 16 lanes' entries
            a = np.where(c < wl[it[..., 0], None, None], codes[np.minimum(ws[it[..., 0], None, None] + c, len(codes) - 1)], pad)
            b = np.where(c < wl[it[..., 1], None, None], codes[np.minimum(ws[it[..., 1], None, None] + c, len(codes) - 1)], pad)
            tl = table_wavefronts(tab(a, b)).sum(axis=(1, 2))        # per item: sum over both half-warps and the K loads
            # build: 4 profile loads per row; the two half-warps read the profile rows of their own reads
            r_all = np.concatenate([np.arange(x) for x in rows])
            item_of_row = np.repeat(np.arange(len(it)), rows)
            depth = sm_depth(r_all, rows[item_of_row])

            def prow(h, s):                                       # profile row (in 16-byte rows) of pair h's read s, each warp-row
                rd = it[item_of_row, h, s]
                return (rc[rd] * NMAT + depth) * 5 + rcodes[off[rd] + r_all]
            bl = 0
            for s in (0, 1):
                w0, w1 = prow(0, s), prow(1, s)
                for t in (0, 1):
                    # both half-warps touch the same words of their 4-word profile rows (the codes of entries t*16 ..):
                    # a conflict is two different rows on the same banks
                    clash = (w0 != w1) & ((w0 - w1) % 8 == 0)
                    bl = bl + np.where(clash, 2, 1)
            tr = (tl * rows).sum() / rows.sum()                      # every row of an item loads the same entries
            row[name] = {"table": tr / K, "table_row": tr, "build_lds": bl.mean(),
                         "build_sts": 4.0, "rowoff": rowoff, "shfl": 8.0}
            v = row[name]
            v["total"] = v["table_row"] + v["build_lds"] + v["build_sts"] + v["rowoff"]
        res[K] = {"items": len(it), "warp_rows": int(rows.sum()), "reads": int((klass == ci).sum()), **row}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reads", type=int, default=200000, help="prefix of the benchmark's 1 M reads to model")
    args = ap.parse_args()
    res = model(args.reads)
    print(f"shared-memory wavefronts per warp-row of pair16_kernel, benchmark resident round ({args.reads} reads)")
    print(f"{'K':>3} {'reads':>7} {'rows':>8} | {'layout':6} {'/LDS.64':>7} {'table':>6} {'build':>6} {'rowoff':>6} {'sts':>4} "
          f"{'total':>6} {'+shfl':>6}")
    for K, r in res.items():
        for name in LAYOUTS:
            v = r[name]
            print(f"{K:>3} {r['reads']:>7} {r['warp_rows']:>8} | {name:6} {v['table']:7.2f} {v['table_row']:6.1f} {v['build_lds']:6.2f} "
                  f"{v['rowoff']:6.1f} {v['build_sts']:4.0f} {v['total']:6.1f} {v['total'] + v['shfl']:6.1f}")
    if 11 in res:
        o = res[11]["old"]
        print(f"K = 11, old layout: {o['total']:.1f} (without shuffles) to {o['total'] + o['shfl']:.1f} (with) wavefronts per "
              f"warp-row; the Nsight Compute capture of the parent code measured {CAPTURE_K11:.1f}")


if __name__ == "__main__":
    main()
