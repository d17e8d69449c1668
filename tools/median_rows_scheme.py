"""The shared-work 5x5 median of k_q8_tail (csrc/median_rows.cuh), restated in numpy and checked against a sort.

Scheme (all lists ascending; a "row" S[y] is the sorted 5-pixel segment of image row y inside the window):

    S[y]        = sort5(row y)                                   9 compare-exchanges, used by five outputs
    PP[q]       = merge(S[q], S[q+1])           q even           13 compare-exchanges, used by four outputs
    QQmid[q]    = ranks 7..12 of merge(PP[q], PP[q+2])           24 comparators / 34 min-max ops, used by two outputs
    out[q+1]    = rank 12 of QQ[q] + S[q-1]  =  rank 5 of (QQmid[q], S[q-1])
    out[q+2]    = rank 12 of QQ[q] + S[q+4]  =  rank 5 of (QQmid[q], S[q+4])

The seven smallest elements of the 20-element QQ have at most 6 + 5 = 11 elements of the window below them and the seven
largest at least 13, so only ranks 7..12 can be the median, which is then rank 12 - 7 = 5 of those six and the five
elements of the remaining row:  rank_5(A, B) = max(A0, min(A1,B4), min(A2,B3), min(A3,B2), min(A4,B1), min(A5,B0)).

Per output: 9 + 13/2 + 24/2 comparators and 8 min/max for the final selection (58 min/max ops) against 9 * 1.5 + 54
(111 ops) for an independent 54-comparator selection network per output.

    python tools/median_rows_scheme.py            # verify the networks (0-1 principle) and the scheme (random windows)
    python tools/median_rows_scheme.py --emit     # write depth_completion_mt_b200/csrc/median_rows.cuh
"""
from __future__ import annotations

import itertools
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

SORT5 = [(0, 1), (3, 4), (2, 4), (2, 3), (0, 3), (0, 2), (1, 4), (1, 3), (1, 2)]
# tools/select_network.py --lists 5,5 --ranks all  (Batcher odd-even merge, 13 compare-exchanges)
MERGE55 = [(0, 5), (4, 9), (4, 5), (2, 7), (2, 4), (7, 5), (1, 6), (3, 8), (3, 6), (1, 2), (3, 4), (6, 7), (8, 5)]
MERGE55_OUT = [0, 1, 2, 3, 4, 6, 7, 8, 5, 9]  # wire that holds rank r
# tools/select_network.py --lists 10,10 --ranks 7,8,9,10,11,12  (24 comparators, 34 live min/max ops)
QQMID = [(9, 19), (3, 13), (5, 17), (4, 14), (2, 12), (6, 16), (5, 11), (13, 11), (9, 11), (1, 15), (7, 15), (7, 13), (9, 13),
         (6, 12), (8, 18), (6, 10), (4, 10), (0, 10), (8, 10), (14, 10), (12, 14), (7, 8), (13, 14), (9, 12)]
QQMID_OUT = [7, 8, 9, 12, 13, 14]  # wires that hold ranks 7..12


def check_01(net, outs, sizes, ranks):
    """0-1 principle restricted to inputs whose lists are sorted."""
    n = sum(sizes)
    base = [sum(sizes[:k]) for k in range(len(sizes))]
    for pat in itertools.product(*[range(s + 1) for s in sizes]):
        w = [0] * n
        for k, ones in enumerate(pat):
            for r in range(sizes[k] - ones, sizes[k]):
                w[base[k] + r] = 1
        for i, j in net:
            w[i], w[j] = min(w[i], w[j]), max(w[i], w[j])
        tot = sum(pat)
        for r, o in zip(ranks, outs):
            assert w[o] == (1 if r >= n - tot else 0), (pat, r)


def run(net, v):
    v = list(v)
    for i, j in net:
        a, b = v[i], v[j]
        v[i], v[j] = np.minimum(a, b), np.maximum(a, b)
    return v


def median_rows(win):
    """win: (..., 9, 5) = nine image rows x five pixels; returns the 5x5 medians of the windows of rows 2..6 centred on
    rows 3 and 4 computed with the shared scheme (q = 2: rows 2..5 shared, singles row 1 and row 6) -- i.e. outputs
    centred on rows 3 (rows 1..5) and 4 (rows 2..6)."""
    S = [run(SORT5, [win[..., y, k] for k in range(5)]) for y in range(9)]
    def pp(a, b):
        m = run(MERGE55, a + b)
        return [m[o] for o in MERGE55_OUT]
    qq = run(QQMID, pp(S[2], S[3]) + pp(S[4], S[5]))
    A = [qq[o] for o in QQMID_OUT]
    def final(B):
        m = A[0]
        for i in range(1, 6):
            m = np.maximum(m, np.minimum(A[i], B[5 - i]))
        return m
    return final(S[1]), final(S[6])


def ssa(net, n_in, outs, in_names):
    """Straight-line code of the live part of a comparator network: list of (name, kind, args), result names."""
    live = set(outs)
    keep = []
    for i, j in reversed(net):
        nmin, nmax = i in live, j in live
        if not (nmin or nmax):
            continue
        keep.append((nmin, nmax, i, j))
        live.add(i)
        live.add(j)
    keep.reverse()
    cur = {w: in_names[w] for w in range(n_in)}
    ops = []
    n = 0
    for nmin, nmax, i, j in keep:
        a, b = cur[i], cur[j]
        lo = None
        if nmin:
            lo = f"t{n}"
            ops.append([lo, "mn", [a, b]])
            n += 1
        if nmax:
            hi = f"t{n}"
            ops.append([hi, "other", [a, b, lo]] if nmin else [hi, "mx", [a, b]])
            n += 1
            cur[j] = hi
        if nmin:
            cur[i] = lo
    res = [cur[o] for o in outs]
    # fold single-use chains of the same kind into the three-input forms
    changed = True
    while changed:
        changed = False
        uses = {}
        for _, _, args in ops:
            for a in args:
                uses[a] = uses.get(a, 0) + 1
        for r in res:
            uses[r] = uses.get(r, 0) + 1
        index = {op[0]: k for k, op in enumerate(ops)}
        for k, (name, kind, args) in enumerate(ops):
            if len(args) != 2 or kind == "other":
                continue
            for pos, a in enumerate(args):
                if a in index and uses.get(a, 0) == 1:
                    src = ops[index[a]]
                    if src[1] == kind and len(src[2]) == 2:
                        ops[k] = [name, kind, [src[2][0], src[2][1], args[1 - pos]]]
                        del ops[index[a]]
                        changed = True
                        break
            if changed:
                break
    return ops, res


def emit_fn(name, doc, net, n_in, outs, in_expr, n_out, sig):
    ops, res = ssa(net, n_in, outs, in_expr)
    n2 = sum(1 for o in ops if len(o[2]) == 2 and o[1] != "other")
    n3 = sum(1 for o in ops if len(o[2]) == 3 and o[1] != "other")
    no = sum(1 for o in ops if o[1] == "other")
    lines = [f"// {doc}", f"// {len(net)} comparators -> {n2} two-input + {n3} three-input min/max ops + {no} `other` ops.",
             "template <class Ops, class T>", f"__device__ __forceinline__ void {name}({sig}) {{"]
    for nm, kind, args in ops:
        fn = kind + ("3" if len(args) == 3 and kind != "other" else "")
        lines.append(f"    const T {nm} = ops.{fn}({', '.join(args)});")
    for r in range(n_out):
        lines.append(f"    o[{r}] = {res[r]};")
    lines += ["}", ""]
    return lines


def emit():
    lines = [
        "// median_rows.cuh -- GENERATED by tools/median_rows_scheme.py (networks found by tools/select_network.py); do not edit.",
        "// Building blocks of the shared-work 5x5 median (cv::medianBlur(5), img_completion.cpp:170): merge of two sorted",
        "// fives, and ranks 7..12 of the merge of two sorted tens.  Ops: mn, mx (two-input min / max), mn3, mx3 (three-input),",
        "// and other(a, b, lo) = the element of {a, b} that is not lo = mn(a, b).",
        "#pragma once", "", "namespace dcmt {", ""]
    lines += emit_fn("merge_5_5", "o = merge(a, b), all ascending", MERGE55, 10, MERGE55_OUT,
                     [f"a[{k}]" for k in range(5)] + [f"b[{k}]" for k in range(5)], 10,
                     "const Ops& ops, const T (&a)[5], const T (&b)[5], T (&o)[10]")
    lines += emit_fn("merge_10_10_ranks_7_12", "o = ranks 7..12 of merge(a, b), all ascending", QQMID, 20, QQMID_OUT,
                     [f"a[{k}]" for k in range(10)] + [f"b[{k}]" for k in range(10)], 6,
                     "const Ops& ops, const T (&a)[10], const T (&b)[10], T (&o)[6]")
    lines += [
        "// rank 5 (0-based) of six sorted values a and five sorted values b: the median of 25 once ranks 7..12 of the",
        "// other twenty are known (tools/median_rows_scheme.py)",
        "template <class Ops, class T>",
        "__device__ __forceinline__ T rank5_of_6_5(const Ops& ops, const T (&a)[6], const T (&b)[5]) {",
        "    const T m0 = ops.mx3(a[0], ops.mn(a[1], b[4]), ops.mn(a[2], b[3]));",
        "    const T m1 = ops.mx3(m0, ops.mn(a[3], b[2]), ops.mn(a[4], b[1]));",
        "    return ops.mx(m1, ops.mn(a[5], b[0]));",
        "}", "", "}  // namespace dcmt", ""]
    out = os.path.join(os.path.dirname(HERE), "depth_completion_mt_b200", "csrc", "median_rows.cuh")
    open(out, "w").write("\n".join(lines))
    print("wrote", out)


if __name__ == "__main__":
    check_01(SORT5, range(5), [1] * 5, range(5))
    check_01(MERGE55, MERGE55_OUT, [5, 5], range(10))
    check_01(QQMID, QQMID_OUT, [10, 10], range(7, 13))
    rng = np.random.default_rng(0)
    for hi in (2, 3, 5, 40, 60000):
        win = rng.integers(0, hi, (40000, 9, 5)).astype(np.int64)
        m3, m4 = median_rows(win)
        assert np.array_equal(m3, np.sort(win[:, 1:6].reshape(-1, 25), axis=1)[:, 12]), hi
        assert np.array_equal(m4, np.sort(win[:, 2:7].reshape(-1, 25), axis=1)[:, 12]), hi
    print("networks and scheme verified")
    if "--emit" in sys.argv:
        emit()
