"""How many column bytes the pruned column pass needs once each query's final k-th score is known (CPU, counts only).

The pruned column pass (slg_columns_ordered_kernel) skips a 512-doc block of a query when the sum of its columns' exact
block maxima (col_tmax, slot order) plus `extra` cannot reach the query's k-th score.  The earlier the k-th score is
close to final, the more blocks are skipped.  This tool takes the final k-th score of every query from the oracle's
exact top-k and counts the blocks whose bound still reaches

    final k-th * 0.99998 - extra * 1.00002

which is what a pass that finds the final k-th before it reads the bulk would have to read.  It sets that against the
blocks of the queries' whole doc range (what a pass reads that skips nothing).

Which queries enter the pass: the loader's columns (`dense_den`, df >= dense_min_df) and the engine's colq_prune rule
applied with the FINAL k-th score (the scan's k-th is at most that, so the real set can only be larger).  The queries
made only of column terms enter whatever the scan found and are reported on their own: that is the lower bound.

    python tools/colpass_headroom.py --docs 2000000 > profiles/r5_colpass_headroom.txt
"""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K1, B = 0.9, 0.4
F = np.float32


def unit_scores(tf: np.ndarray, df: int, doc_len: np.ndarray, avgdl: float, docs: float) -> np.ndarray:
    """oracle score_tf with weight 1, in f32 (query/wand.rs:269-286)"""
    idf = F(max(np.log(F((F(docs) - F(df) + F(0.5)) / (F(df) + F(0.5)))), F(0.0)) + F(1.0))
    norm_dl = doc_len.astype(F) / F(avgdl)
    denom = tf.astype(F) + F(K1) * (F(1.0) - F(B) + F(B) * norm_dl)
    return (idf * (tf.astype(F) * F(K1 + 1.0)) / np.maximum(denom, F(1e-6))).astype(F)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--docs", type=int, default=2_000_000)
    ap.add_argument("--vocab", type=int, default=1_000_000)
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--k", type=int, default=11)
    ap.add_argument("--dense-den", type=int, default=24)
    ap.add_argument("--dense-min-df", type=int, default=256)
    args = ap.parse_args()

    from oracle import slo
    from searchlite_b200 import synth
    t0 = time.time()
    seg = synth.generate_segment(synth.CorpusSpec(n_docs=args.docs, vocab=args.vocab, seed=20260101), "cpu")
    qb = synth.generate_queries(args.queries, args.vocab, seed=20260102)
    terms = [[int(t) for t in qb.terms["term_id"][qb.term_off[q]:qb.term_off[q + 1]]] for q in range(qb.n_queries)]
    t_gen = time.time() - t0
    o = slo.OracleIndex(seg)
    hits, counts = o.search_batch(qb, args.k, "bm25", threads=slo.max_threads())
    t_oracle = time.time() - t0 - t_gen
    avgdl, n = o.avgdl, seg.doc_count
    offs = np.asarray(seg.term_offsets, dtype=np.int64)
    df = np.diff(offs)
    lens = np.asarray(seg.field_lengths)

    # the loader's columns: df * dense_den >= N and df >= dense_min_df, densest first (ties to the lower term id)
    cand = np.nonzero((df >= args.dense_min_df) & (df * args.dense_den >= n))[0]
    cand = cand[np.lexsort((cand, -df[cand]))]
    is_col = np.zeros(len(df), dtype=bool)
    is_col[cand] = True
    n_blocks = (n + 511) // 512
    needed = sorted({t for q in terms for t in q})
    tmax, ub = {}, {}
    for t in needed:
        d = np.asarray(seg.post_docs[offs[t]:offs[t + 1]]).astype(np.int64)
        s = unit_scores(np.asarray(seg.post_tfs[offs[t]:offs[t + 1]]), int(df[t]), lens[d], avgdl, float(n))
        ub[t] = F(s.max()) if len(s) else F(0.0)
        if is_col[t]:
            m = np.zeros(n_blocks, dtype=F)
            np.maximum.at(m, d >> 9, s)
            tmax[t] = m

    kth = np.array([hits[q, args.k - 1]["score"] if counts[q] == args.k else np.nan for q in range(len(terms))], dtype=F)
    rows = []  # (query, all-column, ncol, open blocks)
    for q, tl in enumerate(terms):
        cols = [t for t in tl if is_col[t]]
        if not cols:
            continue
        spars = [t for t in tl if not is_col[t]]
        slots = spars + cols  # slot order: terms without a column first, then those with one, each in query order
        thr = kth[q]
        extra = F(0.0)
        if not np.isnan(thr):
            # colq_prune against the final k-th: priority = larger bound first, ties to the lower slot
            u = [ub[t] for t in slots]
            ess_col = False
            for i, t in enumerate(slots):
                pre = F(0.0)
                for j in range(len(slots)):
                    if u[j] < u[i] or (u[j] == u[i] and j >= i):
                        pre = F(pre + u[j])
                ne = F(pre * F(1.00002)) < thr
                if is_col[t]:
                    ess_col = ess_col or not ne
                elif ne:
                    extra = F(extra + u[i])
            if not ess_col:
                continue
        bound = np.zeros(n_blocks, dtype=F)
        for t in cols:
            bound = (bound + tmax[t]).astype(F)  # (__fadd_rn(bound, __fmul_rn(tmax, 1.0)))
        if np.isnan(thr):
            opened = int(np.count_nonzero(bound))
        else:
            cf = F(F(thr * F(0.99998)) - F(extra * F(1.00002)))
            cut = cf.view(np.uint32) if cf > 0 else np.uint32(0)
            opened = int(np.count_nonzero((bound != 0) & (bound.view(np.uint32) >= cut)))
        rows.append((q, not spars, len(cols), opened))

    def report(sel, name):
        r = [x for x in rows if sel(x)]
        blocks = sum(n_blocks for _ in r)
        opened = sum(x[3] for x in r)
        bytes_all = sum(n_blocks * x[2] * 2048 for x in r)
        bytes_open = sum(x[3] * x[2] * 2048 for x in r)
        print(f"{name}: n_colq {len(r)}, (query, block) pairs {blocks}, open at the final k-th {opened} "
              f"({opened / max(blocks, 1):.4f}); column bytes of the whole range {bytes_all / 1e9:.3f} GB, "
              f"of the open blocks {bytes_open / 1e9:.4f} GB ({bytes_open / max(bytes_all, 1):.4f})")
        if r:
            top = sorted(r, key=lambda x: -x[3])[:5]
            print(f"  largest open-block counts per query: " + ", ".join(f"q{x[0]} {x[3]} of {n_blocks} ({x[2]} col)" for x in top))

    print(f"# colpass_headroom: {n} docs, vocab {args.vocab}, {len(terms)} queries (seed 20260102), k {args.k}, "
          f"dense_den {args.dense_den}; {len(cand)} columns; {n_blocks} blocks of 512 docs")
    print(f"# corpus {t_gen:.0f} s, oracle top-k (bm25, exact) {t_oracle:.0f} s on the CPU; queries without k hits: "
          f"{int(np.isnan(kth).sum())}")
    print(f"# queries naming >= 1 column: {sum(1 for tl in terms if any(is_col[t] for t in tl))}; "
          f"only column terms: {sum(1 for tl in terms if all(is_col[t] for t in tl))}")
    report(lambda x: x[1], "all-column queries (enter the pass whatever the scan found; lower bound)")
    report(lambda x: True, "queries colq_prune keeps at the final k-th (mixed ones with extra at the final k-th)")


if __name__ == "__main__":
    main()
