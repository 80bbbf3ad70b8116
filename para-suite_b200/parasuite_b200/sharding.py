"""Multi-GPU partitioning of the hot path (SURVEY.md 8(e)).

  * error profile : read batches to ranks, one sum all-reduce of the int64 count vector (exact: the outputs are
    commutative integer sums, Java's int wrap-around is applied after the reduction).
  * T>C pileup    : contiguous read ranges (genome regions) to ranks, no bulk collective.  A shard needs one
    (contig, clusterEnd) pair from its predecessor (`carry`), and the reads at its head that continue the
    predecessor's open cluster come back as a "head partial" that the merge folds into that cluster (halo merge).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import abi
from .batch import ReadBatch


def slice_batch(b: ReadBatch, lo: int, hi: int) -> ReadBatch:
    """Reads [lo, hi) of a batch as a new batch (tile offsets recomputed; streams are views where possible)."""
    T = abi.PS_TILE_READS
    n = hi - lo
    meta = b.meta[lo:hi]
    L = (b.meta & 0xFFFF).astype(np.int64)
    nc = ((b.meta >> 16) & 0xFF).astype(np.int64)
    if b.uniform_len:
        bb = (b.uniform_len + 3) // 4
        b_lo, b_hi = lo * bb, hi * bb
        q_lo, q_hi = lo * b.uniform_len, hi * b.uniform_len
        boff = np.arange(0, n + T, T, dtype=np.uint64).clip(max=n) * np.uint64(bb)
        qoff = np.arange(0, n + T, T, dtype=np.uint64).clip(max=n) * np.uint64(b.uniform_len)
    else:
        cb = np.concatenate(([0], np.cumsum((L + 3) // 4)))
        cq = np.concatenate(([0], np.cumsum(L)))
        base0, qual0 = int(b.tile_base_off[0]), int(b.tile_qual_off[0])
        b_lo, b_hi = base0 + int(cb[lo]), base0 + int(cb[hi])
        q_lo, q_hi = qual0 + int(cq[lo]), qual0 + int(cq[hi])
        idx = np.minimum(np.arange(lo, hi + T, T), hi)
        boff = (cb[idx] - cb[lo]).astype(np.uint64)
        qoff = (cq[idx] - cq[lo]).astype(np.uint64)
    if b.uniform_ncigar:
        c_lo, c_hi = lo * b.uniform_ncigar, hi * b.uniform_ncigar
        coff = np.arange(0, n + T, T, dtype=np.uint64).clip(max=n) * np.uint64(b.uniform_ncigar)
    else:
        cc = np.concatenate(([0], np.cumsum(nc)))
        cig0 = int(b.tile_cigar_off[0])
        c_lo, c_hi = cig0 + int(cc[lo]), cig0 + int(cc[hi])
        idx = np.minimum(np.arange(lo, hi + T, T), hi)
        coff = (cc[idx] - cc[lo]).astype(np.uint64)
    n_tiles = (n + T - 1) // T
    boff, qoff, coff = boff[:n_tiles + 1], qoff[:n_tiles + 1], coff[:n_tiles + 1]
    # exceptions: re-key (read_in_tile << 16 | pos) relative to the new tiling
    exc_src = b.exc[: b.exc_count]
    tile_of = np.repeat(np.arange(b.n_tiles, dtype=np.int64), np.diff(b.tile_exc_off.astype(np.int64)))
    gread = tile_of * T + (exc_src >> 16).astype(np.int64)
    sel = (gread >= lo) & (gread < hi)
    gr = gread[sel] - lo
    exc = (((gr % T) << 16) | (exc_src[sel] & 0xFFFF).astype(np.int64)).astype(np.uint32)
    teo = np.searchsorted(gr, np.arange(0, n_tiles + 1) * T).astype(np.uint32)
    pad8 = np.zeros(64, dtype=np.uint8)
    pad32 = np.zeros(16, dtype=np.uint32)
    return ReadBatch(
        n, np.ascontiguousarray(meta), np.ascontiguousarray(b.ref_start[lo:hi]),
        np.concatenate((b.bases2[b_lo:b_hi], pad8)), np.concatenate((b.qual[q_lo:q_hi], pad8)),
        np.concatenate((b.cigar[c_lo:c_hi], pad32)), np.ascontiguousarray(boff), np.ascontiguousarray(qoff),
        np.ascontiguousarray(coff), teo, np.concatenate((exc, pad32)), uniform_len=b.uniform_len,
        uniform_ncigar=b.uniform_ncigar, bases_bytes=b_hi - b_lo, qual_bytes=q_hi - q_lo, cigar_count=c_hi - c_lo,
        exc_count=len(exc), past_end=b.past_end - lo if lo < b.past_end <= hi else 0)


def take_uniform(b: ReadBatch, idx: np.ndarray) -> ReadBatch:
    """Reads `idx` (ascending) of a uniform batch (one length, one cigar op per read, no N calls) as a new batch."""
    if not (b.uniform_len and b.uniform_ncigar == 1) or b.exc_count:
        raise ValueError("take_uniform needs a uniform batch without N calls")
    T = abi.PS_TILE_READS
    L, bb, n = b.uniform_len, (b.uniform_len + 3) // 4, len(idx)
    n_tiles = (n + T - 1) // T
    edges = np.minimum(np.arange(0, n_tiles + 1, dtype=np.uint64) * np.uint64(T), np.uint64(n))
    pad8, pad32 = np.zeros(64, dtype=np.uint8), np.zeros(16, dtype=np.uint32)
    bases = b.bases2[: b.n_reads * bb].reshape(b.n_reads, bb)[idx].reshape(-1)
    qual = b.qual[: b.n_reads * L].reshape(b.n_reads, L)[idx].reshape(-1)
    return ReadBatch(
        n, np.ascontiguousarray(b.meta[idx]), np.ascontiguousarray(b.ref_start[idx]), np.concatenate((bases, pad8)),
        np.concatenate((qual, pad8)), np.concatenate((b.cigar[: b.n_reads][idx], pad32)), edges * np.uint64(bb),
        edges * np.uint64(L), edges.copy(), np.zeros(n_tiles + 1, dtype=np.uint32), pad32.copy(), uniform_len=L,
        uniform_ncigar=1, bases_bytes=n * bb, qual_bytes=n * L, cigar_count=n, exc_count=0,
        past_end=int(np.searchsorted(idx, b.past_end - 1)) + 1 if b.past_end and b.past_end - 1 in idx else 0)


def shard_ranges(n_reads: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous, tile-aligned read ranges per rank."""
    T = abi.PS_TILE_READS
    tiles = (n_reads + T - 1) // T
    cuts = [min(n_reads, (tiles * r // world) * T) for r in range(world)] + [n_reads]
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def _strand(first_reverse: int, minus_after_first: int) -> int:
    return 1 if first_reverse else (2 if minus_after_first else 0)


def _cov_at(cov, pos: np.ndarray) -> np.ndarray:
    p0, a = cov
    idx = pos.astype(np.int64) - p0
    ok = (idx >= 0) & (idx < len(a))
    out = np.zeros(len(pos), dtype=np.uint32)
    out[ok] = a[idx[ok]]
    return out


def _cov_add(x, y):
    (p0, a), (q0, b) = x, y
    if len(a) == 0:
        return q0, b.copy()
    if len(b) == 0:
        return p0, a.copy()
    lo, hi = min(p0, q0), max(p0 + len(a), q0 + len(b))
    out = np.zeros(hi - lo, dtype=np.uint32)
    out[p0 - lo:p0 - lo + len(a)] += a
    out[q0 - lo:q0 - lo + len(b)] += b
    return lo, out


def _merge_sites(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Union of two site lists by position: counts add, first-insertion key is the smaller one."""
    if len(b) == 0:
        return a
    if len(a) == 0:
        return b
    both = np.concatenate((a, b))
    order = np.argsort(both["pos"], kind="stable")
    both = both[order]
    pos, start = np.unique(both["pos"], return_index=True)
    out = np.zeros(len(pos), dtype=abi.SITE_DTYPE)
    out["pos"] = pos
    out["t2c"] = np.add.reduceat(both["t2c"], start)
    out["cov"] = np.add.reduceat(both["cov"], start)
    out["order_key"] = np.minimum.reduceat(both["order_key"], start)
    return out


class _Merger:
    def __call__(self, shard_results: Sequence[dict], read_offsets: Sequence[int]) -> dict:
        """Fold per-shard pileup results (in genome order) into the whole-stream result."""
        clusters: List[np.ndarray] = []
        sites: List[np.ndarray] = []
        n_sites = 0
        counters = dict(num_reads_processed=0, skipped_due_indel=0, double_stranded=0, n_clusters=0, n_sites=0,
                        has_open_cluster=0)
        open_c: Optional[np.ndarray] = None     # running open cluster (a 1-element structured array copy)
        open_s = np.zeros(0, dtype=abi.SITE_DTYPE)
        open_cov = (0, np.zeros(0, dtype=np.uint32))
        created = 0                              # clusters opened so far (closed + open)

        def close_open():
            nonlocal open_c, open_s, n_sites
            if open_c is None:
                return
            c = open_c.copy()
            c["site_begin"] = n_sites
            c["site_end"] = n_sites + len(open_s)
            n_sites += len(open_s)
            clusters.append(c.reshape(1))
            sites.append(open_s)
            open_c, open_s = None, np.zeros(0, dtype=abi.SITE_DTYPE)

        for res, off in zip(shard_results, read_offsets):
            ctr = res["counters"]
            counters["num_reads_processed"] += ctr["num_reads_processed"]
            counters["skipped_due_indel"] += ctr["skipped_due_indel"]
            counters["double_stranded"] += ctr["double_stranded"]
            hp = res.get("head_partial")
            if hp is not None:
                if open_c is None:
                    raise ValueError("head partial without a preceding open cluster")
                hs = res["head_sites"].copy()
                hs["order_key"] += np.uint64(off << 6)
                open_c["num_reads"] += hp["num_reads"]
                open_c["num_t2c"] += hp["num_t2c"]
                open_c["end"] = max(int(open_c["end"]), int(hp["end"]))
                open_c["mask51"] |= hp["mask51"]
                open_c["minus_after_first"] += hp["minus_after_first"]
                if not int(open_c["first_reverse"]):
                    counters["double_stranded"] += int(hp["minus_after_first"])
                open_c["combined_strand"] = _strand(int(open_c["first_reverse"]), int(open_c["minus_after_first"]))
                # baseCoveredMap spans the cut: a site seen on one side is also covered by the other side's reads,
                # so coverage is re-read from the summed dense map of the boundary cluster
                open_cov = _cov_add(open_cov, res["head_cov"])
                open_s = _merge_sites(open_s, hs)
                open_s["cov"] = _cov_at(open_cov, open_s["pos"])
            n_new = len(res["clusters"]) + (1 if res["open_cluster"] is not None else 0)
            if n_new:
                close_open()
            if len(res["clusters"]):
                c = res["clusters"].copy()
                s = res["sites"].copy()
                c["first_read"] += np.uint64(off)
                c["running_id"] += np.uint32(created)
                c["site_begin"] += np.uint64(n_sites)
                c["site_end"] += np.uint64(n_sites)
                s["order_key"] += np.uint64(off << 6)
                n_sites += len(s)
                clusters.append(c)
                sites.append(s)
            if res["open_cluster"] is not None:
                oc = np.array(res["open_cluster"], dtype=abi.CLUSTER_DTYPE).reshape(())
                oc = oc.copy()
                oc["first_read"] += np.uint64(off)
                oc["running_id"] += np.uint32(created)
                open_c = oc
                open_s = res["open_sites"].copy()
                open_s["order_key"] += np.uint64(off << 6)
                open_cov = res["open_cov"]
            created += n_new
        out_c = np.concatenate(clusters) if clusters else np.zeros(0, dtype=abi.CLUSTER_DTYPE)
        out_s = np.concatenate(sites) if sites else np.zeros(0, dtype=abi.SITE_DTYPE)
        counters["n_clusters"] = len(out_c)
        counters["n_sites"] = len(out_s)
        counters["has_open_cluster"] = 1 if open_c is not None else 0
        if open_c is not None:
            open_c["site_begin"] = 0
            open_c["site_end"] = len(open_s)
        return {"clusters": out_c, "sites": out_s, "open_cluster": open_c, "open_sites": open_s,
                "head_partial": None, "head_sites": np.zeros(0, dtype=abi.SITE_DTYPE), "counters": counters}

    @staticmethod
    def carry_after(shard_results: Sequence[dict], prev_carry):
        """(contig, clusterEnd) the next shard must start from: Java's (tempClusterChr, tempClusterEnd)."""
        last = shard_results[-1]
        if last["open_cluster"] is not None:
            return int(last["open_cluster"]["contig"]), int(last["open_cluster"]["end"])
        if last.get("head_partial") is not None and prev_carry is not None:
            return prev_carry[0], max(prev_carry[1], int(last["head_partial"]["end"]))
        return prev_carry


merge_pileup_shards = _Merger()
