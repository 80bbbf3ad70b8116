"""Measurement of the per-position T>C conversion and coverage track (tool `track`) on one GPU.

  python tools/bench_track.py [--steps 20] [--warmup 3] [--bam-reads 300000] [--bam-copies 40] [--out FILE]
  python tools/bench_track.py --base-counts [--steps 20] [--warmup 3] [--out FILE]
  python tools/bench_track.py --indels [--steps 20] [--warmup 3] [--indel-reads 4000000] [--parent-lib SO] [--out FILE]
  python tools/bench_track.py --filters [--steps 20] [--warmup 3] [--filter-reads 4000000] [--parent-lib SO] [--out FILE]

1. Config 2 as bench.py builds it (10 M x 36-nt reads through synth.py against a 100 Mb reference), resident in HBM:
   `--steps` timed passes of ps_track_batch_device after `--warmup` passes, with the five stage times of every pass from
   ps_kernel_times (CUDA events), and the pileup stage on the same batch in the same run for comparison.  A call waits for
   the device before it returns (it reads its sizes back), so the wall time of a pass is its end-to-end device time plus
   the host copies of the rows.  Algorithmic bytes come from the shapes; the fraction is of 6552 GB/s.
2. ps_track_bam on a BAM of bam-reads x bam-copies records: the same synthetic records on bam-copies identical contigs, so
   the file stays coordinate-sorted.  Reads/s over the whole call (decode, device, files).
3. Parity: the timed batch against the C++ restatement (oracle/track_oracle.py).
The card's name and power limit are recorded with the numbers.

--base-counts measures the per-position base counts instead: on the same config-2 batch, the plain call and the call
with base counts (all twelve substitutions, thresholds 1) alternate, `--steps` passes each after `--warmup` of each; the
five stage times of both, the scratch the compact arrays take, the row counts, and the parity of the base-count call with
the C++ restatement (tests/track_bases_oracle.py) go to profiles/track_bench_bases.json (or --out).

--indels measures the per-position deletion and insertion counts: on config 5 (--indel-reads x 150-nt reads with indels
and soft clips, synth mode 1, resident in HBM) and on config 2 (10 M x 36-nt reads, no indel), against the same 100 Mb
reference, the plain call and the call with indel counts (thresholds 1) alternate, `--steps` passes each after `--warmup`
of each.  --parent-lib: a build of the library from before the option (ABI 6); its plain call joins the alternation on
the same device-resident batch, so the plain call of both builds is timed in one run.  The five stage times of every
call, the scratch the compact arrays take, the row counts and the parity of the indel call with the C++ restatement
(tests/track_indels_oracle.py) go to profiles/track_bench_indels.json (or --out).

--filters measures the read and base filters: on config 2 (10 M x 36-nt reads, the bit-parallel path) and config 5
(--filter-reads x 150-nt reads with indels, the per-base path), resident in HBM with numpy-drawn FLAG, MAPQ and
qualities, the plain call and the filtered call (MAPQ >= 10, -F 0x904, Q >= 20) alternate, with the parent build's plain
call (--parent-lib) in the same alternation.  Per-stage medians, the filter counters and the parity of the filtered call
with the C++ restatement (tests/track_filters_oracle.py) go to profiles/track_bench_filters.json (or --out).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in ("para-suite_b200", "oracle"):
    sys.path.insert(0, os.path.join(REPO, p))

import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--bam-reads", type=int, default=300_000)
ap.add_argument("--bam-copies", type=int, default=40)
ap.add_argument("--out", default=None)
ap.add_argument("--base-counts", action="store_true")
ap.add_argument("--indels", action="store_true")
ap.add_argument("--indel-reads", type=int, default=4_000_000)
ap.add_argument("--parent-lib", default=None)
ap.add_argument("--filters", action="store_true")
ap.add_argument("--filter-reads", type=int, default=4_000_000)
args = ap.parse_args()

import torch  # noqa: E402

assert torch.cuda.is_available(), "bench_track.py measures on a GPU"
from parasuite_b200 import abi, synth  # noqa: E402
from parasuite_b200.runtime import Context, DeviceBatch  # noqa: E402

PEAK_GBS = 6552.0
STAGES = ["keys_scans_segments", "segment_placement", "accumulate", "coverage_scans", "select_emit"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def compact_positions(batch):
    """M of the track: segments of the sorted reads (one contig), span + 1 each"""
    n = batch.n_reads
    s = np.asarray(batch.ref_start[:n]).astype(np.int64)
    e = s + batch.uniform_len - 1
    return _segments(s, e)


def compact_positions_cigar(batch):
    """compact_positions for any CIGAR: the reference span of every kept read (mapped, no I or D together with N)"""
    n = batch.n_reads
    meta = np.asarray(batch.meta[:n]).astype(np.int64)
    ncig = (meta >> 16) & 0xFF
    off = np.concatenate([[0], np.cumsum(ncig)])
    cig = np.asarray(batch.cigar[:off[-1]]).astype(np.int64)
    op, ln = cig & 15, cig >> 4
    rid = np.repeat(np.arange(n), ncig)
    span = np.bincount(rid, weights=ln * np.isin(op, [0, 2, 3, 7, 8]), minlength=n).astype(np.int64)
    has = {k: np.bincount(rid, weights=(op == k), minlength=n) > 0 for k in (1, 2, 3)}
    kept = (((meta >> 24) & abi.PS_RF_UNMAPPED) == 0) & ~((has[1] | has[2]) & has[3])
    s = np.asarray(batch.ref_start[:n]).astype(np.int64)[kept]
    return _segments(s, s + span[kept] - 1)


def _segments(s, e):
    pm = np.maximum.accumulate(e)
    new = np.ones(s.size, dtype=bool)
    new[1:] = s[1:] > pm[:-1] + 1
    seg = np.cumsum(new) - 1
    seg_s = s[new]
    seg_e = np.zeros(seg_s.size, dtype=np.int64)
    np.maximum.at(seg_e, seg, e)
    return int((seg_e - seg_s + 2).sum())


out = {"card": card(), "note": "wall time of a pass ends in a device synchronise; stage times are CUDA events"}
ctx = Context(0)
ref = synth.synth_reference(0x5EED0001, [100_000_000])
batch = synth.synth_reads(ref, 10_000_000, 36, seed=0x5EED0002)
ctx.upload_reference(ref)
db = DeviceBatch(batch, "cuda:0")
lib = ctx.lib


def track_once():
    h = C.c_void_p()
    st = lib.ps_track_batch_device(ctx.h, C.byref(db.struct), None, C.byref(h))
    assert st == abi.PS_OK, lib.ps_last_error(ctx.h)
    ctr = abi.ps_track_counters()
    lib.ps_track_counters_get(h, C.byref(ctr))
    lib.ps_track_close(h)
    return ctr


def base_counts_run():
    """plain and base-count calls alternately on the config-2 batch"""
    opts = abi.ps_track_opts(1, 1, 1, 0)

    def once(with_bases):
        h = C.c_void_p()
        st = lib.ps_track_batch_device_ex(ctx.h, C.byref(db.struct), C.byref(opts) if with_bases else None, None,
                                          C.byref(h))
        assert st == abi.PS_OK, lib.ps_last_error(ctx.h)
        ctr, tot = abi.ps_track_counters(), abi.ps_track_base_totals()
        lib.ps_track_counters_get(h, C.byref(ctr))
        if with_bases:
            lib.ps_track_base_totals_get(h, C.byref(tot))
        lib.ps_track_close(h)
        return ctr, tot

    for _ in range(args.warmup):
        once(False)
        once(True)
    res = {False: {"walls": [], "stages": []}, True: {"walls": [], "stages": []}}
    for _ in range(args.steps):
        for wb in (False, True):
            ctx.kernel_times_reset(True)
            t0 = time.perf_counter()
            ctr, tot = once(wb)
            res[wb]["walls"].append(time.perf_counter() - t0)
            res[wb]["stages"].append(ctx.kernel_times_ms().reshape(-1, len(STAGES))[-1])
            res[wb]["ctr"], res[wb]["tot"] = ctr, tot
    M = compact_positions(batch)
    out["config2_base_counts"] = {"reads": batch.n_reads, "compact_positions": M, "steps": args.steps,
                                  "warmup": args.warmup, "order": "plain and base-count calls alternate"}
    for wb, name in ((False, "plain"), (True, "base_counts")):
        st = np.array(res[wb]["stages"])
        out["config2_base_counts"][name] = {
            "wall_ms_median": 1e3 * float(np.median(res[wb]["walls"])),
            "device_ms_median": float(np.median(st.sum(axis=1))),
            "stage_ms_median": {k: float(np.median(st[:, i])) for i, k in enumerate(STAGES)},
            "compact_scratch_bytes": 4 * (2 * (M + 1) + 2 * M) + (40 * M if wb else 0),
            "runs": [int(res[wb]["ctr"].n_runs[0]), int(res[wb]["ctr"].n_runs[1])], "sites": int(res[wb]["ctr"].n_sites),
        }
    out["config2_base_counts"]["base_counts"]["base_rows"] = int(res[True]["tot"].n_rows)
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import track_bases_oracle  # noqa: E402
    got = ctx.track(db, base_counts=True)
    exp = track_bases_oracle.track_bases_cpp(ref, batch)
    out["parity_with_restatement"] = bool(np.array_equal(got["base_rows"], exp["base_rows"]) and
                                          np.array_equal(got["base_totals"], exp["base_totals"]) and
                                          all(np.array_equal(got[k], exp[k]) for k in ("runs_plus", "runs_minus", "sites")))
    print(json.dumps(out, indent=1))
    path = args.out or os.path.join(REPO, "profiles", "track_bench_bases.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    ctx.close()


class ParentTrack:
    """The plain track call of another build of the library, on a context of its own (same device, same process)."""

    def __init__(self, path):
        # RTLD_DEEPBIND: the build's calls between its own functions (track_run, timer_begin, ...) bind to its own
        # definitions, not to those of the library loaded before it with RTLD_GLOBAL, whose ps_ctx layout may differ
        self.lib = C.CDLL(os.path.abspath(path), mode=os.RTLD_LOCAL | os.RTLD_DEEPBIND)
        for name in ("ps_create", "ps_destroy", "ps_last_error", "ps_reference_upload", "ps_track_batch_device",
                     "ps_track_counters_get", "ps_track_close", "ps_kernel_times", "ps_kernel_times_reset"):
            f = getattr(self.lib, name)
            f.restype, f.argtypes = abi.EXPORTS[name]
        self.version = int(self.lib.ps_abi_version())
        self.h = C.c_void_p()
        assert self.lib.ps_create(C.byref(self.h), 0) == abi.PS_OK
        s = ref.as_struct()
        assert self.lib.ps_reference_upload(self.h, C.byref(s)) == abi.PS_OK

    def once(self, dbatch):
        h = C.c_void_p()
        st = self.lib.ps_track_batch_device(self.h, C.byref(dbatch.struct), None, C.byref(h))
        assert st == abi.PS_OK, self.lib.ps_last_error(self.h)
        ctr = abi.ps_track_counters()
        self.lib.ps_track_counters_get(h, C.byref(ctr))
        self.lib.ps_track_close(h)
        return ctr

    def stages(self):
        buf = np.zeros(512, dtype=np.float32)
        n = self.lib.ps_kernel_times(self.h, buf.ctypes.data, buf.size)
        return buf[:max(n, 0)].reshape(-1, len(STAGES))[-1]

    def close(self):
        self.lib.ps_destroy(self.h)


def indels_run():
    """plain and indel calls alternately on config 5 and config 2 (and the parent build's plain call)"""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import track_indels_oracle  # noqa: E402
    iopts = abi.ps_track_indel_opts(1, 1, 1, 0)
    parent = ParentTrack(args.parent_lib) if args.parent_lib else None
    if parent:
        out["parent_lib_abi_version"] = parent.version

    def once(with_indels, dbatch):
        h = C.c_void_p()
        st = lib.ps_track_batch_device_ex2(ctx.h, C.byref(dbatch.struct), None, C.byref(iopts) if with_indels else None,
                                           None, C.byref(h))
        assert st == abi.PS_OK, lib.ps_last_error(ctx.h)
        ctr, tot = abi.ps_track_counters(), abi.ps_track_indel_totals()
        lib.ps_track_counters_get(h, C.byref(ctr))
        if with_indels:
            lib.ps_track_indel_totals_get(h, C.byref(tot))
        lib.ps_track_close(h)
        return ctr, tot

    shapes = (("config5", args.indel_reads, 150, 1), ("config2", 10_000_000, 36, 0))
    parity = True
    for name, n, L, mode in shapes:
        b = synth.synth_reads(ref, n, L, seed=0x5EED0002, mode=mode)
        d = DeviceBatch(b, "cuda:0")
        arms = {"plain": lambda: once(False, d), "indels": lambda: once(True, d)}
        if parent:
            arms["parent_plain"] = lambda: (parent.once(d), None)
        for _ in range(args.warmup):
            for f in arms.values():
                f()
        res = {k: {"walls": [], "stages": []} for k in arms}
        for _ in range(args.steps):
            for k, f in arms.items():
                tctx = parent if k == "parent_plain" else ctx
                if k == "parent_plain":
                    parent.lib.ps_kernel_times_reset(parent.h, 1)
                else:
                    ctx.kernel_times_reset(True)
                t0 = time.perf_counter()
                ctr, tot = f()
                res[k]["walls"].append(time.perf_counter() - t0)
                res[k]["stages"].append(parent.stages() if tctx is parent else
                                        ctx.kernel_times_ms().reshape(-1, len(STAGES))[-1])
                res[k]["ctr"], res[k]["tot"] = ctr, tot
        M = compact_positions_cigar(b)
        o = {"reads": b.n_reads, "read_len": L, "synth_mode": mode, "steps": args.steps, "warmup": args.warmup,
             "order": " / ".join(arms) + " calls alternate"}
        for k in arms:
            st = np.array(res[k]["stages"])
            c = res[k]["ctr"]
            o[k] = {"wall_ms_median": 1e3 * float(np.median(res[k]["walls"])),
                    "device_ms_median": float(np.median(st.sum(axis=1))),
                    "stage_ms_median": {s: float(np.median(st[:, i])) for i, s in enumerate(STAGES)},
                    "stage_ms_min": {s: float(np.min(st[:, i])) for i, s in enumerate(STAGES)},
                    "runs": [int(c.n_runs[0]), int(c.n_runs[1])], "sites": int(c.n_sites),
                    "reads_counted": int(c.reads_counted), "skipped_due_indel": int(c.skipped_due_indel)}
        o["indels"]["indel_totals"] = res["indels"]["tot"].as_dict()
        o["indels"]["indel_rows"] = int(res["indels"]["tot"].n_rows)
        o["compact_positions"] = M
        o["plain"]["compact_scratch_bytes"] = 4 * (2 * (M + 1) + 2 * M)
        o["indels"]["compact_scratch_bytes"] = 4 * (2 * (M + 1) + 2 * M) + 4 * (2 * (M + 1) + 2 * M)
        got = ctx.track(d, indel_counts=True)
        exp = track_indels_oracle.track_indels_cpp(ref, b)
        same = bool(np.array_equal(got["indel_rows"], exp["indel_rows"]) and got["indel_totals"] == exp["indel_totals"]
                    and all(np.array_equal(got[k], exp[k]) for k in ("runs_plus", "runs_minus", "sites")))
        o["parity_with_restatement"] = same
        if parent:
            o["parent_plain_same_counters"] = res["parent_plain"]["ctr"].as_dict() == res["plain"]["ctr"].as_dict()
            same = same and o["parent_plain_same_counters"]
        parity = parity and same
        out[name + "_indels"] = o
        print(json.dumps(o, indent=1), flush=True)
        del d, got, exp
    out["parity_with_restatement"] = parity
    print(json.dumps(out, indent=1))
    path = args.out or os.path.join(REPO, "profiles", "track_bench_indels.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    if parent:
        parent.close()
    ctx.close()


def filters_run():
    """plain and filtered calls alternately on config 2 and config 5 (and the parent build's plain call)"""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import track_filters_oracle  # noqa: E402
    fo = abi.ps_track_filter_opts(10, 0, 0x904, 20)
    parent = ParentTrack(args.parent_lib) if args.parent_lib else None
    if parent:
        out["parent_lib_abi_version"] = parent.version
    out["filter"] = {"min_mapq": 10, "exclude_flags": 0x904, "min_base_quality": 20}

    def once(filtered, dbatch):
        h = C.c_void_p()
        if filtered:
            st = lib.ps_track_batch_device_ex3(ctx.h, C.byref(dbatch.struct), None, None, C.byref(dbatch.aux),
                                               C.byref(fo), None, C.byref(h))
        else:
            st = lib.ps_track_batch_device_ex2(ctx.h, C.byref(dbatch.struct), None, None, None, C.byref(h))
        assert st == abi.PS_OK, lib.ps_last_error(ctx.h)
        ctr, fc = abi.ps_track_counters(), abi.ps_track_filter_counters()
        lib.ps_track_counters_get(h, C.byref(ctr))
        if filtered:
            lib.ps_track_filter_counters_get(h, C.byref(fc))
        lib.ps_track_close(h)
        return ctr, fc

    rng = np.random.default_rng(0x5EED0004)
    parity = True
    for name, n, L, mode in (("config2", 10_000_000, 36, 0), ("config5", args.filter_reads, 150, 1)):
        b = synth.synth_reads(ref, n, L, seed=0x5EED0002, mode=mode)
        # FLAG: 10 % secondary, 2 % supplementary, 1 % QC-fail, 5 % duplicate besides the strand; MAPQ: 8 % below 10;
        # qualities uniform in 2..40 (about half of them below 20)
        rev = ((np.asarray(b.meta[:n]) >> np.uint32(24)) & abi.PS_RF_REVERSE) != 0
        extra = rng.choice(np.array([0x100, 0x800, 0x200, 0x400, 0], dtype=np.uint16), size=n,
                           p=[0.10, 0.02, 0.01, 0.05, 0.82])
        b.sam_flags = (np.where(rev, 0x10, 0) | extra).astype(np.uint16)
        b.mapq = rng.choice(np.array([0, 3, 30, 60], dtype=np.uint8), size=n, p=[0.05, 0.03, 0.22, 0.70])
        b.qual = np.asarray(b.qual).copy()
        b.qual[:b.qual_bytes] = rng.integers(2, 41, size=b.qual_bytes, dtype=np.uint8)
        d = DeviceBatch(b, "cuda:0")
        arms = {"plain": lambda: once(False, d), "filtered": lambda: once(True, d)}
        if parent:
            arms["parent_plain"] = lambda: (parent.once(d), None)
        for _ in range(args.warmup):
            for f in arms.values():
                f()
        res = {k: {"walls": [], "stages": []} for k in arms}
        for _ in range(args.steps):
            for k, f in arms.items():
                if k == "parent_plain":
                    parent.lib.ps_kernel_times_reset(parent.h, 1)
                else:
                    ctx.kernel_times_reset(True)
                t0 = time.perf_counter()
                ctr, fc = f()
                res[k]["walls"].append(time.perf_counter() - t0)
                res[k]["stages"].append(parent.stages() if k == "parent_plain" else
                                        ctx.kernel_times_ms().reshape(-1, len(STAGES))[-1])
                res[k]["ctr"], res[k]["fc"] = ctr, fc
        o = {"reads": b.n_reads, "read_len": L, "synth_mode": mode, "steps": args.steps, "warmup": args.warmup,
             "order": " / ".join(arms) + " calls alternate"}
        for k in arms:
            st = np.array(res[k]["stages"])
            c = res[k]["ctr"]
            o[k] = {"wall_ms_median": 1e3 * float(np.median(res[k]["walls"])),
                    "device_ms_median": float(np.median(st.sum(axis=1))),
                    "stage_ms_median": {s: float(np.median(st[:, i])) for i, s in enumerate(STAGES)},
                    "stage_ms_min": {s: float(np.min(st[:, i])) for i, s in enumerate(STAGES)},
                    "runs": [int(c.n_runs[0]), int(c.n_runs[1])], "sites": int(c.n_sites),
                    "reads_counted": int(c.reads_counted), "fast_path_reads": int(c.fast_path_reads)}
        o["filtered"]["filter_counters"] = res["filtered"]["fc"].as_dict()
        got = ctx.track(d, **out["filter"])
        exp = track_filters_oracle.track_cpp(ref, b, **out["filter"])
        same = bool(got["filter_counters"] == exp["filter_counters"] and got["counters"]["aligned_bases"] ==
                    exp["counters"]["aligned_bases"] and all(np.array_equal(got[k], exp[k])
                                                             for k in ("runs_plus", "runs_minus", "sites")))
        o["parity_with_restatement"] = same
        if parent:
            o["parent_plain_same_counters"] = res["parent_plain"]["ctr"].as_dict() == res["plain"]["ctr"].as_dict()
            same = same and o["parent_plain_same_counters"]
        parity = parity and same
        out[name + "_filters"] = o
        print(json.dumps(o, indent=1), flush=True)
        del d, got, exp
    out["parity_with_restatement"] = parity
    print(json.dumps(out, indent=1))
    path = args.out or os.path.join(REPO, "profiles", "track_bench_filters.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    if parent:
        parent.close()
    ctx.close()


if args.base_counts:
    base_counts_run()
    sys.exit(0)
if args.filters:
    filters_run()
    sys.exit(0)
if args.indels:
    indels_run()
    sys.exit(0)

for _ in range(args.warmup):
    ctr = track_once()
ctx.kernel_times_reset(True)
walls = []
for _ in range(args.steps):
    t0 = time.perf_counter()
    ctr = track_once()
    walls.append(time.perf_counter() - t0)
kt = ctx.kernel_times_ms().reshape(-1, len(STAGES))
stage_ms = {k: float(np.median(kt[:, i])) for i, k in enumerate(STAGES)}
device_ms = float(np.median(kt.sum(axis=1)))

# the pileup stage on the same batch, same run
for _ in range(args.warmup):
    with ctx.pileup_run(db) as r:
        r.counters
pl_walls, pl_dev = [], []
for _ in range(args.steps):
    t0 = time.perf_counter()
    with ctx.pileup_run(db) as r:
        r.counters
    pl_walls.append(time.perf_counter() - t0)
    pl_dev.append(float(ctx.pileup_stage_ms().sum()))

n = batch.n_reads
M = compact_positions(batch)
per_read = (36 + 3) // 4 + 4 * 1 + 8 + (36 + 3) // 4            # the pileup's 30 B
rows = 16 * (ctr.n_runs[0] + ctr.n_runs[1]) + 20 * ctr.n_sites
dense = 2 * 4 * 4 * M                                              # four 4-byte arrays per position, written and read once
alg_bytes = n * per_read + dense + rows
out["config2_batch"] = {
    "reads": n, "compact_positions": M, "runs": [int(ctr.n_runs[0]), int(ctr.n_runs[1])], "sites": int(ctr.n_sites),
    "fast_path_reads": int(ctr.fast_path_reads), "steps": args.steps,
    "track_wall_ms_median": 1e3 * float(np.median(walls)), "track_device_ms_median": device_ms,
    "track_stage_ms_median": stage_ms,
    "pileup_wall_ms_median": 1e3 * float(np.median(pl_walls)), "pileup_device_ms_median": float(np.median(pl_dev)),
    "algorithmic_bytes": int(alg_bytes),
    "algorithmic_bytes_parts": {"reads": n * per_read, "dense_arrays": dense, "rows": int(rows)},
    "fraction_of_6552_GBs_over_device_time": alg_bytes / (device_ms * 1e-3) / (PEAK_GBS * 1e9),
}
print(json.dumps(out["config2_batch"], indent=1), flush=True)

# parity of the timed batch
import track_oracle  # noqa: E402

track_oracle.build()
t0 = time.perf_counter()
exp = track_oracle.track_cpp(ref, batch)
got = ctx.track(db)
same = all(np.array_equal(got[k], exp[k]) for k in ("runs_plus", "runs_minus", "sites"))
same = same and all(got["counters"][k] == exp["counters"][k] for k in ("reads_counted", "aligned_bases", "t2c_events"))
out["parity_with_oracle"] = bool(same)
out["oracle_s"] = time.perf_counter() - t0
print("parity", same, flush=True)
del db

# the file tool
import gzip  # noqa: E402
import struct  # noqa: E402

from parasuite_b200.bamio import _bgzf_block, batch_to_records, write_bam, write_fasta  # noqa: E402

sref = synth.synth_reference(7, [5_000_000], n_run=1000)
sb = synth.synth_reads(sref, args.bam_reads, 36, seed=8)
codes = np.zeros(sref.n_bases, dtype=np.uint8)
for k in range(16):
    codes[k::16] = ((sref.seq2[: (sref.n_bases + 15) // 16] >> (2 * k)) & 3)[: len(codes[k::16])]
asc = np.frombuffer(b"ACGT", dtype=np.uint8)[codes].copy()
asc[np.unpackbits(sref.inv.view(np.uint8), bitorder="little")[: sref.n_bases].astype(bool)] = ord("N")
K = args.bam_copies
names = [f"c{k}" for k in range(K)]
with tempfile.TemporaryDirectory() as td:
    bam1, big, fa = os.path.join(td, "one.bam"), os.path.join(td, "big.bam"), os.path.join(td, "big.fa")
    write_bam(bam1, [("chr1", sref.n_bases)], batch_to_records(sb, sref), level=1)
    data = gzip.open(bam1, "rb").read()
    l_text, = struct.unpack_from("<I", data, 4)
    o = 8 + l_text + 4
    ln, = struct.unpack_from("<I", data, o)
    body = np.frombuffer(data[o + 8 + ln:], dtype=np.uint8)
    offs, q = [], 0
    while q < body.size:
        offs.append(q)
        q += 4 + struct.unpack_from("<i", body, q)[0]
    ref_id = (np.asarray(offs, dtype=np.int64) + 4)[:, None] + np.arange(4)      # refID bytes of every record
    text = b"@HD\tVN:1.4\tSO:coordinate\n" + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (nm.encode(), sref.n_bases) for nm in names)
    buf = bytearray(b"BAM\1" + struct.pack("<I", len(text)) + text + struct.pack("<I", K))
    for nm in names:
        buf += struct.pack("<I", len(nm) + 1) + nm.encode() + b"\0" + struct.pack("<I", sref.n_bases)
    with open(big, "wb") as f:
        for k in range(K):                    # copy k of the records on contig k: the file stays coordinate-sorted
            a = body.copy()
            ids = a[ref_id].view(np.int32).reshape(-1)
            a[ref_id] = np.where(ids >= 0, k, -1).astype(np.int32).view(np.uint8).reshape(-1, 4)
            buf += a.tobytes()
            while len(buf) >= 0xFF00:
                f.write(_bgzf_block(bytes(buf[:0xFF00]), 1))
                del buf[:0xFF00]
        if buf:
            f.write(_bgzf_block(bytes(buf), 1))
        f.write(_bgzf_block(b""))
    write_fasta(fa, [(nm, asc.tobytes()) for nm in names])
    n_big = args.bam_reads * K
    ctx2 = Context(0)
    ctx2.load_fasta(fa)
    res = []
    for _ in range(2):
        t0 = time.perf_counter()
        c2 = ctx2.track_bam(big, os.path.join(td, "trk"))
        res.append(time.perf_counter() - t0)
    out["track_bam"] = {"reads": n_big, "bam_bytes": os.path.getsize(big), "seconds": min(res),
                        "reads_per_s": n_big / min(res), "window_reads": int(os.environ.get("PARASUITE_B200_WINDOW_READS", 1 << 23)),
                        "runs": c2["n_runs"], "sites": c2["n_sites"]}
    ctx2.close()
print(json.dumps(out, indent=1))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
ctx.close()
