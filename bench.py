#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: aligned reads/sec (error profile + T>C pileup) on synthetic PAR-CLIP reads.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path over one batch of synthetic coordinate-sorted reads: the profile kernel (which also
leaves one T>C mask word per read in HBM), read-back of the counts, the pileup kernels (fed with the mask words).
  value : the batch is already resident in HBM; cluster / site records stay in HBM, counters come back.
  e2e   : pinned HOST buffers through the C ABI; every copy -- records in; counts, clusters, sites and the boundary
          clusters out -- and, at N > 1, the halo merge of the cluster that spans a shard cut are inside the timed region.
Workload at every N: BASELINE configs[1] per GPU, 10M x 36-nt reads vs a 100 Mb reference region (weak scaling).  At N > 1
rank r holds region r of an N x 100 Mb genome whose contigs span two regions each, so every other shard cut lies INSIDE a
contig, and a cluster of 256 reads on either side of such a cut makes one cluster span it (open cluster of shard s-1 +
head partial of shard s).  One NCCL all-reduce of the profile count vector and one all-gather of a (contig, end) key per
rank and step; the e2e leg adds one small all-gather of the boundary-cluster pieces.
--impl reference times the CPU restatement of the Java loops (oracle/; plus the jar itself on a sample when `java` is on PATH) on the host cores, on
the whole batch.
--dump-outputs DIR writes what the last timed step of each leg handed back -- the profile arrays, the pileup counters and
records -- as DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output: the workload is
generated from fixed seeds and is the same in every run with the same arguments.
"""
import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(REPO, "para-suite_b200"), os.path.join(REPO, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "aligned reads/sec (profile + T>C pileup)"
UNIT = "reads/s"
BRIDGE = 256          # reads of the cluster placed on either side of a mid-contig shard cut


def workload(n_gpus: int, rank: int, small: bool = False):
    """Returns (name, reference, batch, max_len, info).  The per-GPU workload is the same at every N (weak scaling):
    BASELINE configs[1], 10M x 36-nt PAR-CLIP reads against a 100 Mb reference region."""
    from parasuite_b200 import synth
    region, n_reads = (2_000_000, 200_000) if small else (100_000_000, 10_000_000)
    L = 36
    if n_gpus == 1:
        ref = synth.synth_reference(0x5EED0001, [region])
        batch = synth.synth_reads(ref, n_reads, L, seed=0x5EED0002)
        name = ("config2-small" if small else
                "config2: 10M x 36-nt PAR-CLIP reads (single 36M cigar) vs 100 Mb synthetic reference")
        return name, ref, batch, 51, {"cut_lo_mid_contig": False, "cut_hi_mid_contig": False, "region": region}
    # the N-GPU job: an N x 100 Mb genome, contigs of two regions each (the last one single when N is odd), replicated
    # on every GPU as the tools need it; rank r holds the reads of region r
    lengths = [2 * region] * (n_gpus // 2) + ([region] if n_gpus % 2 else [])
    ref = synth.synth_reference(0x5EED0001, lengths)
    lo, hi = rank * region, (rank + 1) * region
    body = synth.synth_reads(ref, n_reads, L, seed=0x5EED0002 + rank, region=(lo, hi))
    cut_lo_mid = rank > 0 and rank % 2 == 1                 # region boundary r*R lies inside a contig for odd r
    cut_hi_mid = rank < n_gpus - 1 and rank % 2 == 0
    head = synth.bridge_cluster(ref, lo - 31, BRIDGE, L) if cut_lo_mid else None
    tail = synth.bridge_cluster(ref, hi - 33, BRIDGE, L) if cut_hi_mid else None
    if tail is not None:
        assert int(body.ref_start[:body.n_reads].max()) <= hi - 33, "appended cluster would break the sort order"
    batch = synth.concat_uniform(head, body, tail) if (head is not None or tail is not None) else body
    name = (("config2-small" if small else "config2: 10M x 36-nt PAR-CLIP reads (single 36M cigar) vs 100 Mb of synthetic "
             "reference") + f" per GPU (rank r = region r of a {n_gpus} x {region // 1_000_000} Mb genome in contigs of two "
            f"regions, reference replicated; +{BRIDGE} reads on either side of every mid-contig cut so that one cluster "
            "spans it)")
    return name, ref, batch, 51, {"cut_lo_mid_contig": cut_lo_mid, "cut_hi_mid_contig": cut_hi_mid, "region": region}


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def visible_physical_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def bind_to_gpu_numa_node(physical_index: int):
    """Pin this process to the CPUs NVML reports as local to its GPU BEFORE any page-locked buffer is allocated, so that
    the staging memory is first touched -- and therefore placed -- on the GPU's NUMA node.  Returns the CPU list or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(physical_index)
        words = ((os.cpu_count() or 64) + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        cpus = sorted(set(cpus) & os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return cpus
    except Exception:
        pass
    return None


class CpuPath:
    """The reference's CPU algorithm for the whole path: error-profile loop, then the T>C pileup loop.  This is the C++
    restatement under oracle/ (the Java jar cannot run: no JVM in this image).  The Java tools are single-threaded; the
    port is given every host core: the profile loop over read chunks, the pileup loop over contiguous read ranges
    (boundary clusters are not merged -- throughput only)."""

    def __init__(self, ref, batch, max_len, sample, cores):
        import oracle_lib
        from parasuite_b200.sharding import slice_batch
        oracle_lib.build()
        self.o, self.ref, self.batch, self.max_len, self.sample, self.cores = oracle_lib, ref, batch, max_len, sample, cores
        cuts = [sample * k // cores // 256 * 256 for k in range(cores)] + [sample]
        self.shards = [slice_batch(batch, cuts[k], cuts[k + 1]) for k in range(cores) if cuts[k + 1] > cuts[k]]

    def step(self):
        from concurrent.futures import ThreadPoolExecutor
        acc = self.o.profile_acc(self.ref, self.batch, self.max_len, threads=self.cores, first=0, count=self.sample)
        with ThreadPoolExecutor(len(self.shards)) as ex:
            n_cl = sum(ex.map(lambda sh: self.o.pileup_count(self.ref, sh), self.shards))
        return acc, n_cl

    def describe(self):
        whole = "the whole batch" if self.sample == self.batch.n_reads else f"the first {self.sample} reads of the batch"
        return (f"{whole} ({self.sample} reads) per step: error-profile loop ({self.cores} threads over read "
                f"chunks) + T>C pileup loop ({len(self.shards)} threads over contiguous read ranges); C++ restatement of "
                "the Java loops (the jar cannot run: no JVM in this image; the Java tools are single-threaded)")


def run_reference(args):
    """--impl reference: the reference's own CPU algorithm (oracle port; no JVM exists here) on the host cores, on the
    whole batch of rank 0's workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name, ref, batch, max_len, _ = workload(args.gpus, 0, args.small)
    cores = os.cpu_count() or 1
    cpu = CpuPath(ref, batch, max_len, batch.n_reads, cores)
    for _ in range(min(args.warmup, 2)):
        cpu.step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu.step()
    dt = time.perf_counter() - t0
    v = batch.n_reads * args.steps / dt
    try:                    # the jar itself, when this host has a JVM (it does not in the build image or on the GPU box)
        import java_ref
        java = java_ref.time_sample(ref, batch, max_len)
    except Exception as e:  # never let the optional leg break the arm
        java = {"available": False, "why": f"{type(e).__name__}: {e}"}
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": name, "stages": ["profile", "pileup"], "reads_per_step": batch.n_reads,
                   "note": "one rank's batch per step on all host cores (the Java tools are single-threaded; at N > 1 the "
                           "GPU arm processes N such batches per step)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": cpu.describe(), "java": java},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ---- parity against the oracle (outside every timed region) --------------------------------------------------------
CL_FIELDS = ("first_read", "running_id", "contig", "start", "end", "num_reads", "num_t2c", "minus_after_first",
             "first_reverse", "combined_strand", "mask51", "site_begin", "site_end")
SITE_FIELDS = ("pos", "t2c", "cov", "order_key")


def records_equal(got: dict, exp: dict) -> bool:
    """Closed clusters, their sites, the open cluster and the head partial of one shard, field by field."""
    ok = got["counters"] == exp["counters"]
    ok = ok and all(np.array_equal(got["clusters"][f], exp["clusters"][f]) for f in CL_FIELDS)
    ok = ok and all(np.array_equal(got["sites"][f], exp["sites"][f]) for f in SITE_FIELDS)
    for which, sites in (("open_cluster", "open_sites"), ("head_partial", "head_sites")):
        a, b = got.get(which), exp.get(which)
        if (a is None) != (b is None):
            return False
        if a is not None:
            # head partial: first_read / start / first_reverse describe its first read only and it has no id; what the
            # halo merge uses is compared
            fields = CL_FIELDS if which == "open_cluster" else ("end", "num_reads", "num_t2c", "mask51", "minus_after_first")
            sfields = SITE_FIELDS if which == "open_cluster" else ("pos", "t2c", "order_key")
            ok = ok and all(a[f] == b[f] for f in fields)
            ok = ok and all(np.array_equal(got[sites][f], exp[sites][f]) for f in sfields)
    for cov in ("open_cov", "head_cov"):
        if cov in got and cov in exp:
            ok = ok and got[cov][0] == exp[cov][0] and np.array_equal(got[cov][1], exp[cov][1])
    return bool(ok)


def shard_key(ref, batch):
    """max over the kept records of (contig, alignment end): what ps_pileup_max_key computes (uniform 'L M' batches)."""
    n = batch.n_reads
    kept = ((batch.meta[:n] >> 24) & 0x09) == 0           # not unmapped, POS != 0
    if not kept.any():
        return None
    off = ref.contig_off.astype(np.int64)
    g = batch.ref_start[:n][kept].astype(np.int64)
    c = np.searchsorted(off, g, side="right") - 1
    end = g - off[c] + batch.uniform_len
    k = np.lexsort((end, c))[-1]
    return int(c[k]), int(end[k])


BOUNDARY_SITES, BOUNDARY_COV = 64, 1024
BOUNDARY_WORDS = 4 + 8 + 3 * BOUNDARY_SITES + BOUNDARY_COV


def pack_head(res) -> np.ndarray:
    """Head partial of a shard (the reads continuing the preceding shard's open cluster) as a fixed-size int64 record
    for one all-gather: [present, n_sites, cov_pos0, cov_len, cluster (8 words), sites (3 words each), coverage]."""
    out = np.zeros(BOUNDARY_WORDS, dtype=np.int64)
    hp = res.get("head_partial")
    if hp is None:
        return out
    hs, (p0, cov) = res["head_sites"], res["head_cov"]
    if len(hs) > BOUNDARY_SITES or len(cov) > BOUNDARY_COV:
        out[0] = -1                                                    # too big for the fixed record (never in this workload)
        return out
    out[0], out[1], out[2], out[3] = 1, len(hs), p0, len(cov)
    out[4:12] = np.frombuffer(np.asarray(hp).tobytes(), dtype=np.int64)
    out[12:12 + 3 * len(hs)] = np.frombuffer(np.ascontiguousarray(hs).tobytes(), dtype=np.int64)
    out[12 + 3 * BOUNDARY_SITES:12 + 3 * BOUNDARY_SITES + len(cov)] = cov
    return out


def unpack_head(words: np.ndarray):
    from parasuite_b200 import abi
    if words[0] != 1:
        return None
    n_s, p0, n_c = int(words[1]), int(words[2]), int(words[3])
    hp = np.frombuffer(words[4:12].tobytes(), dtype=abi.CLUSTER_DTYPE)[0]
    hs = np.frombuffer(words[12:12 + 3 * n_s].tobytes(), dtype=abi.SITE_DTYPE).copy()
    cov = words[12 + 3 * BOUNDARY_SITES:12 + 3 * BOUNDARY_SITES + n_c].astype(np.uint32)
    return hp, hs, (p0, cov)


def merge_boundary(res, next_head, n_own_reads):
    """Halo merge on the rank that holds the open cluster: fold the next shard's head partial into it."""
    from parasuite_b200 import abi
    from parasuite_b200.sharding import merge_pileup_shards
    if next_head is None or res.get("open_cluster") is None:
        return res.get("open_cluster"), res.get("open_sites")
    hp, hs, hcov = next_head
    nxt = {"clusters": np.zeros(0, dtype=abi.CLUSTER_DTYPE), "sites": np.zeros(0, dtype=abi.SITE_DTYPE),
           "open_cluster": None, "open_sites": np.zeros(0, dtype=abi.SITE_DTYPE), "head_partial": hp, "head_sites": hs,
           "head_cov": hcov, "counters": dict(num_reads_processed=0, skipped_due_indel=0, double_stranded=0)}
    own = dict(res)
    own["clusters"], own["sites"] = own["clusters"][:0], own["sites"][:0]      # only the boundary cluster is merged here
    own["head_partial"] = None
    m = merge_pileup_shards([own, nxt], [0, n_own_reads])
    return m["open_cluster"], m["open_sites"]


DUMP_ROWS = 1 << 17     # record rows per table and rank in --dump-outputs: two legs stay below 64 MB in all
DUMP_SEED = 0x5EED0003


def dump_outputs(out_dir, prefix, profile, pileup, max_rows):
    """Writes one step's results as <out_dir>/<prefix><name>.npy in float64 (every field is an integer below 2^53, so
    the values are exact): profile_<array> for the profile result, pileup_counters in the order of ps_pileup_counters,
    pileup_<table>_<field> for the cluster / site records and the boundary clusters of the shard.  A table longer than
    max_rows is sampled at row indices drawn with a fixed seed, written as pileup_<table>_rows.  What the step did not
    produce writes no file: an empty table, a boundary cluster the shard does not have (a head partial exists only
    behind a shard cut inside a cluster), its sites or coverage when it has none."""
    from parasuite_b200 import abi
    os.makedirs(out_dir, exist_ok=True)

    def save(name, a):
        a = np.asarray(a)
        if a.dtype.kind in "iu" and a.size and int(np.abs(a).max()) >= 1 << 53:
            raise ValueError(f"{name}: values beyond 2^53 have no exact float64")
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a.astype(np.float64))

    for name, a in profile.items():
        save("profile_" + name, a)
    save("pileup_counters", [pileup["counters"][f] for f, _ in abi.ps_pileup_counters._fields_])
    tables = {"clusters": pileup["clusters"], "sites": pileup["sites"]}
    for one, sites, cov in (("open_cluster", "open_sites", "open_cov"), ("head_partial", "head_sites", "head_cov")):
        if pileup.get(one) is not None:
            tables[one], tables[sites] = np.atleast_1d(pileup[one]), pileup[sites]
            if cov in pileup and len(pileup[cov][1]):
                save(f"pileup_{cov}_pos0", [pileup[cov][0]])
                save(f"pileup_{cov}", pileup[cov][1])
    for table, rows in tables.items():
        if not len(rows):
            continue
        idx = np.arange(len(rows))
        if len(rows) > max_rows:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(len(rows), max_rows, replace=False))
            save(f"pileup_{table}_rows", idx)
        for f in rows.dtype.names:
            if f != "reserved":
                save(f"pileup_{table}_{f}", rows[f][idx])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--small", action="store_true", help="CI-sized workload (not a bench value)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer leg (default: --steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step of both legs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and not args.small:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = bind_to_gpu_numa_node(visible_physical_index(local_rank)) if world > 1 else None

    import torch
    import torch.distributed as dist
    from parasuite_b200.distributed import exclusive_prefix_max, gather_keys_device
    from parasuite_b200.runtime import Context, DeviceBatch, PinnedBatch

    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator is created: keep stdout to the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    name, ref, batch, max_len, info = workload(args.gpus, rank, args.small)
    ctx = Context(local_rank)
    ctx.upload_reference(ref)
    dbatch = DeviceBatch(batch, dev)
    alg_bytes = batch.algorithmic_bytes(with_qual=True)
    # an explicit stream for the step: its handle goes to the library with every call (a NULL stream would mean the
    # context's own stream, which torch's streams and collectives know nothing about)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pile = {}
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    red = torch.cuda.Stream(device=dev) if world > 1 else None

    def step_resident(keep=False, hold=False):
        # the whole hot path on a batch that is already in HBM: profile kernel (+ the tiny all-reduce), read-back of
        # the < 10 KB of counts, then the pileup kernels; cluster / site records stay in HBM behind the handle, their
        # counters come back to the host.  hold: the handle is left open in pile["held"], for a fetch of the records
        # after the clock has stopped
        keys = None
        ctx.profile_begin(max_len, emit_t2c_masks=True)
        ctx.profile_batch_device(dbatch, stream.cuda_stream)
        masks = ctx.profile_masks()     # one T>C mask word per read, left in HBM by the profile kernel for the pileup
        if world > 1:
            # region sharding: the maximum (contig, end) of every region, all-gathered; the exclusive prefix-max (this
            # region's carry-in) is taken on the device by the flag kernel -- no host round trip.  The key kernel and its
            # all-gather run on a side stream underneath the profile kernel (launched first, so the host-side cost of
            # the collectives is hidden too)
            with torch.cuda.stream(side):
                keys = gather_keys_device(ctx.pileup_max_key_tensor(dbatch, side.cuda_stream))
            # the all-reduce gets its own stream behind the profile kernel and the counts are read back there
            # (ps_profile_set_stream), so taking the profile back does not wait for the pileup kernels either
            red.wait_stream(stream)
            with torch.cuda.stream(red):
                dist.all_reduce(ctx.profile_acc_tensor())
            ctx.profile_set_stream(red.cuda_stream)
            stream.wait_stream(side)
        # the pileup kernels are queued right behind the profile kernel; the counts of both come back afterwards, so the
        # device does not sit idle between the two tools
        carry_keys = (keys.data_ptr(), rank) if keys is not None else None
        # ps_pileup_submit_device: the call returns behind its launches, so the host takes back the profile (and does its
        # own bookkeeping) while the pileup kernels run; the wait for the pileup is the only one left at the end
        h = ctx.pileup_run(dbatch, first_running_id=1, carry_keys=carry_keys, stream=stream.cuda_stream, defer=True,
                           masks=masks)
        try:
            res = ctx.profile_end()
            pile["counters"] = h.counters
            if keep:
                pile["res_resident"] = h.fetch(boundary=True)
        finally:
            if hold:
                pile["held"] = h
            else:
                h.close()
        return res

    # ---- warm-up ------------------------------------------------------------------------------------
    for _ in range(args.warmup):
        res = step_resident()
    # ---- device-resident timed region ---------------------------------------------------------------
    sampler = ClockSampler(visible_physical_index(local_rank))
    ctx.kernel_times_reset(True)
    launches0 = ctx.kernel_launches()
    stage_ms = []
    barrier()
    sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        res = step_resident(hold=bool(args.dump_outputs) and k + 1 == args.steps)
        stage_ms.append(ctx.pileup_stage_ms())       # events of the step just finished (already synchronised)
    e1.record(stream)
    barrier()
    sampler.stop_flag = True
    dumps = []
    if args.dump_outputs:
        with pile.pop("held") as h:
            dumps.append(("resident_", res, h.fetch(boundary=True)))
    ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches() - launches0
    ktimes = ctx.kernel_times_ms()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    nr = torch.tensor([batch.n_reads], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(nr)
    total_reads = int(nr.item())
    value = total_reads * args.steps / (ms_max * 1e-3)
    res = step_resident(keep=True)                   # one more pass outside the timed region: records for the parity check

    # ---- end-to-end leg: pinned HOST buffers through the C ABI, copies inside the timed region -------
    # one upload of the records serves both tools; every cluster and site record comes back to (pinned) host memory
    e2e_steps = args.e2e_steps or args.steps
    # the compact host form of the batch (ps_read_batch: one flag byte per read instead of the meta word, no cigar stream
    # -- every read of this workload is `36M` -- and qualities packed 6 bits each): 16 of 57 bytes per read less over the
    # host link, expanded on the device by the upload, inside the timed region
    pinned = PinnedBatch(batch, compact=True)
    gathered = torch.empty(world * BOUNDARY_WORDS, dtype=torch.int64, device=dev) if world > 1 else None
    mine_dev = torch.empty(BOUNDARY_WORDS, dtype=torch.int64, device=dev) if world > 1 else None
    mine_pin = torch.empty(BOUNDARY_WORDS, dtype=torch.int64).pin_memory() if world > 1 else None
    got_pin = torch.empty(world * BOUNDARY_WORDS, dtype=torch.int64).pin_memory() if world > 1 else None

    def step_e2e(view, more):
        # records in (one upload serves both tools; the quality bytes, more than half of it, go last).  The pileup starts
        # as soon as the other streams have arrived and its records travel back while the qualities are still on their
        # way up; the profile kernel follows the upload on a stream of its own, and the NEXT step's upload (into the other
        # staging slot of the context) is queued before the host waits for this step's results, so the host link does
        # not idle while the profile kernel of a step runs.  `view`: this step's upload, already queued.
        # Returns (profile result, the next step's view).
        nxt_view = None
        if world == 1:
            with ctx.pileup_run(view) as h:
                pile["res_e2e"] = h.fetch(pinned=True, boundary=True)
            ctx.profile_begin(max_len)
            ctx.profile_batch_device(view, stream.cuda_stream)
            if more:
                nxt_view = ctx.upload(pinned)
            return ctx.profile_end(), nxt_view
        # N > 1: the carry-in stays on the device (key kernel + all-gather on a side stream, ordered behind the part of
        # the upload they read by the library), the all-reduce of the counts runs on its own stream, nothing waits on the
        # host until the records are fetched
        with torch.cuda.stream(side):
            keys = gather_keys_device(ctx.pileup_max_key_tensor(view, side.cuda_stream))
        h = ctx.pileup_run(view, carry_keys=(keys.data_ptr(), rank), stream=side.cuda_stream, defer=True)
        ctx.profile_begin(max_len)
        ctx.profile_batch_device(view, stream.cuda_stream)
        red.wait_stream(stream)
        with torch.cuda.stream(red):
            dist.all_reduce(ctx.profile_acc_tensor())
        ctx.profile_set_stream(red.cuda_stream)
        if more:
            nxt_view = ctx.upload(pinned)
        with h:
            r = h.fetch(pinned=True, boundary=True)
            # halo merge: every shard's head partial goes to the rank in front of it (one small all-gather), which folds
            # it into its open cluster
            mine_pin.numpy()[:] = pack_head(r)
            mine_dev.copy_(mine_pin, non_blocking=True)
            dist.all_gather_into_tensor(gathered, mine_dev)
            got_pin.copy_(gathered, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            nxt = None
            if rank + 1 < world:
                w = got_pin.numpy()[(rank + 1) * BOUNDARY_WORDS:(rank + 2) * BOUNDARY_WORDS]
                if w[0] < 0:
                    raise RuntimeError("boundary cluster does not fit the fixed exchange record")
                nxt = unpack_head(w)
            r["merged_open"] = merge_boundary(r, nxt, batch.n_reads)
            pile["res_e2e"] = r
        return ctx.profile_end(), nxt_view

    v = ctx.upload(pinned)
    for k in range(2):
        _, v = step_e2e(v, k == 0)
    barrier()
    t0 = time.perf_counter()
    v = ctx.upload(pinned)                           # the first step's upload is inside the timed region like all others
    for k in range(e2e_steps):
        res_e2e, v = step_e2e(v, k + 1 < e2e_steps)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms_max = float(t.item())
    e2e_value = total_reads * e2e_steps / (e2e_ms_max * 1e-3)
    pr = pile["res_e2e"]
    d2h = int(res_e2e["wide"].nbytes + 8 + pr["clusters"].nbytes + pr["sites"].nbytes)
    if args.dump_outputs:
        dumps.append(("e2e_", res_e2e, pr))
        for prefix, prof, recs in dumps:
            dump_outputs(args.dump_outputs, (f"rank{rank}_" if world > 1 else "") + prefix, prof, recs, DUMP_ROWS // world)
    h2d = pinned.h2d_bytes

    # ---- what the host link gives a plain pinned copy with every rank copying at once (the ceiling of the e2e leg) ----
    probe = torch.empty(512 << 20, dtype=torch.uint8).pin_memory()
    probe_dev = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    for _ in range(2):
        probe_dev.copy_(probe, non_blocking=True)
    torch.cuda.synchronize()                          # the warm-up copies must be over before the clock starts
    barrier()
    t0 = time.perf_counter()
    for _ in range(6):
        probe_dev.copy_(probe, non_blocking=True)
    torch.cuda.synchronize()
    h2d_ceiling = 6 * probe.numel() / (time.perf_counter() - t0) / 1e9
    t = torch.tensor([h2d_ceiling], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    h2d_ceiling_min = float(t.item())
    del probe, probe_dev

    # ---- parity against the oracle: every rank checks its own shard, ranks in front of a mid-contig cut the merged
    #      boundary cluster ---------------------------------------------------------------------------------------------
    parity, parity_detail = None, {}
    if not args.no_parity:
        import oracle_lib
        from parasuite_b200 import synth
        from parasuite_b200.sharding import slice_batch
        oracle_lib.build()
        cores = max(1, (os.cpu_count() or 1) // world)
        acc = oracle_lib.profile_acc(ref, batch, max_len, threads=cores)
        if world > 1:
            acc_t = torch.from_numpy(acc.copy()).to(dev)
            dist.all_reduce(acc_t)
            acc = acc_t.cpu().numpy()
        ok_profile = bool(np.array_equal(acc, res["wide"]) and np.array_equal(acc, res_e2e["wide"]))
        carry = None
        if world > 1:
            keys_all = [None] * world
            dist.all_gather_object(keys_all, shard_key(ref, batch))
            carry = exclusive_prefix_max(keys_all)[rank]
        exp = oracle_lib.pileup(ref, batch, carry=carry)
        ok_resident = records_equal(pile["res_resident"], exp)
        ok_e2e = records_equal(pr, exp)
        ok_merge = True
        if world > 1 and rank + 1 < world and info["cut_hi_mid_contig"]:
            # the cluster that spans the cut behind this shard: oracle on this shard's last reads followed by the next
            # shard's first BRIDGE reads (the same deterministic cluster the next rank prepended)
            tail_n = min(batch.n_reads, 100_000)
            lo = batch.n_reads - tail_n
            nxt = synth.bridge_cluster(ref, (rank + 1) * info["region"] - 31, BRIDGE, batch.uniform_len)
            joint = synth.concat_uniform(None, slice_batch(batch, lo, batch.n_reads), nxt)
            want = oracle_lib.pileup(ref, joint)
            oc, osites = pr["merged_open"]
            wc, ws = want["open_cluster"], want["open_sites"]
            ok_merge = bool(oc is not None and wc is not None and
                            all(int(oc[f]) == int(wc[f]) for f in ("contig", "start", "end", "num_reads", "num_t2c",
                                                                   "mask51", "minus_after_first", "combined_strand")) and
                            int(oc["first_read"]) == int(wc["first_read"]) + lo and
                            all(np.array_equal(osites[f], ws[f]) for f in ("pos", "t2c", "cov")) and
                            int(oc["num_reads"]) >= 2 * BRIDGE)
        flags = torch.tensor([ok_profile, ok_resident, ok_e2e, ok_merge], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        f = [bool(x) for x in flags.tolist()]
        parity = all(f)
        parity_detail = {"profile_vs_oracle": f[0], "pileup_resident_vs_oracle": f[1], "pileup_e2e_vs_oracle": f[2],
                         "boundary_merge_vs_oracle": f[3],
                         "what": "every rank: all-reduced profile vector == oracle over the union of the shards; its shard's "
                                 "closed clusters, sites, open cluster and head partial == oracle with the same carry-in, for "
                                 "the resident (mask-fed) and the e2e (decoding) pileup; ranks in front of a mid-contig cut: "
                                 "open cluster merged with the next shard's head partial == oracle over the joint reads"}

    if rank == 0:
        peak, peak_src = peaks()
        # timer ring order per step: profile kernel(s), pileup pipeline
        k_prof = float(np.mean(ktimes[0::2])) if len(ktimes) >= 2 else float("nan")
        k_pile = float(np.mean(ktimes[1::2])) if len(ktimes) >= 2 else float("nan")
        k_flag, k_cluster, k_compact = (float(x) for x in np.mean(np.asarray(stage_ms, dtype=np.float64), axis=0))
        cl = pr["clusters"]
        n_cl, n_sites = int(len(cl)), int(len(pr["sites"]))
        covered = int((cl["end"].astype(np.int64) - cl["start"].astype(np.int64) + 1).sum())
        # SURVEY 8(d): records without qualities + 8 B per covered (cluster, locus) + 32 B per cluster record
        pile_bytes = batch.algorithmic_bytes(with_qual=False) + 8 * covered + 32 * n_cl
        step_ms = ms_max / args.steps

        def gbs(nbytes, kms):
            return nbytes / (kms * 1e-3) / 1e9 if kms == kms and kms > 0 else None

        traffic = {}
        try:    # DRAM bytes per launch from the committed ncu --set full capture of this command (tools/ncu_traffic.py)
            traffic = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))["traffic_bytes_per_launch"]
        except Exception:
            pass
        pile_traffic = sum(v for k, v in traffic.items() if k.startswith("pl_")) if traffic else None
        stages = {
            "profile_fast_kernel": {"ms": k_prof, "bytes": alg_bytes, "traffic": traffic.get("profile_fast_kernel")},
            "pileup_stage": {"ms": k_pile, "bytes": pile_bytes, "traffic": pile_traffic,
                             "kernels_ms": {"pl_flag_kernel+expand": k_flag, "pl_cluster_kernel": k_cluster,
                                            "pl_compact_kernel": k_compact}},
            "whole_step": {"ms": step_ms, "bytes": alg_bytes + pile_bytes, "traffic": None},
        }
        for v in stages.values():
            a = gbs(v["bytes"], v["ms"])
            v["achieved_gbs"] = a
            v["frac"] = a / peak if a else None
        # headline roofline entry = the longest single KERNEL of the step (the profile kernel; the pileup stage is three
        # kernels, the longest of which is shorter); every stage is listed under per_stage
        dom_name = "profile_fast_kernel" if not (k_cluster > k_prof) else "pileup_stage"
        dom = stages[dom_name]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": name, "stages": ["profile", "pileup"], "reads_per_gpu": batch.n_reads,
                       "reads_per_step": total_reads,
                       "stage_ms": {"profile_kernel": k_prof, "pileup_device": k_pile, "pl_flag_kernel": k_flag,
                                    "pl_cluster_kernel": k_cluster, "pl_compact_kernel": k_compact},
                       "stage_note": "profile_kernel also writes one T>C mask word per read, which pl_cluster_kernel reads "
                                     "instead of decoding bases and reference again; pl_flag_kernel = flag pass + cl_first "
                                     "expansion",
                       "pileup": {"clusters": n_cl, "sites": n_sites, "covered_loci": covered},
                       "max_read_length": max_len, "l2": "inputs larger than L2 (%.0f MB per pass)" % (alg_bytes / 1e6),
                       "parallelism": f"profile: read-batch sharded x{world} + all-reduce of the count vector; "
                                      f"pileup: region sharded x{world} (every other cut inside a contig), carry-in by "
                                      "all-gathered keys on the device, halo merge of the spanning cluster on the host",
                       "numa_cpus": (f"{numa_cpus[0]}-{numa_cpus[-1]} ({len(numa_cpus)})" if numa_cpus else None)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "host_form": ("compact (flags8 + uniform_cigar" + (" + qual6" if pinned.packed_qual else "") +
                                  (" + start16" if pinned.compact_start else "") + ")") if pinned.compact else "full",
                    "steps": e2e_steps, "ms_per_step": e2e_ms_max / e2e_steps,
                    "h2d_gbs_per_rank": h2d / (e2e_ms_max / e2e_steps * 1e-3) / 1e9,
                    "h2d_ceiling_gbs_per_rank": h2d_ceiling_min,
                    "ceiling_note": "plain 512 MiB pinned cudaMemcpyAsync x6 with every rank copying at once, slowest rank; "
                                    "the e2e step moves h2d_bytes_per_step over the same link"},
            "gpu_launches": int(launches),
            "clocks": sampler.result(),
            "roofline": {"bound": "hbm", "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s",
                         "frac": dom["frac"], "traffic": dom["traffic"] if world == 1 else None,
                         "kernel": dom_name, "kernel_ms": dom["ms"],
                         "algorithmic_bytes_per_launch": dom["bytes"], "peak_source": peak_src,
                         "bytes_note": "SURVEY 8(d) formulas: profile 66 B/read at 36 nt; pileup stage = 30 B/read + 8 B per "
                                       "covered (cluster, locus) + 32 B per cluster, divided by the time of all pileup "
                                       "kernels; whole_step = both over the step time; traffic = DRAM bytes of the "
                                       "committed ncu capture (profiles/traffic.json), not algorithmic",
                         "per_stage": stages},
            "parity": parity, "parity_detail": parity_detail,
        }
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            cpu = CpuPath(ref, batch, max_len, batch.n_reads, cores)
            cpu.step()
            t0 = time.perf_counter()
            cpu.step()
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": batch.n_reads / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": cpu.describe()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
