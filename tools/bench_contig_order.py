#!/usr/bin/env python
"""Pileup stage times of the config-2 batch (36-nt PAR-CLIP reads, one 36M cigar) on a multi-contig genome, in FASTA
order and re-sorted into a permuted contig order with that order set on the context (ps_reference_set_contig_order).
The two batches hold the same reads, so every contig's clusters are the same; the run checks that and prints one JSON
line with the card's name and power limit beside the numbers.  The reads carry no N calls (the re-sort moves whole
reads).  Calls alternate between the two batches.
  python tools/bench_contig_order.py [--reads N] [--contigs C] [--iters K]"""
import argparse
import json
import os
import subprocess
import sys

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(R, "para-suite_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from parasuite_b200 import synth  # noqa: E402
from parasuite_b200.runtime import Context, DeviceBatch  # noqa: E402
from parasuite_b200.sharding import take_uniform  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=10_000_000)
ap.add_argument("--ref", type=int, default=100_000_000, help="bases of the genome, split into --contigs equal contigs")
ap.add_argument("--contigs", type=int, default=8)
ap.add_argument("--iters", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
args = ap.parse_args()


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception:
        power = "unknown"
    return name, power


C = args.contigs
ref = synth.synth_reference(0x5EED0001, [args.ref // C] * C)
plain = synth.synth_reads(ref, args.reads, 36, seed=0x5EED0002, n_ppm=0)
contig = np.searchsorted(ref.contig_off.astype(np.int64), plain.ref_start[:plain.n_reads].astype(np.int64), side="right") - 1
order = [int(c) for c in np.random.default_rng(7).permutation(C)]
while order == sorted(order):
    order = order[1:] + order[:1]
idx = np.concatenate([np.nonzero(contig == c)[0] for c in order])
perm = take_uniform(plain, idx)

ctx = Context(0)
ctx.upload_reference(ref)
legs = {"fasta_order": (DeviceBatch(plain, "cuda:0"), None), "permuted": (DeviceBatch(perm, "cuda:0"), order)}
ms = {k: [] for k in legs}
clusters = {}
for it in range(args.warmup + args.iters):
    for name, (d, o) in legs.items():
        ctx.set_contig_order(o)
        with ctx.pileup_run(d) as h:
            res = h.fetch(boundary=True) if it == 0 else None
            t = ctx.pileup_stage_ms()
        torch.cuda.synchronize()
        if res is not None:       # every cluster of the run (closed ones and the open one), in contig order
            c = res["clusters"]
            rows = [(int(x["contig"]), int(x["start"]), int(x["end"]), int(x["num_reads"]), int(x["num_t2c"])) for x in c]
            if res["open_cluster"] is not None:
                x = res["open_cluster"]
                rows.append((int(x["contig"]), int(x["start"]), int(x["end"]), int(x["num_reads"]), int(x["num_t2c"])))
            clusters[name] = sorted(rows)
        if it >= args.warmup:
            ms[name].append([float(v) for v in t])
ctx.set_contig_order(None)
ctx.close()

gpu, power = card()
out = {"gpu": gpu, "power_limit": power, "reads": args.reads, "contigs": C, "order": order, "iters": args.iters,
       "same_clusters": clusters["fasta_order"] == clusters["permuted"], "n_clusters": len(clusters["fasta_order"])}
for name, v in ms.items():
    a = np.array(v)
    tot = a.sum(axis=1)
    out[name] = {"flag_ms_median": float(np.median(a[:, 0])), "flag_ms_min": float(a[:, 0].min()),
                 "flag_ms_max": float(a[:, 0].max()), "pileup_ms_median": float(np.median(tot)),
                 "pileup_ms_min": float(tot.min()), "pileup_ms_max": float(tot.max()),
                 "reads_per_s": args.reads / (float(np.median(tot)) * 1e-3)}
print(json.dumps(out), flush=True)
