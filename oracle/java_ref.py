"""Run the reference's own jar when a JVM is around (SURVEY 8c / BASELINE.md 4(4)): `java -jar parasuite.jar error ...`
(Main.java:559-600) and `... clust ...` (Main.java:608-640) on a BAM + FASTA written by the test, and hand back the
output files as text.  Test infrastructure only; nothing in the product imports this.

The jar is the one $PARASUITE_JAR names (a build of the reference's bin/parasuite.jar); without it, or without `java`
on the PATH, the tests that use this module skip with the reason spelled out."""
import os
import shutil
import subprocess
import time

JAR_CANDIDATES = (os.environ.get("PARASUITE_JAR", ""),)

PROFILE_SUFFIXES = ("errorprofile", "errorprofile.vcf", "qualityPerMismatch", "indels", "indelprofile", "qualities")
CLUST_FILES = {"pileup": "{out}", "ccr.fasta": "{out}.ccr.fasta", "ccr.tsv": "{out}.ccr.tsv", "report": "{out}.report",
               "sitefrequency": "{bam}.sitefrequency.tsv", "sitepositions": "{bam}.sitepositions.tsv"}


def find():
    """(java executable, jar path) or (None, reason)."""
    java = shutil.which("java")
    if not java:
        return None, "no `java` on PATH"
    for p in JAR_CANDIDATES:
        if p and os.path.exists(p):
            return java, p
    return None, "java found but no parasuite.jar (set PARASUITE_JAR)"


def _run(java, jar, args, timeout):
    t0 = time.perf_counter()
    p = subprocess.run([java, "-Xmx8g", "-jar", jar] + [str(a) for a in args], capture_output=True, text=True, timeout=timeout)
    return p, time.perf_counter() - t0


def run_error(java, jar, bam, fasta, max_len, infer_q=False, timeout=1800):
    """-> ({suffix: text}, seconds, CompletedProcess).  Main.java:565-575: error <bam> <fasta> <maxLen> [-q true]."""
    args = ["error", bam, fasta, max_len] + (["-q", "true"] if infer_q else [])
    p, dt = _run(java, jar, args, timeout)
    out = {}
    for s in PROFILE_SUFFIXES:
        f = f"{bam}.{s}"
        if os.path.exists(f):
            out[s] = open(f).read()
    return out, dt, p


def run_clust(java, jar, bam, fasta, out_path, vcf, min_cov, timeout=1800):
    """-> ({name: text}, seconds, CompletedProcess).  Main.java:615-619: clust <bam> <fasta> <out> <vcf> <minCov>."""
    p, dt = _run(java, jar, ["clust", bam, fasta, out_path, vcf, min_cov], timeout)
    out = {}
    for k, v in CLUST_FILES.items():
        f = v.format(out=out_path, bam=bam)
        if os.path.exists(f):
            out[k] = open(f).read()
    return out, dt, p


def time_sample(ref, batch, max_len, n_reads=200_000, vcf=None):
    """bench.py --impl reference, when a JVM is present: the jar's `error` and `clust` tools timed on the first `n_reads`
    records of the bench batch, written out as a BAM + FASTA (the part of contig 0 they cover).  JVM start-up and file
    I/O are inside the time, as they are for any user of the tool.  -> dict for the JSON line."""
    import tempfile
    import numpy as np
    java, jar = find()
    if java is None:
        return {"available": False, "why": jar}
    from parasuite_b200.bamio import batch_to_records, write_bam, write_fasta
    from parasuite_b200.sharding import slice_batch
    n = min(int(n_reads), batch.n_reads) // 256 * 256
    recs = [r for r in batch_to_records(slice_batch(batch, 0, n), ref) if r.rname == ref.names[0]]
    hi = min(ref.lengths[0], max(r.pos + len(r.seq) for r in recs) + 64)
    k = np.arange(hi, dtype=np.int64)
    code = (ref.seq2[k >> 4] >> ((k & 15) * 2).astype(np.uint32)) & 3
    inv = (ref.inv[k >> 5] >> (k & 31).astype(np.uint32)) & 1
    seq = np.frombuffer(b"ACGT", dtype=np.uint8)[code]
    seq[inv == 1] = ord("N")
    with tempfile.TemporaryDirectory() as d:
        fa, bam, out = os.path.join(d, "ref.fa"), os.path.join(d, "reads.bam"), os.path.join(d, "clusters")
        write_fasta(fa, [(ref.names[0], seq.tobytes())])
        write_bam(bam, [(ref.names[0], hi)], recs)
        _, t_err, p1 = run_error(java, jar, bam, fa, max_len)
        if vcf is None:
            vcf = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden", "config1", "snp_db.vcf.gz")
        _, t_cl, p2 = run_clust(java, jar, bam, fa, out, vcf, 1)
    return {"available": True, "jar": jar, "reads": len(recs), "error_s": t_err, "clust_s": t_cl,
            "reads_per_s": len(recs) / (t_err + t_cl), "exit_codes": [p1.returncode, p2.returncode],
            "note": "single-threaded Java tools on a BAM + FASTA of the sample; JVM start-up and file I/O included"}


def run_comb(java, jar, genomic_bam, transcript_bam, out_bam, timeout=1800):
    """Main.java:438-486: comb -g <genomic.bam> -t <transcript.bam> -o <combined.bam>."""
    return _run(java, jar, ["comb", "-g", genomic_bam, "-t", transcript_bam, "-o", out_bam], timeout)
