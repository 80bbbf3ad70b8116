#!/usr/bin/env python
"""Where the resident step's time goes between kernels: a torch.profiler trace of a few resident steps of the bench
workload (bench.workload(1, 0), the call sequence of bench.step_resident with the timers on, as in the bench's timed
region), reduced to each kernel's start and end, the idle time between consecutive kernels of a step and between steps.

  python tools/step_trace.py [--out DIR] [--steps K] [--small]

Also answers one question the chained launches depend on: does a kernel launched with programmatic stream
serialization still start before its predecessor ends when an event record, a memset or a copy sits between them in
the stream?  Two tiny kernels (compiled with nvcc into a temporary directory): A triggers its dependents at once and
spins for 20 us, B is launched with the attribute and stamps %globaltimer before griddepcontrol.wait; B's stamp minus
A's end < 0 means B became resident while A still ran.

Writes DIR/step_trace.json (default ./step_trace_out) with the card name, power limit and SM clock.  Run it in a process of
its own: tracing slows the host, so its step times are not the bench's.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "para-suite_b200"), os.path.join(REPO, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

PROBE_SRC = r"""
#include <cuda_runtime.h>
#include <cstdint>
__device__ __forceinline__ unsigned long long now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
__global__ void probe_a(unsigned long long* t, unsigned long long spin_ns) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // as the chained kernels do, early
  const unsigned long long t0 = now();
  while (now() - t0 < spin_ns) {}
  __syncthreads();
  if (threadIdx.x == 0) atomicMax(&t[0], now());
}
__global__ void probe_b(unsigned long long* t) {
  if (threadIdx.x == 0) atomicMin(&t[1], now());      // before the wait: when the grid became resident
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (threadIdx.x == 0) atomicMin(&t[2], now());      // after it: when the predecessor's results are visible
}
// mode: 0 nothing between A and B, 1 event record, 2 memset, 3 device-to-host copy; pdl: B gets the attribute.
// out[0] = B resident - A end, out[1] = B past its wait - A end, in ns (min over the blocks)
extern "C" int probe_run(int mode, int pdl, long long* out) {
  unsigned long long *t = nullptr, *h = nullptr;
  cudaStream_t s; cudaEvent_t ev;
  if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) || cudaEventCreate(&ev)) return 1;
  if (cudaMalloc(&t, 64) || cudaHostAlloc(&h, 64, 0)) return 2;
  unsigned long long init[3] = {0, ~0ull, ~0ull};
  cudaMemcpy(t, init, sizeof init, cudaMemcpyHostToDevice);
  probe_a<<<148, 128, 0, s>>>(t, 20000);
  if (mode == 1) cudaEventRecord(ev, s);
  if (mode == 2) cudaMemsetAsync(t + 4, 0, 8, s);
  if (mode == 3) cudaMemcpyAsync(h, t + 4, 8, cudaMemcpyDeviceToHost, s);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(148); cfg.blockDim = dim3(128); cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = pdl;
  cfg.attrs = at; cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, probe_b, t)) return 3;
  if (cudaStreamSynchronize(s)) return 4;
  unsigned long long r[3];
  cudaMemcpy(r, t, sizeof r, cudaMemcpyDeviceToHost);
  out[0] = (long long)(r[1] - r[0]); out[1] = (long long)(r[2] - r[0]);
  cudaFree(t); cudaFreeHost(h); cudaEventDestroy(ev); cudaStreamDestroy(s);
  return 0;
}
"""


def card_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        info["sm_clock_mhz"] = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
        info["sm_clock_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:          # the numbers are context, never a reason to fail the trace
        info["nvml"] = f"{type(e).__name__}: {e}"
    return info


def probe(tmp):
    """Median over repeats of (B resident - A end, B past its wait - A end) in us per (stream op, attribute)."""
    import numpy as np
    nvcc = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
    src, so = os.path.join(tmp, "probe.cu"), os.path.join(tmp, "probe.so")
    with open(src, "w") as f:
        f.write(PROBE_SRC)
    subprocess.check_call([nvcc, "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared",
                           "-o", so, src])
    lib = ctypes.CDLL(so)
    out = {}
    for mode, name in enumerate(("nothing", "event_record", "memset", "d2h_copy")):
        for pdl in (1, 0):
            vals = []
            for _ in range(11):
                buf = (ctypes.c_longlong * 2)()
                rc = lib.probe_run(mode, pdl, buf)
                if rc:
                    raise RuntimeError(f"probe_run({mode}, {pdl}) = {rc}")
                vals.append((buf[0], buf[1]))
            v = np.median(np.asarray(vals, dtype=np.float64), axis=0) / 1e3
            out[f"{name}{'_pdl' if pdl else '_plain'}"] = {"b_resident_minus_a_end_us": float(v[0]),
                                                          "b_past_wait_minus_a_end_us": float(v[1])}
    for name in ("nothing", "event_record", "memset", "d2h_copy"):
        out[f"{name}_pdl"]["starts_early"] = out[f"{name}_pdl"]["b_resident_minus_a_end_us"] < 0
    return out


def trace_steps(steps, small):
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    from parasuite_b200.runtime import Context, DeviceBatch
    _, ref, batch, max_len, _ = bench.workload(1, 0, small)
    ctx = Context(0)
    ctx.upload_reference(ref)
    dev = torch.device("cuda", 0)
    dbatch = DeviceBatch(batch, dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    def step():     # bench.step_resident at one GPU
        ctx.profile_begin(max_len, emit_t2c_masks=True)
        ctx.profile_batch_device(dbatch, stream.cuda_stream)
        masks = ctx.profile_masks()
        h = ctx.pileup_run(dbatch, first_running_id=1, stream=stream.cuda_stream, defer=True, masks=masks)
        try:
            ctx.profile_end()
            h.counters
        finally:
            h.close()

    for _ in range(5):
        step()
    ctx.kernel_times_reset(True)
    torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(steps):
                step()
            torch.cuda.synchronize()
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        ev = json.load(open(path))["traceEvents"]
    ctx.close()
    dev_ops = sorted((e for e in ev if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")),
                     key=lambda e: e["ts"])
    t0 = dev_ops[0]["ts"] if dev_ops else 0.0
    ops = [{"name": e["name"][:80], "cat": e["cat"], "start_us": e["ts"] - t0, "end_us": e["ts"] + e["dur"] - t0,
            "dur_us": e["dur"]} for e in dev_ops]
    # a step starts at its profile kernel
    starts = [i for i, o in enumerate(ops) if o["cat"] == "kernel" and "profile_fast_kernel" in o["name"]]
    per_step = []
    for k, i0 in enumerate(starts):
        i1 = starts[k + 1] if k + 1 < len(starts) else len(ops)
        s_ops = ops[i0:i1]
        kern = [o for o in s_ops if o["cat"] == "kernel"]
        gaps = [{"after": a["name"][:48], "before": b["name"][:48], "idle_us": b["start_us"] - a["end_us"]}
                for a, b in zip(kern, kern[1:])]
        per_step.append({"kernels": [{"name": o["name"][:48], "start_us": o["start_us"], "end_us": o["end_us"]} for o in kern],
                         "other_device_ops": [{"name": o["name"], "start_us": o["start_us"], "dur_us": o["dur_us"]}
                                              for o in s_ops if o["cat"] != "kernel"],
                         "gaps": gaps,
                         "kernel_sum_us": sum(o["dur_us"] for o in kern),
                         "idle_inside_us": sum(max(g["idle_us"], 0.0) for g in gaps),
                         "span_us": kern[-1]["end_us"] - kern[0]["start_us"]})
    between = [ops[starts[k + 1]]["start_us"] - max(o["end_us"] for o in ops[starts[k]:starts[k + 1]])
               for k in range(len(starts) - 1)]
    summ = {"steps": len(per_step),
            "kernel_sum_us_median": float(np.median([s["kernel_sum_us"] for s in per_step])) if per_step else None,
            "idle_inside_us_median": float(np.median([s["idle_inside_us"] for s in per_step])) if per_step else None,
            "span_us_median": float(np.median([s["span_us"] for s in per_step])) if per_step else None,
            "idle_between_steps_us_median": float(np.median(between)) if between else None}
    if per_step:
        ng = len(per_step[0]["gaps"])
        if all(len(s["gaps"]) == ng for s in per_step):
            summ["gap_us_median_by_boundary"] = [
                {"after": per_step[0]["gaps"][j]["after"], "before": per_step[0]["gaps"][j]["before"],
                 "idle_us": float(np.median([s["gaps"][j]["idle_us"] for s in per_step]))} for j in range(ng)]
    return {"summary": summ, "idle_between_steps_us": between, "steps": per_step}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="step_trace_out")
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--small", action="store_true", help="CI-sized workload (not a measurement)")
    ap.add_argument("--no-probe", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"card": card_info(), "pdl_env": os.environ.get("PARASUITE_B200_PDL")}
    if not args.no_probe:
        with tempfile.TemporaryDirectory() as tmp:
            res["stream_op_between_chained_kernels"] = probe(tmp)
    res["trace"] = trace_steps(args.steps, args.small)
    res["card_after"] = card_info()
    path = os.path.join(args.out, "step_trace.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "summary": res["trace"]["summary"],
                      "probe": res.get("stream_op_between_chained_kernels")}, indent=1))


if __name__ == "__main__":
    main()
