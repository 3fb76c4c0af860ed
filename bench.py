#!/usr/bin/env python
"""bench.py -- CacheGen encode+decode throughput of the B200 hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (driver launches N>1 under torchrun)
  python bench.py --impl reference ...                     CPU arm: the oracle port of the reference's path
  python bench.py --config c4|c5 ...                       BASELINE configs[3] / [4]: engines sharing one lm:// server
  python bench.py --dump-outputs DIR ...                   also write the last timed step's results as .npy files, so
                                                           that two builds can be compared output for output

Workload (N=1, default): BASELINE.json configs[1] -- a 32-layer / 32-head / 128-dim, 8192-token bf16 KV block (4 GiB),
chunk_size 256 -> 32 chunks; every rank codes its own block (weak scaling, no data-path collective: the path shards by
independent engines).  One step = encode the whole block (absmax -> fused quantise/CDF/rANS-code/compact -> headers) then
decode it back to bf16 KV, in waves of 8 chunks on one stream (bounded scratch, no host synchronisation inside a step).

Printed JSON line (rank 0):
  value        raw bf16 KV bytes / (encode+decode device time), inputs resident in HBM, CUDA events on the launch stream,
               max over ranks.
  e2e          the same metric through the product's public API with HOST memory on the other side:
               LMCacheEngine.store(tokens, kv) into the compressed page-locked host tier (local_device="cpu",
               local_serde="cachegen": encode || device->host into the slab) then LMCacheEngine.retrieve(tokens)
               (host->device || decode); the KV starts on the GPU, as it does in vLLM.  All copies are inside the timed
               region.  e2e.raw_upload_variant adds an upload of the raw KV from page-locked host memory before every
               store (the round-1 definition), reported separately because that copy is not part of store().
  roofline     algorithmic HBM bytes of the dominant kernel / its live event-timed duration vs MEASURED_PEAKS.json.
  cpu_baseline the CPU oracle (port of the reference path, OpenMP, threads pinned) on a bounded sample of the workload.
  config.entropy_sweep   the same step on data of higher entropy (up to ~4.1 bits/symbol), beside the headline.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "lmsys/longchat-7b-16k"
L, H, D = 32, 32, 128
C = H * D
DUMP_SAMPLE = 1 << 22      # elements per array written by --dump-outputs: 16 MiB of float32 each


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tokens", type=int, default=8192)
    ap.add_argument("--chunk", type=int, default=256)
    ap.add_argument("--heads", type=int, default=32, help="KV heads (32 = BASELINE configs[1]; 8 = GQA shapes, side measurement)")
    ap.add_argument("--cpu-chunks", type=int, default=8, help="chunks in the bounded CPU sample")
    ap.add_argument("--config", default="c2", choices=["c2", "c4", "c5"],
                    help="c2 = BASELINE configs[1] (default, the BENCH/SCALE line); c4 / c5 = configs[3] / [4] (see c45_bench.py)")
    ap.add_argument("--wave", type=int, default=8, help="chunks per wave of the device-timed step")
    ap.add_argument("--no-sweep", action="store_true", help="skip config.entropy_sweep")
    ap.add_argument("--pipelined", action="store_true",
                    help="device step on TWO streams: the decode of wave k runs under the encode of wave k + 1 (measured: +1.4 %%; "
                         "default: one stream, so that the per-kernel times add up to the step)")
    ap.add_argument("--data", default="kv8d", choices=list(DATA_KINDS), help="synthetic KV distribution (kv8d = SURVEY 8d, the headline)")
    ap.add_argument("--coder", default="rans_compact", choices=["rans_compact", "rans", "ac"],
                    help="container: rans_compact = v3 (default: rANS + symbol counts), rans = v2 (rANS + CDF rows), ac = v1")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (rank 0): the decoded "
                         "KV and the last wave's container bytes as float32 (a fixed, seeded sample of each when larger "
                         f"than {DUMP_SAMPLE} elements) and those containers' sizes as float64")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl, args.config) != ("b200", "c2"):
        ap.error("--dump-outputs applies to the GPU arm's default workload (--impl b200 --config c2)")
    return args


# ------------------------------------------------------------------------------------------ synthetic data
DATA_KINDS = ("kv8d", "kv8d_nooutlier", "normal", "uniform", "uniform_signed")


def synth_kv_torch(tokens, device, seed, kind="kv8d"):
    """Synthetic KV, generated with torch on `device` (seeded), cast to bf16.
      kv8d            SURVEY.md 8d: N(0,1) * sigma[l,kv,c], sigma ~ LogNormal(0,0.5) clipped [0.1,8], 1% outlier channels
                      x10 (they pin every token's absmax, so almost every symbol is the centre bin: ~0.5 bits/symbol)
      kv8d_nooutlier  the same without the outlier channels
      normal          N(0,1) in every channel (~3 bits/symbol)
      uniform         torch.rand, the reference's own test data (tests/test_serde.py:10-24): U[0,1), upper bins only
      uniform_signed  U(-1,1): every bin equally likely, the coder's worst case (~4.1 bits/symbol)"""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    sigma = torch.exp(0.5 * torch.randn((L, 2, 1, C), device=device, generator=g)).clamp_(0.1, 8.0)
    outl = torch.rand((L, 2, 1, C), device=device, generator=g) < 0.01
    if kind == "kv8d":
        sigma = torch.where(outl, sigma * 10.0, sigma)
    kv = torch.empty((L, 2, tokens, C), dtype=torch.bfloat16, device=device)
    step = 512
    for t0 in range(0, tokens, step):
        n = min(step, tokens - t0)
        if kind in ("kv8d", "kv8d_nooutlier"):
            blk = torch.randn((L, 2, n, C), device=device, generator=g) * sigma
        elif kind == "normal":
            blk = torch.randn((L, 2, n, C), device=device, generator=g)
        elif kind == "uniform":
            blk = torch.rand((L, 2, n, C), device=device, generator=g)
        elif kind == "uniform_signed":
            blk = torch.rand((L, 2, n, C), device=device, generator=g) * 2.0 - 1.0
        else:
            raise ValueError(kind)
        kv[:, :, t0:t0 + n] = blk.to(torch.bfloat16)
    return kv.reshape(L, 2, tokens, H, D)


# ------------------------------------------------------------------------------------------ CPU arm / baseline
_CPU_THREADS_NOTE = ""


def _cgroup_cpus():
    """CPUs' worth of time the container is granted (cgroup v2 cpu.max or v1 cfs quota), rounded up; None = unlimited"""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return max(1, -(-int(q) // int(p)))
    except (OSError, ValueError):
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0 and p > 0:
            return max(1, -(-q // p))
    except (OSError, ValueError):
        pass
    return None


def cpu_codec_sample(n_chunks, chunk, steps, warmup, seed=4321, coder=0):
    """Time the CPU oracle (C port of the reference path, all host threads via OpenMP) on n_chunks chunks of the
    workload.  Threads are pinned (OMP_PROC_BIND=close, OMP_PLACES=cores, set before libgomp starts) and the sample's
    buffers are first touched by the timed thread team's own warm-up passes, so the figure does not depend on where the
    kernel happened to place threads and pages.  Returns (raw GB/s from the MEDIAN step, seconds [median, min], cores)."""
    # the CPUs this process may use -- asked BEFORE any OpenMP runtime starts: with OMP_PROC_BIND the runtime binds the
    # initial thread to its first place, after which sched_getaffinity() of that thread reports one core (round 2 found the
    # reference arm running on 2 threads of a 128-thread host that way)
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_DYNAMIC", "false")
    import numpy as np
    import torch

    from oracle import oracle as O
    O.build()
    cores = O.set_threads(ncpu)          # all host threads, also under torchrun (which exports OMP_NUM_THREADS=1)
    # every chunk allocates ~400 MB of numpy temporaries; by default glibc mmaps and unmaps each of them, and at 128 threads
    # the page faults -- not the coder -- bound the arm.  Keep freed blocks in the heap so that the timed passes reuse the
    # pages their warm-up passes touched.
    try:
        import ctypes
        libc = ctypes.CDLL("libc.so.6")
        libc.mallopt(-3, 1 << 30)                     # M_MMAP_THRESHOLD
        libc.mallopt(-1, ctypes.c_int(2 ** 31 - 1))   # M_TRIM_THRESHOLD
    except OSError:
        pass
    torch.set_num_threads(ncpu)
    kv = synth_kv_torch(n_chunks * chunk, "cpu", seed)
    bits = kv.view(torch.int16).numpy().view(np.uint16).reshape(L, 2, n_chunks * chunk, C)
    kb, vb = O.make_bins(MODEL)
    chunks = [np.ascontiguousarray(bits[:, :, j * chunk:(j + 1) * chunk]) for j in range(n_chunks)]
    # "All the host threads it can use": a container may SEE every hardware thread of the host and still be limited to a
    # few CPUs' worth of time (cgroup cpu.max; the GPU boxes of this pool: 128 threads visible, 16 CPUs granted) -- 128
    # runnable threads then time-slice and throttle, and the arm runs 3x slower than with 32.  So the thread count is
    # chosen by measurement: the candidates are the visible threads, the granted CPUs and twice that; one chunk each.
    cand = {ncpu}
    quota = _cgroup_cpus()
    if quota:
        cand |= {max(1, min(ncpu, quota)), max(1, min(ncpu, 2 * quota))}
    if len(cand) > 1:
        best_n, best_t = ncpu, None
        for n in sorted(cand):
            O.set_threads(n)
            for rep in range(2):                      # the first pass also warms the heap
                t0 = time.perf_counter()
                O.decode_chunk(O.encode_chunk(chunks[0], O.DT_BF16, kb, vb, coder), O.DT_BF16, kb, vb, O.DT_BF16)
                dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best_n, best_t = n, dt
        cores = O.set_threads(best_n)
    global _CPU_THREADS_NOTE
    _CPU_THREADS_NOTE = (f"{cores} OpenMP threads, the fastest of {sorted(cand)} on one chunk ({ncpu} hardware threads visible, "
                         f"cgroup grants {quota} CPUs)") if len(cand) > 1 else f"{cores} OpenMP threads = every visible hardware thread"
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for x in chunks:
            enc = O.encode_chunk(x, O.DT_BF16, kb, vb, coder)
            O.decode_chunk(enc, O.DT_BF16, kb, vb, O.DT_BF16)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    times.sort()
    med = times[len(times) // 2]
    raw = n_chunks * chunk * L * 2 * C * 2
    return raw / med / 1e9, (med, times[0]), cores


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.cpu_chunks
    steps, warmup = args.steps, args.warmup
    gbs, (med, best), cores = cpu_codec_sample(n, args.chunk, steps, warmup)
    n_all = args.tokens // args.chunk
    sample = (f"{n} of {n_all} chunks ([{L},2,{args.chunk},{H},{D}] bf16 each) per step; median of {steps} steps after "
              f"{warmup} warm-ups ({med:.2f} s, best {best:.2f} s); threads pinned (OMP_PROC_BIND=close); {_CPU_THREADS_NOTE}")
    print(json.dumps({
        "impl": "reference",
        "metric": "kv_encode_decode_raw_GBps", "value": round(gbs, 4), "unit": "GB/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": round(med * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32->u8 (bf16 KV)",
        "data": "synthetic",
        "config": {"workload": f"CacheGen encode+decode, {L}L/{H}H/{D}D {args.tokens}-token bf16 KV block, "
                               f"chunk_size {args.chunk} (BASELINE configs[1])", "sample": sample,
                   "note": "the reference's own coder (torchac_cuda) is absent, so this arm times the C port of the "
                           "reference path with the arithmetic coder of the torchac lineage (container v1); a step codes "
                           f"{n}/{n_all} of the block and value = bytes of those chunks / time"},
        "cpu_baseline": {"value": round(gbs, 4), "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample,
                         "best_GBps": round(n * args.chunk * L * 2 * C * 2 / best / 1e9, 4)},
        "e2e": {"value": round(gbs, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML from a thread every ~2 ms (the default timed
    region is ~55 ms, `nvidia-smi -lms 100` would see one sample), nvidia-smi as the fallback."""

    def __init__(self, index):
        self.nvml = None
        try:
            import threading
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml, self.samples, self.mask, self._stop = pynvml, [], 0, False
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                while not self._stop:
                    try:
                        self.samples.append(pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM))
                        self.mask |= reasons_fn(self.h)
                    except pynvml.NVMLError:
                        pass
                    time.sleep(0.002)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:       # noqa: BLE001 -- no NVML: fall back to the nvidia-smi poller
            self.nvml = None
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index),
                 "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.nvml is not None:
            n = self.nvml
            self._stop = True
            self.thread.join()
            sm = sorted(self.samples)
            try:
                smax = float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM))
            except n.NVMLError:
                smax = None
            bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap}
            reasons = sorted(k for k, b in bits.items() if self.mask & b)
            return {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_max_mhz": smax, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.path)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def parity_spot_check(kv, out, cs):
    """decoded KV of the first and last chunk vs the reference's torch op chain on the same GPU
    (tests/ref_torch.py; not timed)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_torch
    from lmcache_b200.storage_backend.serde.cachegen_basics import CacheGenConfig
    cfg = CacheGenConfig.from_model_name(MODEL)
    kb, vb = torch.tensor(cfg.key_bins_list()), torch.tensor(cfg.value_bins_list())
    T = kv.shape[2]
    ok = True
    for a in sorted({0, ((T - 1) // cs) * cs}):
        want = ref_torch.roundtrip(kv[:, :, a:a + cs], kb, vb, "vllm")
        ok = ok and bool(torch.equal(want.contiguous().view(torch.int16), out[:, :, a:a + cs].contiguous().view(torch.int16)))
    return "bit-exact" if ok else "MISMATCH"


# ------------------------------------------------------------------------------------------ GPU arm
def regen_kv(kv, seed, kind):
    """fill the resident block with another distribution, in place (no second 4 GiB allocation)"""
    import torch
    T = kv.shape[2]
    fresh = synth_kv_torch(min(T, 1024), kv.device, seed, kind)      # slab-wise: at most a 0.5 GiB temporary
    for t0 in range(0, T, fresh.shape[2]):
        n = min(fresh.shape[2], T - t0)
        if t0:
            fresh = synth_kv_torch(n, kv.device, seed + t0, kind)
        kv[:, :, t0:t0 + n] = fresh[:, :, :n]
    torch.cuda.synchronize()


def main():
    args = parse_args()
    global H, C
    H, C = args.heads, args.heads * D
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.config in ("c4", "c5"):
        import c45_bench
        c45_bench.main(args)
        return
    import torch

    import __graft_entry__ as ge
    ge.build_cuda()
    from lmcache_b200 import _native as N
    from lmcache_b200.codec import CacheGenCodec, KvView

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        # the contract is ONE JSON line on stdout: NCCL prints its "NCCL version ..." banner to the C-level stdout when
        # the communicator is created, so file descriptor 1 points at stderr until that has happened
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier(device_ids=[local])
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    T, cs = args.tokens, args.chunk
    n_chunks = (T + cs - 1) // cs
    raw_bytes = L * 2 * T * C * 2
    lib = N.lib()
    codec = CacheGenCodec(MODEL, coder=args.coder)
    kv = synth_kv_torch(T, dev, 1234 + 2 + rank, args.data)
    view = KvView.from_blob(kv, "vllm")
    out = torch.empty_like(kv)
    out_view = KvView.from_blob(out, "vllm")
    stride = codec.out_stride(L, H, D, cs)
    W = max(1, min(args.wave, n_chunks))
    # one wave of containers, reused in stream order.  --pipelined: two buffers, the decode of wave k (second stream) runs
    # while wave k + 1 is being encoded (first stream), so the kernels' last, partly filled rounds of CTAs overlap
    pipelined = args.pipelined
    stagings = [torch.empty(stride * W + N.READ_SLACK, dtype=torch.uint8, device=dev) for _ in range(2 if pipelined else 1)]
    staging = stagings[0]
    stream = torch.cuda.current_stream()
    dstream = torch.cuda.Stream(device=dev) if pipelined else None
    dec_done = [None, None]
    ws_enc = lib.b200kv_encode_workspace_bytes(L, H, D, cs, W, codec.coder_for(cs))
    ws_dec = lib.b200kv_decode_workspace_bytes(L, H, D, cs, W)

    def waves():
        for c0 in range(0, n_chunks, W):
            k = min(W, n_chunks - c0)
            yield c0, k, min(k * cs, T - c0 * cs)

    def step_device(collect=None):
        """encode -> decode, wave by wave on one stream; the decoder takes the slot bound as each container's extent, so
        nothing in the step waits for the host"""
        for w, (c0, k, nt) in enumerate(waves()):
            buf = stagings[w % len(stagings)]
            if pipelined and dec_done[w & 1] is not None:
                stream.wait_event(dec_done[w & 1])                 # the decode that last read this buffer
            ticket = codec.encode_async(view, c0 * cs, nt, cs, out=buf)
            if collect is not None:
                collect(ticket, c0, k)
            if pipelined:
                dstream.wait_event(ticket.event)
            codec.decode_raw(buf.data_ptr(), buf.numel(), [j * stride for j in range(k)], [stride] * k,
                             [min(cs, T - (c0 + j) * cs) for j in range(k)], out_view, [(c0 + j) * cs for j in range(k)],
                             N.DT_BF16, codec.coder_for(cs), dstream)
            if pipelined:
                dec_done[w & 1] = torch.cuda.Event()
                dec_done[w & 1].record(dstream)
        if pipelined:                                              # the step ends when its last decodes do
            for ev in dec_done:
                if ev is not None:
                    stream.wait_event(ev)

    def measure_sizes():
        """container sizes of the resident block; also picks the decoder's table layout the way the product does from
        the headers (b200kv_decode_chunks: transposed above 3.6 payload bits per symbol) -- the timed step hands the
        decoder slot bounds instead of sizes, so it is told through the library's measurement knob"""
        sizes = []
        os.environ.pop("B200KV_DECODE_TABLE", None)
        step_device(lambda ticket, c0, k: sizes.extend(ticket.wait().sizes))
        torch.cuda.synchronize()
        bps = 8.0 * (sum(sizes) - n_chunks * codec.layout(L, H, D, cs).fixed_bytes) / (raw_bytes / 2)
        thr = 4.1 if codec.coder_for(cs) == N.CODER_RANS_COMPACT else 3.6     # the library's own rule (b200kv_decode_chunks)
        os.environ["B200KV_DECODE_TABLE"] = "transposed" if bps > thr else "rows"
        return sizes

    def profile_kernels(steps):
        """per-kernel live timing (events around each launch inside the library), summed over a step's waves"""
        lib.b200kv_profile_enable(1)
        acc = {k: [] for k in N.PROFILE_SLOTS}
        for _ in range(steps):
            tot = {k: 0.0 for k in N.PROFILE_SLOTS}
            for c0, k, nt in waves():
                ticket = codec.encode_async(view, c0 * cs, nt, cs, out=staging)
                codec.decode_raw(staging.data_ptr(), staging.numel(), [j * stride for j in range(k)], [stride] * k,
                                 [min(cs, T - (c0 + j) * cs) for j in range(k)], out_view,
                                 [(c0 + j) * cs for j in range(k)], N.DT_BF16, codec.coder_for(cs))
                buf = (ctypes.c_float * 8)()
                N.check(lib.b200kv_profile_last(buf, 8))
                for i, name in enumerate(N.PROFILE_SLOTS):
                    if buf[i] >= 0:
                        tot[name] += buf[i]
            for name, v in tot.items():
                if v > 0:
                    acc[name].append(v)
        lib.b200kv_profile_enable(0)
        return {k: sum(v) / len(v) for k, v in acc.items() if v}

    def timed(steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            step_device()
        ev1.record(stream)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / steps

    codec_v2 = CacheGenCodec(MODEL, coder="rans") if codec.coder_for(cs) == N.CODER_RANS_COMPACT else None

    def coder_bits():
        """bits per symbol of the rANS streams alone, measured on the first wave with a version-2 container (a version-3
        payload also holds the per-stream histograms, which version 2 keeps as CDF rows in its fixed sections); not timed"""
        if codec_v2 is None:
            return None
        nt = min(W * cs, T)
        k = (nt + cs - 1) // cs
        sz = codec_v2.encode_async(view, 0, nt, cs).wait().sizes
        return round(8.0 * (sum(sz) - k * codec_v2.layout(L, H, D, cs).fixed_bytes) / (L * 2 * nt * C), 4)

    # ---- warm-up + parity spot check (not timed)
    for _ in range(max(args.warmup, 3)):
        step_device()
    sizes = measure_sizes()
    container_bytes = sum(sizes)
    fixed = codec.layout(L, H, D, cs).fixed_bytes
    payload_bytes = container_bytes - n_chunks * fixed
    parity = parity_spot_check(kv, out, cs)
    status_words = codec.decode_status()

    # ---- timed: K steps, device-resident inputs (4 GiB >> 126 MB L2: no reuse between iterations)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step_device()
    ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        nw = sum(1 for _ in waves())
        dump_outputs(args.dump_outputs, out, stagings[(nw - 1) % len(stagings)], stride, n_chunks - (nw - 1) * W, N)
    from lmcache_b200.dist_util import aggregate_gbps, max_over_ranks
    ms_step = max_over_ranks(ms_total, dev) / args.steps          # device time, max over ranks
    value = aggregate_gbps(raw_bytes, ms_step, world)              # weak scaling: every rank codes its own block

    kern_ms = profile_kernels(args.steps)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"
    alg = {  # algorithmic HBM bytes per step (DESIGN.md section 4): read 2 B/elem + write w, and the reverse
        "absmax": raw_bytes,
        "encode": raw_bytes + container_bytes,
        "decode": container_bytes + raw_bytes,
    }
    rl_all = {k: {"ms": round(kern_ms[k], 4), "alg_bytes": alg[k],
                  "achieved_GBps": round(alg[k] / (kern_ms[k] * 1e-3) / 1e9, 1),
                  "frac": round(alg[k] / (kern_ms[k] * 1e-3) / 1e9 / peak, 4)} for k in alg if k in kern_ms}
    dom = max((k for k in ("encode", "decode") if k in kern_ms), key=lambda k: kern_ms[k])
    # DRAM traffic and instruction counts of one launch come from the COMMITTED ncu --set full capture of this workload
    # (profiles/r2_traffic.json, made by profiles/traffic.py from the .ncu-rep); they are not measured in this run
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if tj["workload"] == {"tokens": T, "chunk": cs, "data": args.data, "coder": args.coder}:
            traffic_src = "profiles/r2_traffic.json (committed ncu capture, not measured in this run)"
            sm_mhz = float((clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0)
            n_smsp = torch.cuda.get_device_properties(dev).multi_processor_count * 4
            for k in alg:
                e = tj.get(f"{k}_kernel")
                if k in rl_all and e:
                    rl_all[k]["ncu_dram_bytes"] = e["dram_read_bytes"] + e["dram_write_bytes"]
                    if e.get("warp_inst_executed"):
                        slots = kern_ms[k] * 1e-3 * sm_mhz * 1e6 * n_smsp
                        rl_all[k]["issue"] = {"warp_inst": e["warp_inst_executed"], "issue_slots": round(slots),
                                              "frac": round(e["warp_inst_executed"] / slots, 4),
                                              "ncu_alu_pipe_pct": e.get("ncu_alu_pipe_pct")}
            traffic = rl_all[dom].get("ncu_dram_bytes")
    except (OSError, KeyError, ValueError):
        pass
    roofline = {"kernel": f"{dom}_kernel", "bound": "hbm", "achieved": rl_all[dom]["achieved_GBps"], "peak": peak,
                "unit": "GB/s", "frac": rl_all[dom]["frac"], "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src,
                "note": "integer coder kernels bound by instruction issue / ALU and shared-memory wavefronts (DESIGN.md "
                        "section 5), DRAM below 20 % of peak; achieved = algorithmic bytes of a step / summed live "
                        "event-timed duration of the kernel's launches in that step",
                "kernels": rl_all, "other_kernels_ms": {k: round(v, 4) for k, v in kern_ms.items() if k not in alg}}

    # ---- the same step on data of higher entropy (not the headline; same shape, same code)
    sweep = None
    if not args.no_sweep and world == 1:
        sweep = [{"data": args.data, "payload_bits_per_symbol": round(8.0 * payload_bytes / (raw_bytes / 2), 4),
                  "coder_bits_per_symbol": coder_bits(), "ms_per_step": round(ms_step, 4), "encode_ms": round(kern_ms.get("encode", 0), 4),
                  "decode_ms": round(kern_ms.get("decode", 0), 4), "container_bytes": container_bytes,
                  "GBps": round(value, 1), "parity_spot_check": parity}]
        for kind in [k for k in ("kv8d_nooutlier", "normal", "uniform", "uniform_signed") if k != args.data]:
            regen_kv(kv, 99 + rank, kind)
            step_device()
            sz = measure_sizes()
            par = parity_spot_check(kv, out, cs)
            ms = timed(args.steps)
            km = profile_kernels(2)
            sweep.append({"data": kind, "payload_bits_per_symbol": round(8.0 * (sum(sz) - n_chunks * fixed) / (raw_bytes / 2), 4),
                          "coder_bits_per_symbol": coder_bits(), "ms_per_step": round(ms, 4), "encode_ms": round(km.get("encode", 0), 4),
                          "decode_ms": round(km.get("decode", 0), 4), "container_bytes": sum(sz),
                          "GBps": round(raw_bytes / (ms * 1e-3) / 1e9, 1), "parity_spot_check": par})

    # ---- e2e through LMCacheEngine.store()/retrieve() with the compressed host tier
    e2e = None
    if not args.no_e2e:
        del out, out_view, staging
        stagings.clear()                     # frees the buffers; the list itself is still asked for its former length below
        torch.cuda.empty_cache()
        if sweep is not None:
            kv = synth_kv_torch(T, dev, 1234 + 2 + rank, args.data)
        e2e = run_e2e(args, kv, dev, world, rank, barrier)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        gbs, (med, best), cores = cpu_codec_sample(args.cpu_chunks, cs, 3, 2)
        cpu = {"value": round(gbs, 4), "unit": "GB/s", "cores": cores, "kind": "port",
               "sample": f"{args.cpu_chunks} of {n_chunks} chunks per step, median of 3 steps after 2 warm-ups "
                         f"({med:.2f} s, best {best:.2f} s), OpenMP oracle with pinned threads, arithmetic coder (v1); "
                                   f"{_CPU_THREADS_NOTE}"}

    if rank == 0:
        nlaunch_step = sum(1 for _ in waves()) * 8     # per wave: absmax, encode, scan, compact, finalize + tile_sum, tile_scan, decode
        line = {
            "metric": "kv_encode_decode_raw_GBps", "value": round(value, 2), "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32->u8 (bf16 KV)",
            "data": "synthetic",
            "config": {"workload": f"CacheGen encode+decode, {L}L/{H}H/{D}D {T}-token bf16 KV block per GPU, "
                                   f"chunk_size {cs} -> {n_chunks} chunks" + (" (BASELINE configs[1])" if (H, T) == (32, 8192) else " (BASELINE configs[2] shape: 65536-token offload + reload; e2e is that config's metric)" if (H, T) == (32, 65536) else " (side measurement, not a BASELINE shape)"),
                       "data_kind": args.data, "coder": args.coder + f" (B2KV container v{codec.coder_for(cs) + 1})",
                       "raw_bytes_per_gpu": raw_bytes, "container_bytes": container_bytes,
                       "payload_bits_per_symbol": round(8.0 * payload_bytes / (raw_bytes / 2), 4),
                       "payload_note": "container v3: the payload holds every stream's histogram header (mask + sparse counts) "
                                       "in front of its rANS bytes; coder_bits_per_symbol in entropy_sweep = the rANS bytes alone"
                       if codec_v2 is not None else "payload = the coder's bytes (histograms live in the CDF section)",
                       "wave_chunks": W,
                       "streams": ("2: encode waves on one, each wave's decode on the other (the decode of wave k runs under the "
                                   "encode of wave k + 1); roofline.kernels are per-kernel times measured one kernel at a time, so "
                                   "they may sum to slightly more than ms_per_step") if pipelined else "1",
                       "device_scratch_bytes": {"staging": staging_bytes(stride, W, N) * (2 if pipelined else 1), "encode_workspace": int(ws_enc),
                                                                  "decode_workspace": int(ws_dec)},
                       "l2": "inputs (4 GiB) exceed the 126 MB L2; no flush needed", "parity_spot_check": parity,
                       "decode_status_words_nonzero": sum(1 for w in status_words if w),
                       "entropy_sweep": sweep},
            "encode_GBps": round(raw_bytes / (sum(kern_ms.get(k, 0) for k in ("absmax", "cdf", "encode", "compact")) * 1e-3) / 1e9, 1),
            "decode_GBps": round(raw_bytes / (sum(kern_ms.get(k, 0) for k in ("tile_sum", "tile_scan", "decode")) * 1e-3) / 1e9, 1),
            "gpu_launches": nlaunch_step * args.steps,
            "clocks": clocks, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def staging_bytes(stride, W, N):
    return int(stride * W + N.READ_SLACK)


def _sample(flat, n, seed):
    """all of `flat` if it has at most n elements, else n of them at positions drawn from `seed` (the same every run)"""
    import torch
    if flat.numel() <= n:
        return flat
    idx = torch.randint(0, flat.numel(), (n,), generator=torch.Generator().manual_seed(seed))
    return flat[idx.to(flat.device)]


def dump_outputs(dst, out, buf, stride, k, N):
    """What the last timed step handed back: the decoded KV and the k containers of its last wave (found in `buf`,
    `stride` bytes apart, each as long as its header's total_bytes)."""
    import numpy as np
    import torch
    hdrs = buf[:k * stride].view(k, stride)[:, :N.HEADER_BYTES].cpu().numpy()
    sizes = [int(N.Header.from_buffer_copy(hdrs[j].tobytes()).total_bytes) for j in range(k)]
    containers = torch.cat([buf[j * stride:j * stride + s] for j, s in enumerate(sizes)])
    os.makedirs(dst, exist_ok=True)
    for name, a in (("decoded_kv", _sample(out.reshape(-1), DUMP_SAMPLE, 0).float()),
                    ("containers", _sample(containers, DUMP_SAMPLE, 1).float()),
                    ("container_sizes", torch.tensor(sizes, dtype=torch.float64))):
        np.save(os.path.join(dst, name + ".npy"), a.cpu().numpy())


def run_e2e(args, kv, dev, world, rank, barrier):
    """LMCacheEngine.store(tokens, kv) -> compressed page-locked host tier -> LMCacheEngine.retrieve(tokens), wall clock.
    No stream choreography here: the pipelines (encode || D2H, H2D || decode) live in the product
    (lmcache_b200/pipeline.py, LMCLocalCompressedBackend)."""
    import torch

    from lmcache_b200.cache_engine import LMCacheEngine
    from lmcache_b200.codec import PinnedBuffer
    from lmcache_b200.config import LMCacheEngineConfig, LMCacheEngineMetadata
    from lmcache_b200.dist_util import max_over_ranks
    T, cs = args.tokens, args.chunk
    n_chunks = (T + cs - 1) // cs
    raw_bytes = L * 2 * T * C * 2
    os.environ["LMCACHE_B200_CODER"] = args.coder
    cfg = LMCacheEngineConfig.from_legacy(chunk_size=cs, backend="cpu", local_serde="cachegen")
    engine = LMCacheEngine(cfg, LMCacheEngineMetadata(MODEL, world, rank, "vllm", "bfloat16"))
    backend = engine.engine_
    kv_tuple = tuple((kv[l, 0], kv[l, 1]) for l in range(L))          # the engine's input: L pairs of [T,H,D] tensors
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    tokens = torch.randint(0, 32000, (T,), device=dev, generator=g)
    digest = PinnedBuffer(4096)
    lib = None
    from lmcache_b200 import _native as N
    lib = N.lib()
    cur = torch.cuda.current_stream()
    t_first = time.perf_counter()
    engine.store(tokens, kv_tuple, skip_existing=False, blocking=True)   # also pays the slab's cudaHostAlloc
    first_store_s = time.perf_counter() - t_first
    backend.reserve_host(3 * backend.host_bytes())       # overwriting stores hold the old and the new containers for a moment

    def one_step(upload_from=None):
        if upload_from is not None:                       # round-1 definition: raw KV arrives from page-locked host memory
            N.check(lib.b200kv_copy_async(kv.data_ptr(), upload_from.host_ptr, raw_bytes, cur.cuda_stream))
        t0 = time.perf_counter()
        engine.store(tokens, kv_tuple, skip_existing=False, blocking=True)
        t1 = time.perf_counter()
        ret, mask = engine.retrieve(tokens)
        N.check(lib.b200kv_copy_async(digest.host_ptr, ret[0][0].data_ptr(), 4096, cur.cuda_stream))
        cur.synchronize()
        t2 = time.perf_counter()
        assert int(mask.sum()) == T
        return t1 - t0, t2 - t1

    for _ in range(2):
        one_step()
    host_bytes = backend.host_bytes()
    cont_bytes = sum(e.nbytes for e in backend.dict.values() if e.blk is not None)
    barrier()
    steps = args.steps
    t0 = time.perf_counter()
    parts = [one_step() for _ in range(steps)]
    barrier()
    wall = (time.perf_counter() - t0) / steps
    sec = max_over_ranks(wall, dev)
    ring = backend._pipe.ring
    res = {"value": round(world * raw_bytes / sec / 1e9, 2), "unit": "GB/s",
           "h2d_bytes_per_step": cont_bytes, "d2h_bytes_per_step": cont_bytes + 2 * 32 * n_chunks + 4096,
           "ms_per_step": round(sec * 1e3, 2), "steps": steps,
           "store_ms": round(1e3 * sum(p[0] for p in parts) / steps, 2),
           "retrieve_ms": round(1e3 * sum(p[1] for p in parts) / steps, 2),
           "first_store_s": round(first_store_s, 2),
           "host_tier_bytes": host_bytes, "slab_segments": backend.slab.stats()[0],
           "device_scratch_bytes": {"encode_ring": ring.scratch_bytes() if ring else None,
                                    "wave_chunks": ring.wave if ring else None},
           "path": "LMCacheEngine.store(tokens, kv_tuple, blocking=True) [sha256 chain on its own stream, keys consumed as "
                   "they appear || waves: b200kv_encode_chunks on the caller's stream || device->host of the previous wave's "
                   "containers into the page-locked slab] then LMCacheEngine.retrieve(tokens) [sha256 chain || per wave of "
                   "keys: host->device of containers || b200kv_decode_chunks into one blob]; KV starts and ends on the GPU "
                   "(retrieve returns CUDA tensors, 4 KiB of the result is read back); wall clock incl. every copy and "
                   "host-side step"}
    # the round-1 variant: the raw KV is first uploaded from page-locked host memory (not part of store(); PCIe-bound)
    if world == 1 and raw_bytes <= (8 << 30):
        host_raw = PinnedBuffer(raw_bytes)
        N.check(lib.b200kv_copy_async(host_raw.host_ptr, kv.data_ptr(), raw_bytes, cur.cuda_stream))
        cur.synchronize()
        one_step(host_raw)
        t0 = time.perf_counter()
        for _ in range(steps):
            one_step(host_raw)
        w2 = (time.perf_counter() - t0) / steps
        host_raw.close()
        res["raw_upload_variant"] = {"value": round(raw_bytes / w2 / 1e9, 2), "unit": "GB/s", "ms_per_step": round(w2 * 1e3, 2),
                                     "h2d_bytes_per_step": raw_bytes + cont_bytes,
                                     "note": "same engine calls preceded by an upload of the raw KV from page-locked host "
                                             "memory (round 1's e2e definition); that copy dominates and is not part of "
                                             "the product path"}
    engine.close()
    digest.close()
    return res


if __name__ == "__main__":
    main()
