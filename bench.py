#!/usr/bin/env python
"""bench.py — Mbases/s depth-counted on a synthetic 30x WGS-shaped alignment stream (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload wgs|chr20] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR : after the timed steps, rank 0 repeats one step of `value` and one of `e2e` untimed and writes what a
        caller of those paths receives as DIR/*.npy (float64, or float32 for text bytes; under 64 MB): window sums and
        class runs of every contig, and the BED text lengths plus a seeded sample of the text.  The workload is seeded, so
        two builds run with the same arguments can be compared output for output.

Workload (default, every N): BASELINE configs[2], the 25 primary GRCh38 contigs (3,088,286,401 bp) at 30x / 150 bp
reads, W=500 — STRONG scaling: the same genome at every N, contigs dealt to the ranks longest-first (gl_lpt_assign, the
function the CLI's --gpus uses), no data-path collective.  A "step" = one pass of the depth hot path over the rank's
contigs; time = max over ranks; value = genome bases / that time.
    --workload chr20 : BASELINE configs[1] (one 64,444,167 bp contig per rank, weak-scaling replicas; round 1's bench).

value : the rank's contigs already resident in HBM in the engine's segment format (packed8); per step, per contig:
        gl_depth_begin / add_segments_packed8_device / gl_depth_reduce (window sums + class runs stay on the device).
e2e   : the drop-in call, per contig: gl_depth_bed_contig — decoder-native int32 (start,end) segments in PINNED HOST
        memory in, finished .depth.bed + .callable.bed BYTES out in pinned host memory.  The host repack to fixed-block
        packed16 (when the rank owns >= 48 host threads), the H2D, every kernel, the device %.4g row formatter and the D2H
        of the text are inside the timed region, every step.  Two gl_ctx lanes per GPU (one host thread each) take the
        rank's contigs; every call is the synchronous call.  This is the work the reference arm is charged for (per-base
        counting + window/class walk + BED text).
extras (N=1): chr20 through every path, other shapes of chr20 (5x, maxmeandepth, W=250, W=1, long reads), the CLI on a BAM;
        every N: the 2504-sample indexcov cohort (configs[3]); N>1: the 500 x 6.18 M depthwed matrix (configs[4]).
roofline / cpu_baseline : DESIGN.md §3.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools", "synth"))

W = 500
MINCOV = 4
MAXMEAN = 0
STEP = 10_000_000           # depth/depth.go:48,132 (a multiple of W=500)
METRIC = "Mbases/s depth-counted (synth 30x WGS)"
WORKLOADS = {
    "wgs": "depth: synthetic 30x whole genome (25 GRCh38 contigs, 3,088,286,401 bp, 150 bp reads), W=500, 1 sample, contigs sharded over the GPUs",
    "chr20": "depth: synthetic 30x chr20 (64,444,167 bp, 150 bp reads), W=500, 1 sample",
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            t = [x.strip() for x in ln.split(",")]
            if len(t) < 6:
                continue
            try:
                sm.append(float(t[0])); mx.append(float(t[1]))
            except ValueError:
                continue
            for nm, v in zip(names, t[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(kernel):
    """dram__bytes_read+write per launch of `kernel` from the committed ncu --set full captures (profiles/), or None"""
    for name in ("r02_ncu_full_summary.json", "r01_ncu_full_summary.json"):
        try:
            j = json.load(open(os.path.join(ROOT, "profiles", name)))
            return int(j[kernel]["traffic_bytes"]), name
        except Exception:
            continue
    return None, None


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def contig_list(workload, world):
    import glsynth
    if workload == "wgs":
        return [(nm, ln, i) for i, (nm, ln) in enumerate(glsynth.GRCH38)]
    return [("chr20", glsynth.CHR20_LEN, 19 + r) for r in range(world)]      # one replica per rank (seed differs)


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_genome_pass(orc, contigs, threads):
    """The reference's CPU path, chunk-parallel like `goleft depth -p` (depth.go:132,392: one worker per 10 Mb chunk):
    per chunk, per-base counting (the samtools child) + the callback's window/class walk + BED text, on `threads` C
    workers (oracle/oracle_depth.c::orc_depth_jobs_mt).  contigs: [(name, length, start, end)] sorted by start.
    Returns (seconds, text bytes, chunks)."""
    t0 = time.perf_counter()
    chunks, nbytes = orc.depth_jobs_mt(contigs, W, MINCOV, MAXMEAN, threads)
    return time.perf_counter() - t0, nbytes, chunks


def sorted_copy(s, e):
    if s.size and not (np.diff(s) >= 0).all():
        o = np.argsort(s, kind="stable")
        return s[o], e[o]
    return s, e


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: neither go nor samtools exists in
    this image, so oracle/_ref cannot be built), all host threads, the same workload as the GPU arm."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    import glsynth
    from oracle import loader as orc
    threads = os.cpu_count() or 1
    contigs = []
    t0 = time.time()
    for nm, ln, idx in contig_list(args.workload, 1):
        s, e = glsynth.segments(ln, idx, threads=threads)
        s, e = sorted_copy(s, e)
        contigs.append((nm, ln, s, e))
    total = sum(c[1] for c in contigs)
    nseg = sum(c[2].size for c in contigs)
    log(f"[reference] synth: {nseg} segments over {total} bp in {time.time() - t0:.1f}s; {threads} threads")
    times, chunks = [], 0
    for i in range(args.warmup + args.steps):
        dt, _, chunks = cpu_genome_pass(orc, contigs, threads)
        if i >= args.warmup:
            times.append(dt)
    t = float(np.mean(times))
    val = total / t / 1e6
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mbases/s", "n_gpus": args.gpus,
           "steps": len(times), "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
           "scaling": "strong" if args.workload == "wgs" else "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
           "config": {"workload": WORKLOADS[args.workload], "window": W, "mincov": MINCOV, "segments": int(nseg)},
           "cpu_baseline": {"value": val, "unit": "Mbases/s", "cores": min(threads, chunks), "cores_available": threads, "kind": "port",
                            "sample": f"the whole workload per step: {chunks} chunks of 10 Mb, one worker per chunk (the reference's unit of "
                                      "parallelism, depth.go:132,392) on all host threads; per-base counting + window/class walk + BED text "
                                      "(BGZF inflate and samtools' text print/parse excluded: it under-estimates the reference)"},
           "e2e": {"value": val, "unit": "Mbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def comm_setup(ctx, dist, rank, world):
    """the library's own NCCL communicator (gl_comm_init) over the ranks torchrun started: rank 0's unique id is broadcast"""
    import torch
    from goleft_b200 import capi
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(capi.comm_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(uid, src=0)
    ctx.comm_init(bytes(uid.cpu().tolist()), rank, world)


def indexcov_cohort_leg(ctx, dist, rank, world, S=2504, T=191_000, reps=3):
    """BASELINE configs[3]: a 2504-sample 1000G-shaped .bai cohort (T tiles of 16 KB per sample), samples sharded over the
    ranks (SURVEY 8(e)): per rank I1 (offset deltas) + I2/I3 (scale + normalise) + I4/I5 (slot histograms, counters) + the
    "%.3g" tokens of I6 on its samples, device-resident; at N>1 the float32 depths [samples x T] are all-gathered so every
    rank holds the whole cohort (what I6's rows / I7 need).  Medians of three samples per rank are compared with the oracle."""
    from goleft_b200 import capi, multigpu
    lo, hi = multigpu.shard_range(S, rank, world)
    Sg, width = hi - lo, multigpu.padded_width(S, world)
    rng = np.random.default_rng(1234)
    one = np.round(rng.lognormal(np.log(1.6e9), 0.25, T)).astype(np.int64)
    cn = np.repeat(rng.choice([1.0, 0.5, 1.5, 0.0], size=T // 64 + 1, p=[0.97, 0.01, 0.01, 0.01]), 64)[:T]   # ~1 Mb blocks
    one = np.round(one * cn).astype(np.int64)
    def sample_sizes(k):
        return np.roll(one, (k * 97) % T) + np.int64(k % 1000)
    # linear-index virtual offsets of the shard: per sample T+1 offsets (prefix sums), uploaded in pieces
    d_voff = ctx.dev_empty(Sg * (T + 1) * 8)
    for j in range(Sg):
        v = np.empty(T + 1, np.uint64)
        v[0] = 100000
        np.cumsum(sample_sizes(lo + j), out=v[1:].view(np.int64))
        v[1:] += np.uint64(100000)
        capi.lib.gl_memcpy_h2d(ctx.h, d_voff.ptr + j * (T + 1) * 8, v.ctypes.data, v.nbytes)
    voff_off = ctx.dev_array(np.arange(Sg, dtype=np.int64) * (T + 1))
    n_intv = ctx.dev_array(np.full(Sg, T + 1, np.int32))
    size_off = ctx.dev_array(np.arange(Sg, dtype=np.int64) * T)
    d_sizes = ctx.dev_empty(Sg * T * 8)
    d_ptr = ctx.dev_array(np.arange(Sg + 1, dtype=np.int64) * T)
    d_med, d_dep = ctx.dev_empty(Sg * 8), ctx.dev_empty(width * T * 4)
    d_tok = ctx.dev_empty(Sg * T * 10)
    n_ref = 24                                                    # 24 reported references of ~T/24 tiles each
    bounds = np.linspace(0, T, n_ref + 1).astype(np.int64)
    seg_start = (np.arange(Sg, dtype=np.int64)[None, :] * T + bounds[:-1, None]).reshape(-1)
    seg_len = np.repeat(np.diff(bounds), Sg)
    d_ss, d_sl, d_lg = ctx.dev_array(seg_start), ctx.dev_array(seg_len), ctx.dev_array(seg_len)
    nseg = seg_start.size
    d_c, d_b = ctx.dev_empty(nseg * 70 * 4), ctx.dev_empty(nseg * 32)
    d_all = ctx.dev_empty(width * T * 4 * world) if world > 1 else None
    L = capi.lib
    def ck(rc):
        if rc != 0:
            raise RuntimeError("indexcov leg: rc %d" % rc)
    t = {"sizes": [], "cohort": [], "counts": [], "tokens": [], "allgather": [], "total": []}
    for it in range(reps + 1):
        ctx.flush_l2(); ctx.sync()
        if dist is not None:
            dist.barrier()
        ctx.timer_start()
        ck(L.gl_indexcov_sizes_batch_device(ctx.h, d_voff.ptr, voff_off.ptr, n_intv.ptr, size_off.ptr, Sg, d_sizes.ptr))
        a = ctx.timer_stop_ms(); ctx.timer_start()
        ctx.indexcov_cohort_device(d_sizes, d_ptr, Sg, d_med, d_dep)
        b = ctx.timer_stop_ms(); ctx.timer_start()
        ck(L.gl_indexcov_counts_segs_device(ctx.h, d_dep.ptr, d_ss.ptr, d_sl.ptr, d_lg.ptr, nseg, d_c.ptr, d_b.ptr))
        c = ctx.timer_stop_ms(); ctx.timer_start()
        ck(L.gl_format_g3_device(ctx.h, d_dep.ptr, Sg * T, d_tok.ptr))
        d = ctx.timer_stop_ms()
        g = 0.0
        if d_all is not None:
            dist.barrier(); ctx.timer_start()
            ctx.allgather_device(d_dep, d_all, width * T * 4)
            g = ctx.timer_stop_ms()
        if it:
            for k, v in zip(("sizes", "cohort", "counts", "tokens", "allgather"), (a, b, c, d, g)):
                t[k].append(v)
            t["total"].append(a + b + c + d + g)
    fallbacks = ctx.indexcov_cohort_fallbacks()
    med = d_med.download(np.float64, Sg)
    from oracle import loader as orc                              # the checker: three samples of this rank's shard
    ok = True
    for j in (0, Sg // 2, Sg - 1):
        sz = sample_sizes(lo + j)
        m = float(orc.ic_median(sz))
        ok = ok and med[j] == m
        dj = np.empty(T, np.float32)
        capi.lib.gl_memcpy_d2h(ctx.h, dj.ctypes.data, d_dep.ptr + j * T * 4, T * 4)
        ok = ok and bool(np.array_equal(dj.view(np.uint32), orc.ic_normalize(sz, m).view(np.uint32)))
    if d_all is not None:                                         # the gathered matrix: first sample of every rank's block
        for r in range(world):
            rlo, _ = multigpu.shard_range(S, r, world)
            sz = sample_sizes(rlo)
            dj = np.empty(T, np.float32)
            capi.lib.gl_memcpy_d2h(ctx.h, dj.ctypes.data, d_all.ptr + r * width * T * 4, T * 4)
            ok = ok and bool(np.array_equal(dj.view(np.uint32), orc.ic_normalize(sz, float(orc.ic_median(sz))).view(np.uint32)))
    for bf in (d_voff, voff_off, n_intv, size_off, d_sizes, d_ptr, d_med, d_dep, d_tok, d_ss, d_sl, d_lg, d_c, d_b) + ((d_all,) if d_all is not None else ()):
        bf.free()
    means = {k: float(np.mean(v)) for k, v in t.items()}
    if dist is not None:
        import torch
        tt = torch.tensor([means[k] for k in ("sizes", "cohort", "counts", "tokens", "allgather", "total")] + [0.0 if ok else 1.0, float(fallbacks)],
                          dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        means = dict(zip(("sizes", "cohort", "counts", "tokens", "allgather", "total"), (float(x) for x in tt[:6])))
        ok, fallbacks = float(tt[6]) == 0.0, int(tt[7])
    peak, _ = peaks()
    alg = 12 * Sg * T                                             # SURVEY 8(d): 8 B offsets in + 4 B float out per tile-sample
    k_ms = means["sizes"] + means["cohort"]
    return {"samples": S, "tiles_per_sample": T, "samples_per_rank": Sg, "ms": means, "scaling": "strong (2504 samples at every N)",
            "tile_samples_per_s": S * T / (means["total"] * 1e-3),
            "roofline_I1_I2_I3": {"alg_bytes_per_rank": alg, "ms": k_ms, "achieved_gbs": alg / (k_ms * 1e-3) / 1e9, "frac": alg / (k_ms * 1e-3) / 1e9 / peak,
                                  "basis": "12 B per tile-sample (8 B offsets in + 4 B float32 out), ic_sizes_batch_kernel + ic_cohort2_kernel"},
            "allgather_bytes": width * T * 4 * world if world > 1 else 0,
            "allgather_busbw_gbs": (width * T * 4 * (world - 1) / (means["allgather"] * 1e-3) / 1e9) if world > 1 and means["allgather"] > 0 else None,
            "cohort_fallback_samples_max_rank": fallbacks, "bit_exact_vs_oracle": bool(ok),
            "note": "device-resident, CUDA events, L2 flushed, max over ranks; medians + float32 depths of 3 samples per rank (and of the gathered "
                    "matrix at N>1) compared bit for bit with the oracle (oracle_indexcov.c)"}


def depthwed_leg(ctx, dist, rank, world, local, S=500, R=6_176_584, n_chunks=8, reps=3):
    import torch
    from goleft_b200 import capi, multigpu
    lo, hi = multigpu.shard_range(S, rank, world)
    width = multigpu.padded_width(S, world)
    base = ((np.arange(R, dtype=np.int64) * 2654435761) % 97).astype(np.int32)        # depth of (sample s, row r) = base[r] + s
    d_depth = ctx.dev_empty(width * R * 4)
    for k in range(width):
        col = base + np.int32(min(lo + k, S - 1))
        capi.lib.gl_memcpy_h2d(ctx.h, d_depth.ptr + k * R * 4, col.ctypes.data, R * 4)
    d_local, d_all = ctx.dev_empty(R * width * 4), ctx.dev_empty(R * width * 4 * world)
    d_ovf = ctx.dev_array(np.zeros(4, np.int32))
    t_over, t_agg, t_gather = [], [], []
    for it in range(reps + 1):
        ctx.sync(); dist.barrier()
        t0 = time.perf_counter()
        multigpu.depthwed_gather_overlapped(ctx, d_depth, width, R, world, d_local, d_all, d_ovf, n_chunks)
        t1 = time.perf_counter()
        ctx.sync(); dist.barrier()
        ctx.timer_start()
        ctx.depthwed_aggregate_i32_device(d_depth, width, R, None, 0, R, d_local.ptr, d_ovf)
        a = ctx.timer_stop_ms()
        dist.barrier()
        ctx.timer_start()
        ctx.allgather_device(d_local, d_all, R * width * 4)                             # one piece, on the compute stream: the plain busbw
        g = ctx.timer_stop_ms()
        if it:
            t_over.append((t1 - t0) * 1e3); t_agg.append(a); t_gather.append(g)
    # verify on every rank: the overlapped, chunked result (rows at the head, in the middle and at the tail)
    multigpu.depthwed_gather_overlapped(ctx, d_depth, width, R, world, d_local, d_all, d_ovf, n_chunks)
    ok = int(d_ovf.download(np.int32, 1)[0]) == 0
    for g0, g1 in (multigpu.chunk_bounds(R, n_chunks)[0], multigpu.chunk_bounds(R, n_chunks)[n_chunks // 2], multigpu.chunk_bounds(R, n_chunks)[-1]):
        rows = min(2000, g1 - g0)
        for r in range(world):
            rlo, rhi = multigpu.shard_range(S, r, world)
            buf = np.empty(rows * width, np.int32)
            off = (g0 * width * world + r * (g1 - g0) * width) * 4
            capi.lib.gl_memcpy_d2h(ctx.h, buf.ctypes.data, d_all.ptr + off, buf.nbytes)
            blk = buf.reshape(rows, width)
            for k in (0, rhi - rlo - 1):
                ok = ok and bool(np.array_equal(blk[:, k], base[g0:g0 + rows] + np.int32(rlo + k)))
    d_local.free(); d_all.free()
    # ---- the fused form: the aggregation kernel stores each row into the row-major R x (width*world) matrix of EVERY rank
    #      through NVLink peer mappings (gl_ipc_*): no all-gather pass, no block re-assembly
    t_p2p, ok_p2p = [], True
    try:
        wpad = (width + 3) // 4 * 4                                   # 16-byte stores: every rank's column block starts on a multiple of 4
        row_stride = wpad * world
        d_full = ctx.dev_empty(R * row_stride * 4)
        mine = torch.tensor(list(ctx.ipc_export(d_full)), dtype=torch.uint8, device="cuda")
        hs = [torch.zeros(64, dtype=torch.uint8, device="cuda") for _ in range(world)]
        dist.all_gather(hs, mine)
        ptrs = [d_full.ptr if r == rank else ctx.ipc_open(bytes(hs[r].cpu().tolist())) for r in range(world)]
        for it in range(reps + 1):
            ctx.sync(); dist.barrier()
            ctx.timer_start()
            ctx.depthwed_aggregate_i32_p2p(d_depth, width, R, None, 0, R, ptrs, row_stride, rank * wpad, d_ovf)
            ms_k = ctx.timer_stop_ms()
            dist.barrier()
            if it:
                t_p2p.append(ms_k)
        ok_p2p = int(d_ovf.download(np.int32, 1)[0]) == 0
        for g0 in (0, R // 2, R - 2000):                              # rows of the finished matrix on THIS rank: every rank's columns
            buf = np.empty(2000 * row_stride, np.int32)
            capi.lib.gl_memcpy_d2h(ctx.h, buf.ctypes.data, d_full.ptr + g0 * row_stride * 4, buf.nbytes)
            m = buf.reshape(2000, row_stride)
            for r in range(world):
                rlo, rhi = multigpu.shard_range(S, r, world)
                for k in (0, rhi - rlo - 1):
                    ok_p2p = ok_p2p and bool(np.array_equal(m[:, r * wpad + k], base[g0:g0 + 2000] + np.int32(rlo + k)))
        dist.barrier()
        for r in range(world):
            if r != rank:
                ctx.ipc_close(ptrs[r])
        dist.barrier()
        d_full.free()
    except Exception as ex:
        t_p2p, ok_p2p = [float("nan")], False
        log(f"[rank {rank}] fused p2p depthwed leg failed: {ex}")
    tt = torch.tensor([np.mean(t_over), np.mean(t_agg), np.mean(t_gather), 0.0 if ok else 1.0, float(np.mean(t_p2p)), 0.0 if ok_p2p else 1.0],
                      dtype=torch.float64, device="cuda")
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    for b in (d_depth, d_ovf):
        b.free()
    total = R * width * 4 * world
    return {"samples": S, "rows": R, "dtype": "int32", "matrix_bytes": total, "chunks": n_chunks,
            "aggregate_ms": float(tt[1]), "allgather_ms": float(tt[2]),
            "allgather_busbw_gbs": total * (world - 1) / world / (float(tt[2]) * 1e-3) / 1e9,
            "allgather_algbw_gbs": total / (float(tt[2]) * 1e-3) / 1e9,
            "overlapped_ms": float(tt[0]), "sequential_ms": float(tt[1]) + float(tt[2]),
            "overlapped_busbw_gbs": total * (world - 1) / world / (float(tt[0]) * 1e-3) / 1e9,
            "verified_on_every_rank": float(tt[3]) == 0.0,
            "fused_p2p": {"ms": float(tt[4]), "busbw_gbs": total * (world - 1) / world / (float(tt[4]) * 1e-3) / 1e9,
                          "matrix_layout": "row-major n-sites x (ceil4(samples per rank) * ranks) int32 on every rank",
                          "verified_on_every_rank": float(tt[5]) == 0.0,
                          "note": "depthwed_i32_p2p_kernel: aggregate + store every row into all ranks' row-major matrices over NVLink peer memory "
                                  "(one kernel per rank, CUDA-event time, max over ranks); busbw by the all-gather formula for comparison"},
            "note": "sample-sharded; per rank: depthwed_i32_kernel over 8 row chunks on the compute stream, ncclAllGather of each finished chunk "
                    "on the communication stream (gl_allgather_device_async); times are max over ranks"}


def config_legs(ctx, L, nm, n_cpus, timed_dev, timed_host, kernel_times, check):
    """chr20-sized contig in other shapes, each: resident step (device-timed, per-kernel ms), the drop-in call (int32 host
    segments -> BED bytes, host-timed), class runs, path taken; the first 10 Mb chunk's bytes are compared with the oracle."""
    import glsynth
    from goleft_b200 import capi
    shapes = [
        ("cov5_mincov4", dict(coverage=5.0, read_len=150), dict(W=500, mincov=4, maxmean=0)),
        ("cov30_maxmeandepth40", dict(coverage=30.0, read_len=150), dict(W=500, mincov=4, maxmean=40)),
        ("cov30_W250_default", dict(coverage=30.0, read_len=150), dict(W=250, mincov=4, maxmean=0)),
        ("cov30_W1", dict(coverage=30.0, read_len=150), dict(W=1, mincov=4, maxmean=0)),
        ("longreads_20kb_cov30", dict(coverage=30.0, read_len=20000), dict(W=500, mincov=4, maxmean=0)),
    ]
    res = {}
    for key, gen, par in shapes:
        if par["W"] == 1:                                    # W=1: one window per base, the text alone is 1.6 GB: resident only, 10 Mb
            Lc = 10_000_000
        else:
            Lc = L
        h_s, h_e = glsynth.segments(Lc, 19, threads=n_cpus, alloc=ctx.pinned_empty, **gen)
        n = int(h_s.size)
        short = gen["read_len"] <= 400
        n_win = (Lc - 1) // par["W"] + 1
        if short:
            qa, qd, ql = capi.pack_segments8(h_s, h_e, threads=0)
            dv = [ctx.dev_array(a) for a in (qa, qd, ql)]
            def resident():
                ctx.depth_begin(0, Lc)
                ctx.depth_add_segments_packed8_device(dv[0], dv[1], dv[2], qa.size)
                ctx.depth_reduce(par["W"], par["mincov"], par["maxmean"], STEP)
        else:
            dv = [ctx.dev_array(h_s), ctx.dev_array(h_e)]
            def resident():
                ctx.depth_begin(0, Lc)
                ctx.depth_add_segments_device(dv[0], dv[1], n)
                ctx.depth_reduce(par["W"], par["mincov"], par["maxmean"], STEP)
        t_res = timed_dev(resident, 5)
        k_ms, _ = kernel_times(3, resident)
        path = ctx.depth_last_path()
        _, n_runs, max_depth = ctx.depth_result_sizes()
        ent = {"bases": Lc, "segments": n, "read_len": gen["read_len"], "coverage": gen["coverage"], "window": par["W"], "mincov": par["mincov"],
               "maxmeandepth": par["maxmean"], "runs": int(n_runs), "max_depth": int(max_depth), "path": int(path),
               "resident": {"ms": t_res, "value": Lc / t_res / 1e3, "kernel_ms": k_ms,
                            "format": "packed8" if short else "int32 (start,end)"}}
        if par["W"] > 1:
            o_hd = ctx.pinned_empty(int(capi.lib.gl_depth_text_bound(nm.encode(), n_win)), np.uint8)
            o_ca = ctx.pinned_empty(max(1 << 20, 48 * (int(n_runs) + 16)), np.uint8)
            call = lambda: ctx.depth_bed_contig(nm, Lc, h_s, h_e, par["W"], par["mincov"], par["maxmean"], STEP, out=(o_hd, o_ca), raw=True)
            t_e2e = timed_host(call, 5)
            hl, cl = call()
            st = ctx.depth_transport_stats()
            ent["e2e_text_int32"] = {"ms": t_e2e, "value": Lc / t_e2e / 1e3, "h2d_bytes": st[2], "d2h_bytes": int(hl + cl), "transport": st[0],
                                     "host_pack_ms": st[1] * 1e3, "depth_path": ctx.depth_last_path(),
                                     "host_phases_ms": dict(zip(("setup", "pack_and_enqueue_loop", "reduce_text_d2h"), [x * 1e3 for x in ctx.depth_transport_phases()]))}
            if check:
                from oracle import loader as orc
                s_, e_ = sorted_copy(np.array(h_s), np.array(h_e))
                ce = min(STEP, Lc)
                hi = int(np.searchsorted(s_, ce, "left"))
                d = orc.pileup_diff(s_[:hi], e_[:hi], 0, ce)
                h, c = orc.walk_chunk(nm, 0, ce, par["W"], par["mincov"], par["maxmean"], d)
                got_hd = bytes(o_hd[:hl])
                got_ca = bytes(o_ca[:cl])
                # the first chunk's rows are a prefix of both files (chunk edges are run breaks)
                ent["first_chunk_bytes_equal_oracle_walker"] = bool(got_hd.startswith(h) and got_ca.startswith(c))
        for b in dv:
            b.free()
        res[key] = ent
    return res


def cli_wallclock(n_cpus):
    """`bin/goleft depth` end to end on a synthetic 30x chr20 BAM + BAI (tools/synth/bamsynth.c: the reads `e2e` uses, all
    flag/MAPQ classes, BGZF blocks that records straddle): wall clock, inflate rate, GPU busy fraction."""
    import glsynth
    import shutil
    import tempfile
    from goleft_b200 import capi
    exe = os.path.join(ROOT, "bin", "goleft")
    if not os.path.exists(exe):
        return {"error": "bin/goleft not built"}
    tmp = tempfile.mkdtemp(prefix="glbench_")
    try:
        bam = os.path.join(tmp, "chr20.bam")
        t0 = time.perf_counter()
        glsynth.write_bam(bam, [("chr20", glsynth.CHR20_LEN, 19)])
        t_write = time.perf_counter() - t0
        open(os.path.join(tmp, "ref.fa.fai"), "w").write("chr20\t%d\t6\t60\t61\n" % glsynth.CHR20_LEN)
        def run_cli(env_extra, reps):
            walls, tim = [], None
            for _ in range(reps):
                t0 = time.perf_counter()
                p = subprocess.run([exe, "depth", "--timing", "-w", str(W), "--prefix", os.path.join(tmp, "out"), "-r", os.path.join(tmp, "ref.fa"), bam],
                                   capture_output=True, text=True, env=dict(os.environ, **env_extra))
                walls.append(time.perf_counter() - t0)
                if p.returncode != 0:
                    raise RuntimeError(p.stderr[-300:])
                t = json.loads(p.stderr.strip().splitlines()[-1])["goleft_depth_timing"]
                if tim is None or t["wall_s"] < tim["wall_s"]:
                    tim = t
            return walls, tim
        walls, tim = run_cli({}, 3)                                   # default: the GPU feeder (BGZF inflate + record parse on the device)
        walls_h, tim_h = run_cli({"GL_GPU_FEED": "0"}, 2)             # the host feeder (zlib on the pool threads)
        ctxp = capi.Ctx(0)
        bfe = capi.Bam(bam)
        dev = [capi.bam_decode_device(ctxp, bfe, 0) for _ in range(3)][-1]      # steady state of the device feeder alone (third call)
        dev = {k: v for k, v in dev.items() if k not in ("start", "end", "d_start", "d_end")}
        bfe.close(); ctxp.close()
        # the same decode on 7 threads = the reference's parallelism on chr20 (one samtools child per 10 Mb chunk)
        b = capi.Bam(bam)
        d7 = b.decode(0, threads=7)
        dall = b.decode(0, threads=0)
        b.close()
        hd_bytes = os.path.getsize(os.path.join(tmp, "out.depth.bed"))
        # BED mode (depth.go:103-120: one samtools child per line in the reference): an exome-shaped BED, chr20's share of ~200 k
        # targets = 4,200 lines of 120-400 bp; here one pass over the span they cover + gl_depth_interval_sums for the edge windows
        bed_leg = None
        try:
            rng = np.random.default_rng(20)
            starts = np.sort(rng.integers(100_000, glsynth.CHR20_LEN - 1000, 4200))
            lens = rng.integers(120, 400, starts.size)
            with open(os.path.join(tmp, "exome.bed"), "w") as fh:
                for a_, l_ in zip(starts, lens):
                    fh.write("chr20\t%d\t%d\n" % (a_, a_ + l_))
            wb, tb = [], None
            for _ in range(2):
                t0 = time.perf_counter()
                pb = subprocess.run([exe, "depth", "--timing", "-w", "250", "--bed", os.path.join(tmp, "exome.bed"), "--prefix", os.path.join(tmp, "ex"),
                                     "-r", os.path.join(tmp, "ref.fa"), bam], capture_output=True, text=True)
                wb.append(time.perf_counter() - t0)
                if pb.returncode != 0:
                    raise RuntimeError(pb.stderr[-300:])
                tb = json.loads(pb.stderr.strip().splitlines()[-1])["goleft_depth_timing"]
            bed_leg = {"lines": int(starts.size), "window": 250, "process_wall_s_all": wb, "in_process": tb,
                       "depth_bed_rows": sum(1 for _ in open(os.path.join(tmp, "ex.depth.bed"))),
                       "note": "goleft depth --bed on the same chr20 BAM: the reference would start 4,200 samtools children"}
        except Exception as ex:
            bed_leg = {"error": str(ex)[:300]}
        return {"bam_bytes": os.path.getsize(bam), "bam_write_s": t_write, "process_wall_s": min(walls), "process_wall_s_all": walls,
                "in_process": tim, "depth_bed_bytes": hd_bytes, "bed_mode_exome": bed_leg,
                "value": glsynth.CHR20_LEN / min(walls) / 1e6, "unit": "Mbases/s",
                "gpu_feeder": {"steady_state_call": dev,
                               "note": "gl_bam_decode_device on the chr20 BAM, third call: parallel pread of the compressed range, H2D, bgzf_inflate_kernel "
                                       "(one warp per BGZF member), two bam_parse passes; inflate_s / parse_s are device times"},
                "host_feeder": {"process_wall_s_all": walls_h, "in_process": tim_h,
                                "inflate_MBps_per_thread": tim_h["bgzf_bytes_out"] / 1e6 / max(tim_h["inflate_thread_s_sum"], 1e-9)},
                "decode_only": {"threads_all": {"wall_s": dall["wall_s"], "records": dall["n_records"]},
                                "threads_7": {"wall_s": d7["wall_s"], "note": "BGZF inflate + parse of the same BAM on 7 threads: what the reference's 7 "
                                                                              "samtools children must at least do before the CPU port's work starts"}},
                "note": "process wall clock includes CUDA context creation and process start; in_process.wall_s is measured inside main()"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


DUMP_TEXT_SAMPLE = 1 << 20           # bytes of each BED text kept by --dump-outputs (a seeded sample when the text is longer)
DUMP_MAX_WINDOWS = 6_500_000         # float64 window sums kept (the whole 25-contig genome has 6,176,584 windows at W=500)
DUMP_MAX_RUNS = 100_000


def fixed_sample(a, cap, seed):
    """a itself when it has at most cap elements, else cap elements at seeded positions (in order)"""
    if a.size <= cap:
        return a
    return a[np.sort(np.random.default_rng(seed).integers(0, a.size, cap))]


def dump_outputs(out_dir, resident, texts):
    """resident: per contig (window sums, run starts, run classes) of the resident step; texts: per contig (.depth.bed,
    .callable.bed) bytes of the drop-in call.  Writes out_dir/*.npy; integers are exact in float64."""
    def text_sample(parts, seed):
        return fixed_sample(np.frombuffer(b"".join(parts), np.uint8), DUMP_TEXT_SAMPLE, seed).astype(np.float32)
    arrays = {
        "depth_contig_sizes": np.array([(ws.size, rs.size) for ws, rs, _ in resident], np.float64),
        "depth_window_sum": fixed_sample(np.concatenate([r[0] for r in resident]).astype(np.float64), DUMP_MAX_WINDOWS, 1),
        "depth_run_start": fixed_sample(np.concatenate([r[1] for r in resident]).astype(np.float64), DUMP_MAX_RUNS, 2),
        "depth_run_class": fixed_sample(np.concatenate([r[2] for r in resident]).astype(np.float64), DUMP_MAX_RUNS, 2),
        "e2e_text_lengths": np.array([(len(h), len(c)) for h, c in texts], np.float64),
        "e2e_depth_bed_bytes": text_sample([t[0] for t in texts], 3),
        "e2e_callable_bed_bytes": text_sample([t[1] for t in texts], 4),
    }
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[dump] {len(arrays)} arrays, {total} bytes -> {out_dir}")


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("GL_BENCH_WORKLOAD", "wgs"), choices=["wgs", "chr20"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-path extras (int32 / general path / packed e2e variants)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the timed paths as DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        return run_reference(args)

    rank, world, local = dist_env()
    dist = None
    os.environ.setdefault("NCCL_DEBUG", "WARN")          # as in round 1: NCCL's one-line version banner precedes the JSON line (the last line of stdout)
    from goleft_b200 import capi
    import glsynth
    if capi.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; goleft_b200 has no CPU fallback")

    # ---- NUMA placement BEFORE any pinned allocation or pool thread exists: this rank's threads and staging buffers go
    #      next to its GPU's PCIe root; ranks that share a socket split its cores.
    nodes = [capi.device_numa_node(d) for d in range(world)] if world <= capi.device_count() else [-1] * world
    my_node = nodes[local] if local < len(nodes) else -1
    share = [r for r in range(world) if nodes[r] == my_node] if my_node >= 0 else list(range(world))
    node, n_cpus = capi.bind_numa_for_device(local, share.index(local) if local in share else 0, len(share))
    if node < 0:
        n_cpus = max(1, (os.cpu_count() or 1) // world)
        os.environ.setdefault("GL_THREADS", str(n_cpus))

    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # ---- this rank's share of the workload
    contigs = contig_list(args.workload, world)
    lengths = [c[1] for c in contigs]
    if args.workload == "wgs":
        bin_of, load = capi.lpt_assign(lengths, world)
        mine = [i for i in range(len(contigs)) if bin_of[i] == rank]
    else:
        load = np.array(lengths, np.int64)
        mine = [rank]
    total_bases = int(sum(lengths))
    my_bases = int(sum(lengths[i] for i in mine))

    ctx = capi.Ctx(local)
    t0 = time.time()
    work = []               # per contig: dict(name, L, h_s, h_e (pinned int32), d_a, d_d, d_l (device packed8), nb, n_win)
    for i in mine:
        nm, L, idx = contigs[i]
        h_s, h_e = glsynth.segments(L, idx, threads=n_cpus, alloc=ctx.pinned_empty)
        qa, qd, ql = capi.pack_segments8(h_s, h_e, threads=0)
        work.append({"name": nm, "L": L, "h_s": h_s, "h_e": h_e, "nseg": int(h_s.size), "nb": int(qa.size),
                     "d_a": ctx.dev_array(qa), "d_d": ctx.dev_array(qd), "d_l": ctx.dev_array(ql),
                     "p8_bytes": int(qa.nbytes + qd.nbytes + ql.nbytes), "n_win": (L - 1) // W + 1, "qa": qa, "qd": qd, "ql": ql})
    nseg = sum(w["nseg"] for w in work)
    log(f"[rank {rank}] numa node {node}, {n_cpus} cpus; {len(work)} contigs, {my_bases} bp, {nseg} segments in {time.time() - t0:.1f}s")
    max_win = max(w["n_win"] for w in work)
    longest_name = max((w["name"] for w in work), key=len)
    o_hd = ctx.pinned_empty(int(capi.lib.gl_depth_text_bound(longest_name.encode(), max_win)), np.uint8)
    o_ca = ctx.pinned_empty(max(1 << 20, max(w["L"] for w in work) // 64), np.uint8)
    ctx.flush_l2()

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    def step_resident(keep=None):
        for w in work:
            ctx.depth_begin(0, w["L"])
            ctx.depth_add_segments_packed8_device(w["d_a"], w["d_d"], w["d_l"], w["nb"])
            ctx.depth_reduce(W, MINCOV, MAXMEAN, STEP)
            if keep is not None:
                keep.append((ctx.depth_get_windows(),) + ctx.depth_get_runs())

    text_bytes = [0, 0]
    tr = {"h2d": 0, "pack_s": 0.0, "escaped": 0, "paths": set(), "kinds": set()}

    # ---- e2e runs TWO lanes per GPU: two gl_ctx on the same device, one host thread each (a ctx is one host thread at a time;
    #      different ctxs are independent — SURVEY 8(b)), the rank's contigs dealt to the lanes longest first.  While lane A waits
    #      for its contig's last upload chunk, kernels, text and D2H, lane B packs and uploads the next contig: the call's serial
    #      tail disappears behind the other lane's PCIe time.  Every call is still the synchronous drop-in call.
    from concurrent.futures import ThreadPoolExecutor
    ctx_b = capi.Ctx(local)
    lanes = [{"ctx": ctx, "o": (o_hd, o_ca), "work": []},
             {"ctx": ctx_b, "o": (ctx_b.pinned_empty(o_hd.size, np.uint8), ctx_b.pinned_empty(o_ca.size, np.uint8)), "work": []}]
    lane_load = [0, 0]
    for w in sorted(work, key=lambda w: -w["nseg"]):
        k = 0 if lane_load[0] <= lane_load[1] else 1
        lanes[k]["work"].append(w); lane_load[k] += w["nseg"]
    lane_pool = ThreadPoolExecutor(max_workers=2)

    def run_lane(lane, keep=None):
        c, o = lane["ctx"], lane["o"]
        hb = cb = 0
        h2d, pack_s, esc = 0, 0.0, 0
        kinds, paths = set(), set()
        for w in lane["work"]:
            hl, cl = c.depth_bed_contig(w["name"], w["L"], w["h_s"], w["h_e"], W, MINCOV, MAXMEAN, STEP, threads=0, out=o, raw=True)
            if keep is not None:
                keep.append((bytes(o[0][:hl]), bytes(o[1][:cl])))
            hb += hl; cb += cl
            kind, ps, nb, ne = c.depth_transport_stats()
            h2d += nb; pack_s += ps; esc += ne
            kinds.add(kind); paths.add(c.depth_last_path())
        return hb, cb, h2d, pack_s, esc, kinds, paths

    def step_e2e(n_lanes=2):
        if n_lanes == 1:
            res = [run_lane({"ctx": ctx, "o": (o_hd, o_ca), "work": work})]
        else:
            res = [f.result() for f in [lane_pool.submit(run_lane, ln) for ln in lanes]]
        text_bytes[0], text_bytes[1] = sum(r[0] for r in res), sum(r[1] for r in res)
        tr["h2d"], tr["pack_s"], tr["escaped"] = sum(r[2] for r in res), sum(r[3] for r in res), sum(r[4] for r in res)
        for r in res:
            tr["kinds"] |= r[5]; tr["paths"] |= r[6]

    # ---- warm-up (also sizes every grow-only buffer)
    for _ in range(args.warmup):
        step_resident()
    n_runs = 0
    for w in work:
        ctx.depth_begin(0, w["L"])
        ctx.depth_add_segments_packed8_device(w["d_a"], w["d_d"], w["d_l"], w["nb"])
        ctx.depth_reduce(W, MINCOV, MAXMEAN, STEP)
        w["n_runs"] = ctx.depth_result_sizes()[1]
        n_runs += w["n_runs"]
    for _ in range(args.warmup):
        step_e2e()

    # ---- e2e parity check (outside the timed regions): the bytes of the drop-in call against the oracle's walker
    e2e_check = None
    if rank == 0:
        from oracle import loader as orc
        mid = [w for w in work if 1_000_000 <= w["L"] <= 70_000_000]
        pick = ([min(mid, key=lambda w: w["L"])] if mid else []) + [w for w in work if w["L"] < 1_000_000]
        checked = []
        ok = True
        for w in pick:
            got = ctx.depth_bed_contig(w["name"], w["L"], w["h_s"], w["h_e"], W, MINCOV, MAXMEAN, STEP)
            s_, e_ = sorted_copy(np.array(w["h_s"]), np.array(w["h_e"]))
            hd, ca = [], []
            for cs, ce in orc.gen_chunks(w["L"], W):
                lo = max(0, int(np.searchsorted(s_, cs - 1024, "left")) - 4096)
                hi = int(np.searchsorted(s_, ce, "left"))
                d = orc.pileup_diff(s_[lo:hi], e_[lo:hi], cs, ce)
                h, c = orc.walk_chunk(w["name"], cs, ce, W, MINCOV, MAXMEAN, d)
                hd.append(h); ca.append(c)
            ok = ok and got[0] == b"".join(hd) and got[1] == b"".join(ca)
            checked.append(w["name"])
        e2e_check = {"contigs": checked, "bytes_equal_oracle_walker": bool(ok),
                     "inside_timed_region": ["host pool: int32 -> fixed-block packed16 (pipelined with the upload)", "H2D packed16 words (pinned)", "depth_unpack16_kernel", "K_index/K_fused/K_gather", "device %.4g row formatter (bed_rows/scan/emit)",
                                             "D2H .depth.bed + .callable.bed bytes (pinned)"],
                     "outside": ["BGZF inflate + BAM record parse (the feeder; see cli_wallclock)"]}
        if not ok:
            raise SystemExit("bench.py: e2e text differs from the oracle walker")

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- timed: device-resident.  L2 is flushed (256 MiB memset) before every timed step; each step is timed with CUDA
    #      events on the ctx stream (every launch of the step is on that stream) and the K step times are summed.
    barrier()
    l0 = ctx.launch_count()
    ms = 0.0
    for _ in range(args.steps):
        ctx.flush_l2()
        ctx.timer_start()
        step_resident()
        ms += ctx.timer_stop_ms()
    launches = ctx.launch_count() - l0
    barrier()

    # ---- timed: end to end through the C ABI with pinned host buffers (H2D + kernels + formatter + D2H inside)
    #      Host wall clock around the step: every call is synchronous (its results are in host memory when it returns), so the
    #      wall time bounds the device time of both lanes from above.
    ms_e2e = 0.0
    for _ in range(args.steps):
        ctx.flush_l2()
        ctx.sync(); ctx_b.sync()
        te0 = time.perf_counter()
        step_e2e()
        ms_e2e += (time.perf_counter() - te0) * 1e3
    barrier()
    ms_e2e_one_lane = 0.0                                  # the same step through one ctx, contig after contig (reported beside it)
    n_one = max(3, args.steps // 4)
    for _ in range(n_one):
        ctx.flush_l2(); ctx.sync()
        te0 = time.perf_counter()
        step_e2e(1)
        ms_e2e_one_lane += (time.perf_counter() - te0) * 1e3
    ms_e2e_one_lane /= n_one
    barrier()
    if args.dump_outputs and rank == 0:
        resident, texts = [], []
        step_resident(resident)
        run_lane({"ctx": ctx, "o": (o_hd, o_ca), "work": work}, texts)
        dump_outputs(args.dump_outputs, resident, texts)

    # ---- per-kernel live timing for the roofline: CUDA events on the launching stream around every kernel of the same
    #      step (library-side, gl_profile_*), averaged over the repetitions
    def kernel_times(reps, step):
        ctx.profile_enable(True)
        ctx.profile_read()
        acc, cnt = {}, {}
        for _ in range(reps):
            ctx.flush_l2()
            step()
            for nm, t in ctx.profile_read():
                acc[nm] = acc.get(nm, 0.0) + t
                cnt[nm] = cnt.get(nm, 0) + 1
        ctx.profile_enable(False)
        return {k: v / reps for k, v in acc.items()}, {k: v // reps for k, v in cnt.items()}
    reps = max(3, min(args.steps, 10))
    k_ms, k_n = kernel_times(reps, step_resident)
    path = ctx.depth_last_path()
    k_ms_e2e, _ = kernel_times(min(reps, 3), lambda: step_e2e(1))

    # ---- extras (rank 0, N=1): the other entries on the largest contig that fits the old chr20-sized buffers
    extras = {}
    if world == 1 and not args.no_extras:
        w = min(work, key=lambda w: abs(w["L"] - glsynth.CHR20_LEN))
        L, nm = w["L"], w["name"]
        d_s, d_e = ctx.dev_array(w["h_s"]), ctx.dev_array(w["h_e"])
        h8 = [ctx.pinned_empty(a.size, a.dtype) for a in (w["qa"], w["qd"], w["ql"])]
        for dst, src in zip(h8, (w["qa"], w["qd"], w["ql"])):
            dst[:] = src

        def one_resident():
            ctx.depth_begin(0, L)
            ctx.depth_add_segments_packed8_device(w["d_a"], w["d_d"], w["d_l"], w["nb"])
            ctx.depth_reduce(W, MINCOV, MAXMEAN, STEP)

        def one_int32():
            ctx.depth_begin(0, L)
            ctx.depth_add_segments_device(d_s, d_e, w["nseg"])
            ctx.depth_reduce(W, MINCOV, MAXMEAN, STEP)

        def timed_dev(fn, n):
            for _ in range(2):
                fn()
            t = 0.0
            for _ in range(n):
                ctx.flush_l2(); ctx.timer_start(); fn(); t += ctx.timer_stop_ms()
            return t / n

        def timed_host(fn, n):
            for _ in range(2):
                fn()
            t = 0.0
            for _ in range(n):
                ctx.flush_l2(); ctx.sync()
                t0_ = time.perf_counter(); fn(); t += (time.perf_counter() - t0_) * 1e3
            return t / n
        n_x = max(5, min(args.steps, 20))
        x_res = timed_dev(one_resident, n_x)
        x_res_k, _ = kernel_times(5, one_resident)
        x_i32 = timed_dev(one_int32, n_x)
        x_i32_k, _ = kernel_times(5, one_int32)
        ctx.depth_set_path(4)
        x_gen = timed_dev(one_int32, max(3, n_x // 2))
        x_gen_k, _ = kernel_times(3, one_int32)
        ctx.depth_set_path(2)
        x_hbm = timed_dev(one_int32, max(3, n_x // 2))
        x_hbm_k, _ = kernel_times(3, one_int32)
        ctx.depth_set_path(0)
        x_e2e_text = timed_host(lambda: ctx.depth_bed_contig(nm, L, w["h_s"], w["h_e"], W, MINCOV, MAXMEAN, STEP, out=(o_hd, o_ca), raw=True), n_x)
        x_e2e_stats = ctx.depth_transport_stats() + (ctx.depth_last_path(), [x * 1e3 for x in ctx.depth_transport_phases()])
        os.environ["GL_BED_PACK"] = "0"
        x_e2e_plain = timed_host(lambda: ctx.depth_bed_contig(nm, L, w["h_s"], w["h_e"], W, MINCOV, MAXMEAN, STEP, out=(o_hd, o_ca), raw=True), n_x)
        del os.environ["GL_BED_PACK"]
        x_e2e_p8 = timed_host(lambda: ctx.depth_bed_contig_packed8(nm, L, h8[0], h8[1], h8[2], W, MINCOV, MAXMEAN, STEP, out=(o_hd, o_ca), raw=True), n_x)
        run_cap = L // 16 + 4096
        o_sum, o_rs, o_rc = ctx.pinned_empty(w["n_win"], np.int64), ctx.pinned_empty(run_cap, np.int32), ctx.pinned_empty(run_cap, np.uint8)
        x_k_only = timed_host(lambda: ctx.depth_region_packed8(0, L, h8[0], h8[1], h8[2], W, MINCOV, MAXMEAN, STEP, out=(o_sum, o_rs, o_rc)), n_x)
        t_pack = timed_host(lambda: capi.pack_segments8(w["h_s"], w["h_e"], threads=0), 5)
        extras = {"contig": nm, "bases": L, "segments": w["nseg"],
                  "resident_packed8": {"ms": x_res, "value": L / x_res / 1e3, "kernel_ms": x_res_k},
                  "resident_int32": {"ms": x_i32, "value": L / x_i32 / 1e3, "kernel_ms": x_i32_k,
                                     "note": "plain int32 (start,end) device arrays: K_index + K_fused + K_gather"},
                  "general_path": {"ms": x_gen, "value": L / x_gen / 1e3, "kernel_ms": x_gen_k,
                                   "note": "bucketed events (any order, any segment length): K_evcount + K_evscan + K_evscatter + K_evtile + K_gather"},
                  "hbm_difference_array_path": {"ms": x_hbm, "value": L / x_hbm / 1e3, "kernel_ms": x_hbm_k,
                                                "note": "the pipeline north_star sketches, on request (gl_depth_set_path(2)): memset + K_scatter "
                                                        "(red.global) + K_super + K_scan + K_gather"},
                  "e2e_text_int32": {"ms": x_e2e_text, "value": L / x_e2e_text / 1e3, "h2d_bytes": x_e2e_stats[2], "transport": x_e2e_stats[0],
                                     "host_pack_ms": x_e2e_stats[1] * 1e3, "escaped_segments": x_e2e_stats[3], "depth_path": x_e2e_stats[4],
                                     "host_phases_ms": dict(zip(("setup", "pack_and_enqueue_loop", "reduce_text_d2h"), x_e2e_stats[5])),
                                     "call": "gl_depth_bed_contig (what `e2e` times, on this contig alone): int32 arrays in, repacked by the host pool to "
                                             "fixed-block packed16 (4 B/segment) chunk by chunk while the previous chunk is on the wire"},
                  "e2e_text_int32_plain_upload": {"ms": x_e2e_plain, "value": L / x_e2e_plain / 1e3, "h2d_bytes": 8 * w["nseg"],
                                                  "call": "the same call with GL_BED_PACK=0: the int32 arrays go over PCIe as they are (8 B/segment)"},
                  "e2e_text_packed8_words": {"ms": x_e2e_p8, "value": L / x_e2e_p8 / 1e3, "h2d_bytes": w["p8_bytes"],
                                             "call": "gl_depth_bed_contig_packed8: the feeder's own packed8 words (what the BAM decoder emits) in, BED bytes out"},
                  "e2e_kernels_only": {"ms": x_k_only, "value": L / x_k_only / 1e3, "h2d_bytes": w["p8_bytes"],
                                       "call": "gl_depth_region_packed8: packed8 words in, int64 window sums + runs out, no text (round 1's e2e)"},
                  "host_pack_ms": {"gl_pack_segments8_mt": t_pack, "threads": n_cpus,
                                   "note": "int32 -> packed8 on the host pool; NOT inside e2e (e2e uploads the int32 arrays as they are)"}}
        d_s.free(); d_e.free()
        # ---- other shapes of the same contig (VERDICT r1 #7): low coverage (thousands of class runs), maxmeandepth > 0,
        #      the reference's default W=250 (depth.go:164), long reads (20 kb segments -> the general path)
        try:
            extras["configs"] = config_legs(ctx, L, nm, n_cpus, timed_dev, timed_host, kernel_times, rank == 0)
        except Exception as ex:
            extras["configs"] = {"error": str(ex)[:300]}
        # ---- the product CLI on a real BAM of the same reads: BGZF inflate + record parse + GPU + text, wall clock
        try:
            extras["cli_wallclock"] = cli_wallclock(n_cpus)
        except Exception as ex:                              # the leg is informative; never let it take the bench line down
            extras["cli_wallclock"] = {"error": str(ex)[:300]}
    clocks = sampler.stop() if rank == 0 else None

    # ---- the path's one collective (BASELINE configs[4]): the depthwed n-sites x n-samples matrix, 500 samples x 6,176,584
    #      windows of int32, sample-sharded; every rank aggregates its columns chunk by chunk and all-gathers each finished chunk
    #      over NVLink on a second stream while the next chunk is aggregated.  Verified on every rank.
    depthwed = None
    cohort = None
    if not args.no_extras:
        comm_ok = dist is not None
        if dist is not None:
            try:
                comm_setup(ctx, dist, rank, world)
            except Exception as ex:
                comm_ok, depthwed = False, {"error": "gl_comm_init: " + str(ex)[:300]}
        if comm_ok:
            try:
                depthwed = depthwed_leg(ctx, dist, rank, world, local)
            except Exception as ex:
                depthwed = {"error": str(ex)[:300]}
        # ---- BASELINE configs[3]: the 2504-sample indexcov cohort, samples sharded over the ranks (+ all-gather of the depths at N>1)
        try:
            cohort = indexcov_cohort_leg(ctx, dist if comm_ok else None, rank, world if comm_ok else 1)
        except Exception as ex:
            cohort = {"error": str(ex)[:300]}

    per_rank = None
    if dist is not None:
        import torch
        t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
        g = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        per_rank = [[float(x[0]) / args.steps, float(x[1]) / args.steps] for x in g]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = (float(x) for x in t)
        cnt = torch.tensor([float(launches), float(nseg), float(n_runs), float(text_bytes[0] + text_bytes[1]), float(tr["h2d"])],
                           dtype=torch.float64, device="cuda")
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        launches_all, nseg_all, n_runs_all, d2h_all, h2d_all = (int(x) for x in cnt)
    else:
        launches_all, nseg_all, n_runs_all, d2h_all, h2d_all = launches, nseg, n_runs, text_bytes[0] + text_bytes[1], tr["h2d"]

    if rank == 0:
        peak, peak_src = peaks()
        ms_step = ms / args.steps
        ms_e2e_step = ms_e2e / args.steps
        units = total_bases if args.workload == "wgs" else world * lengths[0]
        val = units / (ms_step * 1e-3) / 1e6
        e2e_val = units / (ms_e2e_step * 1e-3) / 1e6
        # ALGORITHMIC bytes (DESIGN.md §3): rank 0's share, per step
        n_win0 = sum(w["n_win"] for w in work)
        p8_bytes0 = sum(w["p8_bytes"] for w in work)
        survey_bytes = 8 * nseg + 8 * my_bases + 12 * n_win0 + 9 * n_runs          # SURVEY.md §8(d): HBM difference-array pipeline
        own = {"depth_fused8_kernel": p8_bytes0 + 8 * n_win0 + 5 * n_runs,
               "depth_tileidx8_kernel": sum(4 * w["nb"] + 8 * ((w["L"] - 1) // 4096 + 1) for w in work)}
        dom = max((k for k in k_ms if k.startswith("depth_")), key=lambda k: k_ms[k])
        n_launch = max(1, k_n.get(dom, 1))
        dom_ms_launch = k_ms[dom] / n_launch
        achieved = survey_bytes / n_launch / (dom_ms_launch * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic(dom)
        out = {"metric": METRIC, "value": val, "unit": "Mbases/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
               "scaling": "strong" if args.workload == "wgs" else "weak",
               "vs_baseline": None, "dtype": "int32", "data": "synthetic",
               "config": {"workload": WORKLOADS[args.workload], "window": W, "mincov": MINCOV, "run_break": STEP,
                          "segments": nseg_all, "runs": n_runs_all, "contigs": len(contigs), "contigs_rank0": [w["name"] for w in work],
                          "assignment": "gl_lpt_assign (longest contig first onto the least loaded GPU)" if args.workload == "wgs" else "one replica per rank",
                          "imbalance": float(load.max() / (load.sum() / world)) if args.workload == "wgs" else 1.0,
                          "resident_format": "packed8 (64-slot blocks: int32 anchor + uint8 start delta + uint8 length per segment)",
                          "path": {1: "fused (sorted int32 segments -> smem difference tiles)", 2: "general (HBM difference array)",
                                   3: "packed8 (packed words -> smem difference tiles)"}.get(path, str(path)),
                          "l2": "L2 flushed (256 MiB memset) before every timed step; per-step CUDA-event times summed; inputs (>= 1.3 GB per step at N=1) exceed L2",
                          "numa": {"node": node, "cpus": n_cpus}},
               "e2e": {"value": e2e_val, "unit": "Mbases/s", "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all,
                       "ms_per_step": ms_e2e_step, "kernel_ms_rank0": k_ms_e2e,
                       "call": "gl_depth_bed_contig per contig: int32 (start,end) segments in pinned host memory -> .depth.bed + .callable.bed bytes in pinned host memory",
                       "transport": "auto (fixed-block packed16, 4 B/segment, packed by 16 pool threads, when the rank's host pool has >= 48 threads; else plain int32, 8 B/segment)",
                       "host_pool_threads": int(capi.lib.glhost_pool_size()),
                       "lanes": "2 gl_ctx per GPU, one host thread each, the rank's contigs dealt longest first; every call is the synchronous drop-in call",
                       "one_lane_ms_per_step_rank0": ms_e2e_one_lane,
                       "rank0": {"transport": sorted(tr["kinds"]), "host_pack_ms_per_step": tr["pack_s"] * 1e3, "escaped_segments": tr["escaped"],
                                 "depth_paths": sorted(tr["paths"]),
                                 "note": "gl_depth_transport_stats / gl_depth_last_path per contig: transport 16 = fixed-block packed16, 0 = plain int32; "
                                         "path 1 = fused int32 kernels"}},
               "e2e_check": e2e_check,
               "gpu_launches": int(launches_all),
               "roofline": {"bound": "hbm", "kernel": dom, "unit": "GB/s", "peak": peak, "peak_source": peak_src,
                            # contract definition: SURVEY.md §8(d)'s algorithmic bytes x the units one launch processes; the dominant
                            # kernel performs that whole per-base pipeline on chip, so this is its EFFECTIVE bandwidth ...
                            "achieved": achieved, "frac": achieved / peak,
                            "alg_bytes_per_launch": survey_bytes / n_launch, "launches_per_step_rank0": n_launch,
                            "ms_per_launch": dom_ms_launch,
                            "basis": "SURVEY.md 8(d): 8*N_seg + 8*L + 12*ceil(L/W) + 9*runs per contig (HBM difference-array pipeline), "
                                     "averaged over the rank's contig launches; effective bandwidth of the kernel that does that pipeline's work",
                            # ... and these are the bytes the kernel itself has to move, with the ncu DRAM traffic beside them:
                            "own": {"alg_bytes_per_launch": own.get(dom, 0) / n_launch,
                                    "achieved": own.get(dom, 0) / n_launch / (dom_ms_launch * 1e-3) / 1e9,
                                    "frac": own.get(dom, 0) / n_launch / (dom_ms_launch * 1e-3) / 1e9 / peak,
                                    "note": "packed words in + 8 B/window + 5 B/run out: the 8 B/base difference array never exists in HBM; "
                                            "the kernel is issue-bound, not HBM-bound (profiles/)"},
                            "traffic": traffic, "traffic_source": traffic_src, "kernel_ms": k_ms,
                            "step": {"survey_alg_bytes": survey_bytes, "achieved": survey_bytes / (ms_step * 1e-3) / 1e9,
                                     "frac": survey_bytes / (ms_step * 1e-3) / 1e9 / peak}},
               "clocks": clocks}
        if depthwed is not None:
            out["depthwed_allgather"] = depthwed
        if cohort is not None:
            out["indexcov_cohort"] = cohort
        if per_rank is not None:
            out["per_rank_ms"] = {"resident": [p[0] for p in per_rank], "e2e": [p[1] for p in per_rank]}
        if extras:
            out["single_contig"] = extras
        if not args.no_cpu_baseline and world == 1:         # rank 0 at N=1 only (the other ranks' feeders share the host cores at N>1)
            from oracle import loader as orc       # cpu_baseline leg: the oracle port timed on this box's host cores
            threads = os.cpu_count() or 1
            os.sched_setaffinity(0, range(threads))          # the CPU leg may use every core of the box
            cc = [(w["name"], w["L"]) + sorted_copy(np.array(w["h_s"]), np.array(w["h_e"])) for w in work]
            reps_c, tot, chunks = 0, 0.0, 0
            cpu_genome_pass(orc, cc[-1:], threads)
            while reps_c < 3 and tot < 20.0:
                dt, _, chunks = cpu_genome_pass(orc, cc, threads)
                tot += dt; reps_c += 1
            out["cpu_baseline"] = {"value": units / (tot / reps_c) / 1e6, "unit": "Mbases/s", "cores": min(threads, chunks),
                                   "cores_available": threads, "kind": "port",
                                   "sample": f"{reps_c} x the whole workload ({chunks} chunks of 10 Mb, one worker per chunk = the reference's unit of "
                                             "parallelism, all host threads): per-base counting + window/class walk + BED text; "
                                             "BGZF inflate and samtools text print/parse excluded"}
        print(json.dumps(out), flush=True)

    lane_pool.shutdown()
    ctx_b.close()
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
