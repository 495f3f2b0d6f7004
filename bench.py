#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on its configs[1] workload: batched zstd_decompress of 16,384 independent
64 KiB frames (1 GiB of content) per B200, frames produced by the reference's libzstd at level 3.

    python bench.py --gpus N --steps K --warmup W            our CUDA path through the C ABI (libzstdlite_gpu.so)
    python bench.py --impl reference ...                      the reference's own libzstd on the host cores

One JSON line on stdout (rank 0).  `value`  = whole-job GB/s of uncompressed bytes, inputs resident in HBM;
`e2e` = same metric through the C ABI with pinned HOST buffers (H2D of the frames and D2H of the output inside the
timed region); `roofline` = dominant kernel against the measured HBM copy bandwidth; `cpu_baseline` = the reference's
libzstd, frame-parallel on all host cores, on a bounded sample of the same frames; `compress` = the level-1/level-3
compressor on configs[2] (4 GiB per GPU as 128 KiB frames, made on the device; reported beside the headline at every N;
BASELINE.json's metric is "decompress+compress").
Multi-GPU: frames are independent, so every rank decodes its own 16,384-frame shard (weak scaling, no collective on
the data path; barrier + max-over-ranks timing only).

oracle/ is used here only for (1) producing the compressed input corpus with the reference's libzstd before any timed
region, (2) the cpu_baseline leg and (3) --impl reference.  The measured path never touches it.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MIX = (("text", 0.4), ("rdf", 0.4), ("lowent", 0.1), ("rand", 0.1))          # SURVEY.md 8d, config 2
METRIC = "decompress_GBps_uncompressed"
UNIT = "GB/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DUMP_BYTES = 8 << 20          # decoded bytes sampled by --dump-outputs: 32 MiB as float32, the rest of 64 MB left to the per-frame results


def dump_outputs(out_dir, torch, dst, res, n, fb):
    """--dump-outputs: what the last timed step handed its caller, as .npy files under `out_dir` -- every frame's result
    (float64: the decoded size, or -code for a ZSTD error, which is returned as 2**64 - code and would round to one value as a
    float) and the decoded bytes (float32) of a fixed, seeded sample of frames, rows in ascending frame order; the sample covers
    at most DUMP_BYTES bytes, so two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    k = max(1, min(n, DUMP_BYTES // fb))
    rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    sample = dst[:n * fb].view(n, fb)[torch.from_numpy(rows).to(dst.device), :min(fb, DUMP_BYTES)]
    np.save(os.path.join(out_dir, "decoded_sample.npy"), sample.float().cpu().numpy())
    results = np.array([r if r < 2**63 else -(2**64 - r) for r in res], dtype=np.float64)
    np.save(os.path.join(out_dir, "frame_results.npy"), results if results.nbytes <= (16 << 20) else results[rows])


def make_corpus(nframes, frame_bytes, level=3, pool=64, seed_shift=0):
    """-> (raw [nframes, frame_bytes] uint8, list of compressed frames).  Every frame is distinct (rotated copies of `pool`
    frames per family) and the families are interleaved by a fixed permutation; the frames are compressed by the reference's
    libzstd on all host cores (oracle/cpu_bench.c) before any timed region."""
    from zstdlite_b200 import corpus
    from oracle import cpubench
    data, fams = corpus.mixed_frames(nframes, frame_bytes, mix=MIX, pool=pool, rotate=True)
    data = data[np.random.default_rng(20261017 + seed_shift).permutation(nframes)]
    bound = frame_bytes + (frame_bytes >> 8) + 64
    fs = cpubench.FrameSet(data.reshape(-1), [frame_bytes] * nframes)
    _, res, dst, doffs = cpubench.run("compress", fs, [bound] * nframes, os.cpu_count() or 1, level=level)
    frames = [dst[int(o):int(o) + int(r)].tobytes() for o, r in zip(doffs, res)]
    return data, frames


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 50 ms during the timed region
    (same fields as the nvidia-smi line in B200_PROFILING.md; nvidia-smi's piped output is block-buffered)."""

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.sm, self.reasons, self.max = [], set(), None
        self._stop = threading.Event()
        self.t = None
        self.err = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.idx
            if vis:
                try:
                    idx = int(vis.split(",")[self.idx])
                except (ValueError, IndexError):
                    pass
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                     "hw_power_brake_slowdown": 0x80}
            while not self._stop.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except AttributeError:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                self._stop.wait(0.05)
        except Exception as e:                                           # NVML missing: say so in the JSON line
            self.err = repr(e)

    def start(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def stop(self):
        self._stop.set()
        if self.t:
            self.t.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max,
               "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.err:
            out["error"] = self.err
        return out


def cpu_leg(frames_sample, frame_bytes, budget_s, threads):
    """reference libzstd, frame-parallel on `threads` host cores -> (GB/s, seconds per pass, passes)."""
    from oracle import cpubench
    blob = np.frombuffer(b"".join(frames_sample), dtype=np.uint8)
    fs = cpubench.FrameSet(blob, [len(f) for f in frames_sample])
    caps = [frame_bytes] * len(frames_sample)
    t_pass, *_ = cpubench.run("decompress", fs, caps, threads)        # warm-up pass (page faults, contexts)
    passes = max(1, min(50, int(budget_s / max(t_pass, 1e-3))))
    best, *_ = cpubench.run("decompress", fs, caps, threads, passes=passes)
    return len(frames_sample) * frame_bytes / best / 1e9, best, passes


def cpu_compress_variants(buf, frame_bytes, level, threads, budget_s=4.0):
    """BASELINE.md section 3 on `buf` (uint8 array, a whole number of frames): the reference's libzstd (i) one thread over the frames,
    (ii) ZSTD_c_nbWorkers = threads on the buffer as ONE frame (the reference's num_threads semantics, src/cctx.c:269-277), (iii) frame-parallel
    on `threads` cores.  -> dict of GB/s (uncompressed bytes) and compressed sizes."""
    from oracle import cpubench
    n = buf.size // frame_bytes
    bound = frame_bytes + (frame_bytes >> 8) + 64
    fs = cpubench.FrameSet(buf, [frame_bytes] * n)
    t_fp, res, _, _ = cpubench.run("compress", fs, [bound] * n, threads, level=level)
    passes = max(1, min(5, int(budget_s / 3 / max(t_fp, 1e-3))))
    t_fp = min(t_fp, cpubench.run("compress", fs, [bound] * n, threads, level=level, passes=passes)[0])
    n1 = max(1, min(n, int(n * (budget_s / 3) / max(t_fp * threads, 1e-3))))          # one thread: a share it finishes in ~budget/3
    fs1 = cpubench.FrameSet(buf[:n1 * frame_bytes], [frame_bytes] * n1)
    t_1, *_ = cpubench.run("compress", fs1, [bound] * n1, 1, level=level)
    t_w, size_w = cpubench.run_workers(buf, level=level, workers=threads, passes=2)
    return {"cores": threads, "level": level, "frame_parallel_GBps": buf.size / t_fp / 1e9, "one_thread_GBps": n1 * frame_bytes / t_1 / 1e9,
            "nbWorkers_one_frame_GBps": buf.size / t_w / 1e9, "frames": n, "one_thread_frames": n1,
            "frame_parallel_bytes": int(res.sum()), "nbWorkers_one_frame_bytes": size_w, "kind": "reference",
            "sample": f"{n} x {frame_bytes // 1024} KiB slabs of the GPU's buffer ({buf.size / 2**20:.0f} MiB) copied to the host; one_thread over the first {n1}"}


def run_reference(args, rank, world):
    """The reference's own libzstd on the host cores, frame-parallel with every host thread, over ALL frames of the workload."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    data, frames = make_corpus(args.frames, args.frame_bytes)
    from oracle import cpubench, ref
    blob = np.frombuffer(b"".join(frames), dtype=np.uint8)
    fs = cpubench.FrameSet(blob, [len(f) for f in frames])
    caps = [args.frame_bytes] * len(frames)
    for _ in range(args.warmup):
        cpubench.run("decompress", fs, caps, threads)
    times = [cpubench.run("decompress", fs, caps, threads)[0] for _ in range(args.steps)]
    total = sum(times)
    val = len(frames) * args.frame_bytes * args.steps / total / 1e9
    desc = f"all {args.frames} frames of one GPU's shard, {threads} threads, one DCtx per thread (system libzstd {ref.version()}, oracle/cpu_bench.c)"
    out = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8", "data": "synthetic", "impl": "reference",
           "config": workload_config(args, world),
           "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "reference", "sample": desc},
           "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def workload_config(args, world):
    return {"workload": f"configs[1]: batched zstd_decompress of {args.frames} independent {args.frame_bytes // 1024} KiB frames "
                        f"({args.frames * args.frame_bytes / 2**30:.2f} GiB content) per GPU, libzstd level-3 frames, families text/rdf/lowent/rand 40/40/10/10",
            "frames_per_gpu": args.frames, "frame_bytes": args.frame_bytes, "level": 3, "checksum": False,
            "sharding": f"{world} x independent frame shards, no collective",
            "cache": "working set (compressed in + 1 GiB out per step) exceeds the 126 MB L2; no explicit flush"}


def measured_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback (of fallback)"


def compress_traffic(level):
    """DRAM bytes of the compress kernels from the committed ncu capture (profiles/compress_kernel_traffic.json), or None."""
    path = os.path.join(ROOT, "profiles", "compress_kernel_traffic.json")
    try:
        return json.load(open(path)).get(f"level{level}")
    except (OSError, ValueError):
        return None


def compress_traffic_bytes(level, nblocks):
    """the capture's total DRAM bytes scaled to `nblocks` blocks (the capture holds fewer blocks of the same mix), or None"""
    t = compress_traffic(level)
    if not t:
        return None, None
    return int(t["dram_bytes_total"] * nblocks / t["blocks_in_capture"]), t.get("source")


def pin_to_gpu_numa_node(local):
    """Bind this process (and the pinned host buffers it allocates afterwards) to the CPUs NVML reports as local to its GPU: with one
    process per GPU on a two-socket box, host staging otherwise lands on whichever node the launcher started on."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        idx = local
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                idx = int(vis.split(",")[local])
            except (ValueError, IndexError):
                pass
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        ncpu = os.cpu_count() or 1
        words = nv.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1 and 64 * w + b < ncpu}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
        return {"cpus": len(cpus) if cpus else len(allowed), "of": len(allowed), "bound": bool(cpus and cpus != allowed)}
    except Exception as e:                                            # no NVML / not permitted: run unbound, say so
        return {"error": repr(e)}


def pcie_probe(torch, dist, dev, world, h2d_bytes, d2h_bytes, reps=3):
    """Raw ceiling of the end-to-end arm: the step's H2D and D2H volumes as two plain concurrent cudaMemcpyAsync between pinned host
    memory and HBM, on every rank at once -> (ms of the slower direction, max over ranks)."""
    hs = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    hd = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    ds = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
    dd = torch.zeros(d2h_bytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    best = None
    for _ in range(reps + 1):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
        a0, a1, b0, b1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        with torch.cuda.stream(s1):
            a0.record(); ds.copy_(hs, non_blocking=True); a1.record()
        with torch.cuda.stream(s2):
            b0.record(); hd.copy_(dd, non_blocking=True); b1.record()
        torch.cuda.synchronize()
        t = max(a0.elapsed_time(a1), b0.elapsed_time(b1))
        best = t if best is None else min(best, t)
    if world > 1:
        tt = torch.tensor([best], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        best = float(tt[0])
    del hs, hd, ds, dd
    return best


def compress_leg(torch, dist, z, args, dev, rank, world):
    """configs[2]: a raw buffer of `--compress-frames` x 128 KiB slabs per GPU (default 32,768 = 4 GiB), made on the device, every
    slab an independent frame at levels 1 and 3, device-resident; all ranks run it (weak scaling, max-over-ranks time).  Rank 0
    checks a sample of frames through the reference's libzstd and compares sizes with libzstd on the same slabs."""
    from zstdlite_b200 import corpus
    n, fb = args.compress_frames, 131072
    src, pools, meta = corpus.device_mixed_slabs(n, fb, MIX, index=11 + rank, device=dev)
    bound = int(z._lib.lib().ZSTD_compressBound(fb))
    slot = (bound + 255) // 256 * 256
    dst = torch.zeros(n * slot + 64, dtype=torch.uint8, device=dev)
    out = {}
    for lvl in (1, 3):
        cctx = z.zstd_cctx(level=lvl)
        plan = z.BatchPlan([src.data_ptr() + i * fb for i in range(n)], [fb] * n, [dst.data_ptr() + i * slot for i in range(n)], [bound] * n)
        res = None
        for _ in range(2):
            res = plan.compress(cctx)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        cctx.set_stream(torch.cuda.current_stream().cuda_stream)
        t0.record()
        iters = 3
        for _ in range(iters):
            res = plan.compress(cctx)
        t1.record(); torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / iters
        # per-kernel times of the LAST device-resident call (read now: the end-to-end call below runs the pipelined chunks)
        L = z._lib.lib()
        kernel_ms = cctx.last_kernel_ms
        stages = {nm: L.zl_cctx_last_stage_ms(cctx._p, k) for k, nm in enumerate(("match", "parse", "literals", "sequences", "plan+assemble"))}
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        sizes = np.array(list(res), dtype=np.int64)
        assert not any(z.is_error(int(s)) for s in sizes), "compress errors"
        csize = int(sizes.sum())
        # end to end: the buffer as ONE pinned host buffer through zl_compress_split (what zstd_compress(frame_size=) calls): host-to-device
        # staging, kernels and the copy back of the multi-frame stream inside the timed region; every rank at once (N > 1: 1 GiB per rank)
        e2e = None
        if lvl == 3 and not args.no_compress_e2e:
            import ctypes as C
            ne = n if world == 1 else min(n, 8192)
            hsrc = torch.empty(ne * fb, dtype=torch.uint8).pin_memory(); hsrc.copy_(src.reshape(-1)[:ne * fb])
            hcap = ne * (bound + 8)
            hdst = torch.empty(hcap, dtype=torch.uint8).pin_memory()
            tt = []
            for _ in range(3):
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                t0w = time.time()
                r = L.zl_compress_split(cctx._p, C.c_void_p(hdst.data_ptr()), hcap, C.c_void_p(hsrc.data_ptr()), ne * fb, fb, None, 0)
                tt.append(time.time() - t0w)
                assert not z.is_error(r), z.error_name(r)
            assert int(r) == int(sizes[:ne].sum())
            te = min(tt[1:])
            if world > 1:
                t = torch.tensor([te], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                te = float(t[0])
            e2e = {"GBps": world * ne * fb / te / 1e9, "ms": 1e3 * te, "h2d_bytes": ne * fb, "d2h_bytes": int(r), "frames_per_gpu": ne,
                   "how": "zl_compress_split on one pinned host buffer per rank, wall clock of the call (max over ranks), best of 2 after a warm-up call"}
            del hsrc, hdst
        if rank != 0:
            continue
        # a sample of frames: round trip through libzstd and libzstd's own size for the same slab at the same level
        from oracle import ref
        ours = theirs = 0
        for i in range(0, n, max(1, n // 128)):
            fam, row, shift = meta[i]
            want = np.roll(pools[fam][row], shift).tobytes()
            frame = dst[i * slot:i * slot + int(sizes[i])].cpu().numpy().tobytes()
            assert ref.decompress(frame) == want, "GPU frame does not round-trip through libzstd"
            ours += len(frame); theirs += len(ref.compress(want, lvl))
        alg = n * fb + csize                                              # SURVEY.md 8d: uncompressed read + compressed written
        peak, peak_src = measured_peak()
        dom = max((k for k in stages if stages[k] > 0), key=lambda k: stages[k], default=None)
        out[f"level{lvl}"] = {"GBps": world * n * fb / ms / 1e6, "ms": ms, "ratio": n * fb / csize, "size_vs_libzstd": ours / theirs,
                              "size_vs_libzstd_how": f"{len(range(0, n, max(1, n // 128)))} sampled frames, libzstd at the same level on the same slabs",
                              "kernel_ms": kernel_ms, "stages_ms": stages, "steps": iters,
                              "stages_how": "CUDA events between the kernels, summed over the waves of the last device-resident call (a call of more than 8,192 blocks runs in waves)",
                              "frames_per_gpu": n, "frame_bytes": fb, "n_gpus": world,
                              "roofline": {"bound": "hbm", "achieved": alg / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": alg / ms / 1e6 / peak,
                                           "peak_source": peak_src, "algorithmic_bytes_per_call": int(alg), "call_ms": ms,
                                           "dominant_kernel": ("zl_k_" + dom) if dom else None,
                                           "dominant_share_of_wave": (stages[dom] / sum(v for v in stages.values() if v > 0)) if dom else None,
                                           "traffic": compress_traffic_bytes(lvl, n)[0], "traffic_source": compress_traffic_bytes(lvl, n)[1]}}
        if e2e:
            out[f"level{lvl}"]["e2e"] = e2e
        if world == 1 and not args.no_cpu:
            nb = min(n, args.cpu_compress_frames)
            host = src.reshape(-1)[:nb * fb].cpu().numpy()
            out[f"level{lvl}"]["cpu_baseline"] = cpu_compress_variants(host, fb, lvl, os.cpu_count() or 1)
    return out


MIX5 = (("text", 0.3), ("rdf", 0.3), ("lowent", 0.15), ("rand", 0.15), ("rle", 0.1))                      # SURVEY.md 8d, config 5


def config5_leg(torch, dist, z, args, dev, rank, world):
    """configs[4]: the 32 GiB mixed corpus (262,144 x 128 KiB frames, families text/rdf/lowent/rand/rle 30/30/15/15/10) sharded by
    frame across the ranks (STRONG scaling: the total is fixed, every rank takes 1/N of the frame list), made on the device from
    the seed; level-3 compress with checksums, then decompress; the round trip is compared on the device.  A rank works through
    its share in sub-shards of <= 65,536 frames (8 GiB), so the footprint does not depend on N; the times are summed."""
    from zstdlite_b200 import corpus
    from oracle import ref
    total_frames, fb = args.config5_frames, 131072
    n = total_frames // world
    bound = int(z._lib.lib().ZSTD_compressBound(fb))
    slot = (bound + 255) // 256 * 256
    cctx, dctx = z.zstd_cctx(level=3, include_checksum=True), z.zstd_dctx()
    stream = torch.cuda.current_stream()
    cctx.set_stream(stream.cuda_stream); dctx.set_stream(stream.cuda_stream)
    sub, chunk = 65536, 32768
    ms_c = 0.0
    DEC_REPS = 5
    dec_reps = [0.0] * DEC_REPS
    csize = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for s0 in range(0, n, sub):
        m = min(sub, n - s0)
        src, pools, meta = corpus.device_mixed_slabs(m, fb, MIX5, index=31 + rank * 64 + s0 // sub, device=dev)
        comp = torch.empty(m * slot + 64, dtype=torch.uint8, device=dev)
        back = torch.empty((m, fb), dtype=torch.uint8, device=dev)
        cplan = z.BatchPlan([src.data_ptr() + i * fb for i in range(m)], [fb] * m, [comp.data_ptr() + i * slot for i in range(m)], [bound] * m)
        if s0 == 0:
            cplan.compress(cctx)                                        # warm-up (arenas, contexts)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
        e0.record(stream); res = cplan.compress(cctx); e1.record(stream); torch.cuda.synchronize()
        ms_c += e0.elapsed_time(e1)
        sizes = [int(r) for r in res]
        assert not any(z.is_error(v) for v in sizes), "compress errors"
        csize += sum(sizes)
        # decoded in calls of <= 32,768 frames: the decoder's arenas (literals, 8-byte records) are sized per call
        dplans = [z.BatchPlan([comp.data_ptr() + i * slot for i in range(a, min(m, a + chunk))], sizes[a:a + chunk],
                              [back.data_ptr() + i * fb for i in range(a, min(m, a + chunk))], [fb] * (min(m, a + chunk) - a)) for a in range(0, m, chunk)]
        if s0 == 0:
            dplans[0].decompress(dctx)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()
        for rep in range(DEC_REPS):                                     # repeated: one slow call used to decide this leg's number
            e0.record(stream)
            bad = 0
            for p in dplans:
                bad += sum(1 for r in p.decompress(dctx) if int(r) != fb)
            e1.record(stream); torch.cuda.synchronize()
            dec_reps[rep] += e0.elapsed_time(e1)
            assert bad == 0, "decode errors"
        assert torch.equal(back, src), "round trip differs"
        if rank == 0:
            for i in range(0, m, max(1, m // 8)):                       # sampled frames through the reference's libzstd
                fam, row, shift = meta[i]
                assert ref.decompress(comp[i * slot:i * slot + sizes[i]].cpu().numpy().tobytes()) == np.roll(pools[fam][row], shift).tobytes()
        del src, comp, back, cplan, dplans
    # the leg's decompress time: for every repeat the max over ranks, then the median of the repeats; per-rank min / median beside it
    reps = torch.tensor(dec_reps, dtype=torch.float64, device=dev)
    t = torch.tensor([ms_c, float(csize)], dtype=torch.float64, device=dev)
    per_rank = [reps.clone() for _ in range(world)]
    if world > 1:
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(t)
        dist.all_gather(per_rank, reps)
        dist.all_reduce(reps, op=dist.ReduceOp.MAX)
        ms_c, csize = float(mx[0]), float(t[1])
    if rank != 0:
        return None
    ms_d = float(reps.median())
    tot = n * world * fb
    return {"frames": n * world, "frame_bytes": fb, "bytes": tot, "n_gpus": world, "scaling": "strong", "level": 3, "checksum": True,
            "compress_GBps": tot / ms_c / 1e6, "compress_ms": ms_c, "decompress_GBps": tot / ms_d / 1e6, "decompress_ms": ms_d,
            "decompress_how": f"median of {DEC_REPS} repeats of (max over ranks); compress: one pass, max over ranks",
            "decompress_ms_repeats_max_over_ranks": [float(v) for v in reps],
            "decompress_ms_per_rank_min_median": [[float(r.min()), float(r.median())] for r in per_rank],
            "ratio": tot / float(csize), "round_trip": "device compare of every byte + sampled frames through libzstd"}


def dict_leg(torch, z, args, dev):
    """configs[3]: 1e5 small objects, dictionary trained ON THE GPU on the first 1e4 (5,000 B; the reference's ZDICT timed beside it), level 3;
    device-resident batch compress then decompress with the dictionary; sizes compared with libzstd + the same dictionary."""
    from oracle import ref
    from zstdlite_b200 import corpus
    import warnings
    n = args.dict_objects
    objs = corpus.small_objects(n)
    train = objs[:min(n, 10000)]
    # training: the GPU trainer (csrc/zl_dict_train.cuh) against the reference's ZDICT_trainFromBuffer on the same samples
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        z.zstd_train_dict_compress(train, 5000)                         # warm-up (contexts and arenas of the trainer are kept for the process)
        t0 = time.time(); d = z.zstd_train_dict_compress(train, 5000); t_gpu = time.time() - t0
    t0 = time.time(); d_ref = ref.train_dict(train, 5000); t_ref = time.time() - t0
    sizes = [len(o) for o in objs]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    total = int(offs[-1])
    src = torch.from_numpy(np.frombuffer(b"".join(objs), dtype=np.uint8).copy()).to(dev)
    L = z._lib.lib()
    caps = [int(L.ZSTD_compressBound(s)) for s in sizes]
    coffs = np.concatenate([[0], np.cumsum([(c + 15) // 16 * 16 for c in caps])]).astype(np.int64)
    cdst = torch.zeros(int(coffs[-1]) + 64, dtype=torch.uint8, device=dev)
    cctx, dctx = z.zstd_cctx(level=3, dict=d), z.zstd_dctx(dict=d)
    stream = torch.cuda.current_stream()
    cctx.set_stream(stream.cuda_stream); dctx.set_stream(stream.cuda_stream)
    cplan = z.BatchPlan([src.data_ptr() + int(o) for o in offs[:-1]], sizes, [cdst.data_ptr() + int(o) for o in coffs[:-1]], caps)
    res = None
    for _ in range(2):
        res = cplan.compress(cctx)
    csz = [int(r) for r in res]
    assert not any(z.is_error(r) for r in csz[:256])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(3):
        cplan.compress(cctx)
    e1.record(stream); torch.cuda.synchronize()
    ms_c = e0.elapsed_time(e1) / 3
    ddst = torch.zeros(total + 64, dtype=torch.uint8, device=dev)
    dplan = z.BatchPlan([cdst.data_ptr() + int(o) for o in coffs[:-1]], csz, [ddst.data_ptr() + int(o) for o in offs[:-1]], sizes)
    for _ in range(2):
        dres = dplan.decompress(dctx)
    assert all(int(r) == s for r, s in zip(dres, sizes)), "dictionary decode errors"
    assert bytes(ddst[:total].cpu().numpy()) == b"".join(objs), "dictionary round trip differs"
    e0.record(stream)
    for _ in range(3):
        dplan.decompress(dctx)
    e1.record(stream); torch.cuda.synchronize()
    ms_d = e0.elapsed_time(e1) / 3
    rc, rd, rc_ref = ref.CCtx(level=3, dict=d), ref.DCtx(dict=d), ref.CCtx(level=3, dict=d_ref)
    step = max(1, n // 5000)
    host = cdst.cpu().numpy()
    ours = theirs = refpipe = 0
    for i in range(0, n, step):                       # bounded sample for the libzstd comparison + cross-decode
        c = host[int(coffs[i]):int(coffs[i]) + csz[i]].tobytes()
        assert rd.decompress(c, cap=sizes[i]) == objs[i], "GPU dictionary frame does not decode with libzstd"
        ours += csz[i]; theirs += len(rc.compress(objs[i])); refpipe += len(rc_ref.compress(objs[i]))
    return {"objects": n, "bytes": total, "dict_bytes": len(d), "level": 3, "steps": 3, "compress_GBps": total / ms_c / 1e6, "compress_ms": ms_c,
            "decompress_GBps": total / ms_d / 1e6, "decompress_ms": ms_d, "ratio": total / sum(csz),
            "size_vs_libzstd_same_dict": ours / theirs, "size_vs_reference_pipeline": ours / refpipe,
            "size_vs_reference_pipeline_how": "GPU-trained dictionary + GPU compressor against ZDICT-trained dictionary + libzstd, level 3",
            "sampled_objects": len(range(0, n, step)),
            "train": {"samples": len(train), "sample_bytes": sum(len(o) for o in train), "gpu_s": t_gpu, "zdict_s": t_ref,
                      "dict_id": z.zstd_dict_id(d), "zdict_dict_id": z.zstd_dict_id(d_ref)}}


def large_frame_leg(torch, z, args, dev):
    """configs[0]: zstd_serialize / zstd_unserialize of a 1e6-row data.frame (R's binary serialization restated, ~16 MB), level 3.
    The reference compresses it into ONE frame (2 MB window, ~128 dependent blocks, num_threads = 1); the GPU decodes that
    frame with the block-parallel large-frame path and compresses the payload as one frame of independent blocks."""
    from oracle import ref
    from zstdlite_b200 import corpus
    payload = corpus.r_data_frame(args.df_rows)
    n = len(payload)
    t0 = time.time(); frame = ref.compress(payload, 3); t_cc = time.time() - t0
    t0 = time.time(); back = ref.decompress(frame); t_cd = time.time() - t0
    assert back == payload
    from oracle import cpubench
    threads = os.cpu_count() or 1
    t_w, size_w = cpubench.run_workers(np.frombuffer(payload, dtype=np.uint8), level=3, workers=threads, passes=3)
    src = torch.from_numpy(np.frombuffer(frame, dtype=np.uint8).copy()).to(dev)
    dst = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
    dctx = z.zstd_dctx()
    stream = torch.cuda.current_stream(); dctx.set_stream(stream.cuda_stream)
    plan = z.BatchPlan([src.data_ptr()], [len(frame)], [dst.data_ptr()], [n])
    for _ in range(2):
        res = plan.decompress(dctx)
    assert int(res[0]) == n and bytes(dst[:n].cpu().numpy()) == payload, "large-frame decode differs from libzstd"
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(5):
        plan.decompress(dctx)
    e1.record(stream); torch.cuda.synchronize()
    ms_d = e0.elapsed_time(e1) / 5
    # compress: the payload resident in HBM -> one frame
    raw = torch.from_numpy(np.frombuffer(payload, dtype=np.uint8).copy()).to(dev)
    cap = int(z._lib.lib().ZSTD_compressBound(n))
    cdst = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    cctx = z.zstd_cctx(level=3); cctx.set_stream(stream.cuda_stream)
    cplan = z.BatchPlan([raw.data_ptr()], [n], [cdst.data_ptr()], [cap])
    for _ in range(2):
        cres = cplan.compress(cctx)
    csz = int(cres[0])
    ours = bytes(cdst[:csz].cpu().numpy())
    assert ref.decompress(ours) == payload, "GPU frame does not decode with libzstd"
    e0.record(stream)
    for _ in range(5):
        cplan.compress(cctx)
    e1.record(stream); torch.cuda.synchronize()
    ms_c = e0.elapsed_time(e1) / 5
    return {"rows": args.df_rows, "bytes": n, "frame_bytes_libzstd": len(frame), "frame_bytes_ours": csz, "size_vs_libzstd": csz / len(frame),
            "decompress_GBps": n / ms_d / 1e6, "decompress_ms": ms_d, "compress_GBps": n / ms_c / 1e6, "compress_ms": ms_c, "steps": 5,
            "libzstd_1thread_decompress_GBps": n / t_cd / 1e9, "libzstd_1thread_compress_GBps": n / t_cc / 1e9,
            "libzstd_nbWorkers_compress_GBps": n / t_w / 1e9, "libzstd_nbWorkers": threads, "libzstd_nbWorkers_frame_bytes": size_w,
            "cpu_baseline_how": "the reference's path for this config: one frame, level 3; num_threads = 1 (ZSTD_compress2 / ZSTD_decompressDCtx) and "
                                "num_threads = cores (ZSTD_c_nbWorkers, src/cctx.c:269-277; compression only -- libzstd decompresses single-threaded)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=16384)
    ap.add_argument("--frame-bytes", type=int, default=65536)
    ap.add_argument("--cpu-frames", type=int, default=16384, help="frames handed to the CPU baseline (default: all of them)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--cpu-compress-frames", type=int, default=4096, help="128 KiB slabs of the compress leg handed to the CPU baselines (512 MiB)")
    ap.add_argument("--no-affinity", action="store_true", help="do not bind the process to the CPUs local to its GPU")
    ap.add_argument("--compress-frames", type=int, default=32768)
    ap.add_argument("--no-compress", action="store_true")
    ap.add_argument("--no-compress-e2e", action="store_true")
    ap.add_argument("--dict-objects", type=int, default=100000)
    ap.add_argument("--no-dict", action="store_true")
    ap.add_argument("--df-rows", type=int, default=1000000)
    ap.add_argument("--no-large", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--config5-frames", type=int, default=262144, help="frames of configs[4] in total (32 GiB), split over the ranks")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output under DIR as .npy files (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    # stdout carries exactly ONE JSON line: anything libraries print to fd 1 meanwhile (NCCL's version banner) goes to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; zstdlite_b200 has no CPU path (use --impl reference for the CPU arm)")
    affinity = {"bound": False, "off": True} if args.no_affinity else pin_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import zstdlite_b200 as z

    t_prep = time.time()
    data, frames = make_corpus(args.frames, args.frame_bytes, seed_shift=rank * 17)
    n, fb = args.frames, args.frame_bytes
    sizes = [len(f) for f in frames]
    csize = sum(sizes)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    blob = np.frombuffer(b"".join(frames), dtype=np.uint8)
    log(f"[rank {rank}] corpus {n} x {fb}: ratio {n * fb / csize:.3f}, prep {time.time() - t_prep:.1f}s")

    # ---- device-resident arm
    src = torch.zeros(csize + 64, dtype=torch.uint8, device=dev)
    src[:csize].copy_(torch.from_numpy(blob.copy()))
    dst = torch.zeros(n * fb + 64, dtype=torch.uint8, device=dev)
    dctx = z.zstd_dctx()
    stream = torch.cuda.current_stream()
    dctx.set_stream(stream.cuda_stream)
    plan = z.BatchPlan([src.data_ptr() + int(o) for o in offs[:-1]], sizes, [dst.data_ptr() + i * fb for i in range(n)], [fb] * n)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        res = plan.decompress(dctx)
    assert all(int(r) == fb for r in res), "decode errors in warm-up"
    got = dst[:n * fb].cpu().numpy().reshape(n, fb)
    assert (got == data).all(), "GPU output differs from the original bytes"
    del got
    sampler = ClockSampler(local)
    stage_names = ("literals", "sequences", "execute", "checksum")
    launches0 = dctx.launch_count
    sync_all()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        res = plan.decompress(dctx)
    e1.record(stream)
    sync_all()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    launches = dctx.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, dst, res, n, fb)
    # per-kernel durations: the same batch as ONE slice on ONE stream with CUDA events between the kernels (the timed
    # region above runs the slice pipeline, where kernels of different slices overlap and have no duration of their own)
    dctx.set_profile(True)
    stage_ms = np.zeros(4)
    plan.decompress(dctx)
    for _ in range(args.steps):
        plan.decompress(dctx)
        stage_ms += [z._lib.lib().zl_dctx_last_stage_ms(dctx._p, k) for k in range(4)]
    stage_ms /= args.steps
    serial_ms = float(stage_ms.sum())
    dctx.set_profile(False)

    # ---- end-to-end arm: pinned host buffers in, pinned host buffer out, through the same C-ABI call
    hsrc = torch.from_numpy(blob.copy()).pin_memory()
    hdst = torch.zeros(n * fb, dtype=torch.uint8).pin_memory()
    hplan = z.BatchPlan([hsrc.data_ptr() + int(o) for o in offs[:-1]], sizes, [hdst.data_ptr() + i * fb for i in range(n)], [fb] * n)
    for _ in range(max(3, args.warmup)):
        hplan.decompress(dctx, device=False)
    assert (hdst.numpy().reshape(n, fb) == data).all()
    sync_all()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    e2e_steps = args.steps                  # the same K steps as the device-resident arm (five used to scatter by +-3 % between runs)
    for _ in range(e2e_steps):
        hplan.decompress(dctx, device=False)
    e3.record(stream)
    sync_all()
    ms_e2e = e2.elapsed_time(e3)
    # the same call with PAGEABLE host buffers (what the reference's C layer hands over: R-allocated vectors, src/raw-file.c:166,189)
    psrc = blob.copy()
    pdst = np.zeros(n * fb, dtype=np.uint8)
    pplan = z.BatchPlan([psrc.ctypes.data + int(o) for o in offs[:-1]], sizes, [pdst.ctypes.data + i * fb for i in range(n)], [fb] * n)
    for _ in range(3):
        pplan.decompress(dctx, device=False)
    assert (pdst.reshape(n, fb) == data).all()
    sync_all()
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e4.record(stream)
    for _ in range(3):
        pplan.decompress(dctx, device=False)
    e5.record(stream)
    sync_all()
    ms_page = e4.elapsed_time(e5) / 3
    del psrc, pdst, pplan
    # raw ceiling of that arm on this box: the step's two copies alone, every rank at once
    ms_pcie = pcie_probe(torch, dist, dev, world, int(csize), int(n * fb))

    if world > 1:
        t = torch.tensor([ms_total, ms_e2e, ms_page], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e, ms_page = float(t[0]), float(t[1]), float(t[2])
    total_bytes = world * n * fb
    value = total_bytes * args.steps / ms_total / 1e6
    e2e_value = total_bytes * e2e_steps / ms_e2e / 1e6

    # ---- compress leg (configs[2]); every rank takes part, so it runs before rank 0 goes on alone
    comp = None
    if not args.no_compress:
        del hsrc, hdst, hplan
        try:
            comp = compress_leg(torch, dist, z, args, dev, rank, world)
        except Exception as e:                                          # the headline is the decode arm; report, don't hide
            if world > 1:
                raise
            comp = {"error": repr(e)}

    c5 = None
    if not args.no_config5:
        if comp is not None:
            torch.cuda.empty_cache()
        try:
            c5 = config5_leg(torch, dist, z, args, dev, rank, world)
        except Exception as e:
            if world > 1:
                raise
            c5 = {"error": repr(e)}
        torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = measured_peak()
        k = int(np.argmax(stage_ms))
        alg_bytes = csize + n * fb                                     # SURVEY.md 8d: compressed read + uncompressed written
        achieved = alg_bytes / stage_ms[k] / 1e6
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "u8", "data": "synthetic", "config": workload_config(args, world),
               "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(csize + n * 80), "d2h_bytes_per_step": int(n * fb + n * 8),
                       "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps, "host_buffers": "pinned",
                       "pcie_ceiling_GBps": total_bytes / ms_pcie / 1e6, "frac_of_pcie_ceiling": (total_bytes * e2e_steps / ms_e2e) / (total_bytes / ms_pcie),
                       "pcie_ceiling_how": "this step's H2D and D2H byte counts as two plain concurrent cudaMemcpyAsync (pinned <-> HBM) on every rank at once, "
                                           "slower direction, max over ranks, best of 3",
                       "pageable": {"value": total_bytes / ms_page / 1e6, "unit": UNIT, "ms_per_step": ms_page, "steps": 3,
                                    "how": "the same call with malloc'ed (pageable) host buffers, as the reference's C layer passes them"},
                       "cpu_affinity": affinity},
               "gpu_launches": int(launches), "clocks": clocks,
               "roofline": {"bound": "hbm", "kernel": "zl_k_" + stage_names[k], "achieved": achieved, "peak": peak, "unit": "GB/s",
                            "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                            "algorithmic_bytes_per_launch": int(alg_bytes), "kernel_ms": float(stage_ms[k]),
                            "kernel_ms_how": "whole batch as one launch per kernel on one stream, CUDA events between kernels, mean of %d passes; "
                                             "the timed region runs the slice pipeline (8 slices on 8 streams)" % args.steps,
                            "serial_pipeline_ms": serial_ms,
                            "whole_pipeline_frac": (alg_bytes / (ms_total / args.steps) / 1e6) / peak},
               "stages_ms": {nm: float(v) for nm, v in zip(stage_names, stage_ms)},
               "steps_note": "--steps sets the device-resident and pinned end-to-end arms; the pageable arm and the compress, config5, "
                             "dict and large_frame legs time fixed repetitions, given in each as steps or in its how",
               "compression_ratio_of_input": n * fb / csize}
        traffic_path = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
        if os.path.exists(traffic_path):
            try:
                tr = json.load(open(traffic_path))
                if tr.get("kernel") == out["roofline"]["kernel"]:
                    out["roofline"]["traffic"] = tr.get("dram_bytes_per_launch_at_bench_size")
                    out["roofline"]["traffic_source"] = tr.get("source")
            except (ValueError, OSError):
                pass
        if world == 1 and not args.no_cpu:
            from oracle import ref
            threads = os.cpu_count() or 1
            nsample = min(n, args.cpu_frames)
            step = max(1, n // nsample)
            sample = frames[::step][:nsample]
            v, t_pass, passes = cpu_leg(sample, fb, args.cpu_seconds, threads)
            v1, _, _ = cpu_leg(sample[:max(1, len(sample) // threads)], fb, 2.0, 1)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "reference",
                                   "sample": f"{len(sample)} of the {n} frames" + (f" (every {step}th, same family mix)" if step > 1 else "") +
                                             f", frame-parallel, best of {passes} passes, system libzstd {ref.version()}, one DCtx per thread",
                                   "one_thread_GBps": v1,
                                   "note": "libzstd has no multi-threaded decompression: num_threads = cores changes nothing on this side (BASELINE.md section 3)"}
        if comp is not None:
            out["compress"] = comp
        if c5 is not None:
            out["config5"] = c5
        if world == 1 and not args.no_dict:
            try:
                out["dict"] = dict_leg(torch, z, args, dev)
            except Exception as e:
                out["dict"] = {"error": repr(e)}
        if world == 1 and not args.no_large:
            try:
                out["large_frame"] = large_frame_leg(torch, z, args, dev)
            except Exception as e:
                out["large_frame"] = {"error": repr(e)}
        print(json.dumps(out), file=real_stdout, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
