#!/usr/bin/env python
"""bench.py — compression throughput of the zstd hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--config C]            # our CUDA path
  python bench.py --impl reference --steps K --warmup W [--config C]    # reference libzstd on the host cores
  python bench.py ... --dump-outputs DIR                                # also write the last timed step's frames to DIR

--config selects one of BASELINE.json's workloads (default 2, the one the metric is quoted on):
  2  datagen -g1GB -P50, level 1, one frame per GPU (weak scaling: every rank owns one 1 GiB shard, seed = rank)
  3  8 GiB of datagen -P30 as 128 independent 64 MiB frames (seed = frame index), --fast=3, the frame list
     partitioned over the ranks (strong scaling: the job is the same 8 GiB at every N)
  4  datagen -g2GB -P90, level 3 (doubleFast), one frame per GPU (weak scaling)
  5  1 048 576 x 1 KiB records (datagen -g1GB -P50 cut up) + one 16 KiB ZDICT dictionary, level 1, records partitioned
     over the ranks (strong scaling)
With N > 1 the ranks' compressed buffers are gathered to rank 0 over NCCL inside the timed region
(zstd_b200/sharding.py: point-to-point, straight to their final offsets; the gather of step k runs while step k+1
compresses, the last one is waited for before the clock stops).
"""
import argparse
import ctypes
import hashlib
import json
import os

# the host path keeps ~10 streams busy (8 wave streams + upload + download): give every one its own hardware
# queue, else a download can sit behind another wave's kernels (profiles/r1_e2e_timeline.md).  Must be set
# before the CUDA context exists; INTEGRATION.md tells embedders to do the same.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "compress GB/s (input) at level 1"
GiB = 1 << 30
MiB = 1 << 20
_sz = ctypes.c_size_t


# ----------------------------------------------------------------------------------------------- workloads
class Workload:
    """What one rank compresses: `src` bytes, the frames inside it, level, optional dictionary."""

    def __init__(self, config, rank, world, scale=1.0):
        import zref
        self.config, self.rank, self.world = config, rank, world
        self.dict = None
        gen = "reference tests/datagen" if zref.have_datagen() else "zbo_synthetic (datagen binary absent)"

        def data(size, p, seed):
            return zref.datagen(size, p, seed) if zref.have_datagen() else zref.synthetic(size, seed, p / 100.0)

        if config == 2:
            size = int(GiB * scale)
            self.level, self.scaling = 1, "weak"
            self.src = data(size, 50, rank)
            self.frames = [(0, size)]
            self.total_input = size * world
            self.desc = f"datagen -g{size} -P50 -s<rank> per GPU, level 1, one frame per GPU, 128 KiB blocks"
        elif config == 4:
            size = int(2 * GiB * scale)
            self.level, self.scaling = 3, "weak"
            self.src = data(size, 90, rank)
            self.frames = [(0, size)]
            self.total_input = size * world
            self.desc = f"datagen -g{size} -P90 -s<rank> per GPU, level 3 (doubleFast), one frame per GPU"
        elif config == 3:
            from zstd_b200.sharding import partition_frames
            fs, nf = 64 * MiB, max(world, int(128 * scale))
            self.level, self.scaling = -3, "strong"
            b, e = partition_frames([fs] * nf, world)[rank]
            self.src = b"".join(data(fs, 30, f) for f in range(b, e))
            self.frames = [(i * fs, fs) for i in range(e - b)]
            self.total_input = fs * nf
            self.desc = f"{nf} independent frames of datagen -g{fs} -P30 -s<frame> ({fs * nf} bytes in all), --fast=3 (level -3), frames partitioned over the GPUs"
        elif config == 5:
            from zstd_b200.sharding import partition_frames
            rec, nrec = 1024, max(world, int((1 << 20) * scale))
            self.level, self.scaling = 1, "strong"
            allrec = data(rec * nrec, 50, 0)
            self.dict = zref.train_dict(allrec, rec, min(20000, nrec), 16 << 10) if zref.have_ref() else allrec[-(16 << 10):]
            b, e = partition_frames([rec] * nrec, world)[rank]
            self.src = allrec[b * rec:e * rec]
            self.frames = [(i * rec, rec) for i in range(e - b)]
            self.total_input = rec * nrec
            self.desc = (f"{nrec} records of {rec} B (datagen -g{rec * nrec} -P50 cut up) + one {len(self.dict)} B "
                         f"{'ZDICT_trainFromBuffer' if zref.have_ref() else 'raw-content'} dictionary, level 1, records partitioned over the GPUs")
        else:
            raise SystemExit(f"bench.py: unknown --config {config}")
        self.data = f"synthetic: {gen}"
        self.size = len(self.src)
        n = len(self.frames)
        self.offs = (_sz * n)(*[o for o, _ in self.frames])
        self.sizes = (_sz * n)(*[s for _, s in self.frames])
        self.nframes = n


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json (burst copy figure: kernels are timed alone)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.samples, self.index, self.proc, self.windows = [], index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def mark(self):
        """Start (or restart) a timed window: only samples taken inside windows are reported."""
        self.windows.append([time.perf_counter(), None])

    def unmark(self):
        self.windows[-1][1] = time.perf_counter()

    def stop(self):
        if self.proc:
            self.proc.terminate()
        inside = [s for t, s in self.samples if any(a <= t <= (b or 1e30) for a, b in self.windows)]
        sm = sorted(int(s[0]) for s in inside if s and s[0].isdigit())
        mx = max([int(s[1]) for s in inside if len(s) > 1 and s[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in inside for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons, "samples": len(sm),
                "sampled": "nvidia-smi -lms 20 during the timed device-resident and end-to-end loops"}


# ----------------------------------------------------------------------------------------------- reference on the host cores
def host_description():
    model, phys = "unknown CPU", None
    try:
        cores = set()
        with open("/proc/cpuinfo") as f:
            pid = cid = None
            for line in f:
                if line.startswith("model name") and model == "unknown CPU":
                    model = line.split(":", 1)[1].strip()
                elif line.startswith("physical id"):
                    pid = line.split(":", 1)[1].strip()
                elif line.startswith("core id"):
                    cid = line.split(":", 1)[1].strip()
                elif not line.strip():
                    if pid is not None and cid is not None:
                        cores.add((pid, cid))
                    pid = cid = None
        phys = len(cores) or None
    except Exception:
        pass
    return f"{model}, {phys if phys else '?'} physical cores, {os.cpu_count()} hardware threads"


def ref_lib():
    import zref
    R = zref.ref()
    vp, ci = ctypes.c_void_p, ctypes.c_int
    R.ZSTD_createCCtx.restype = vp
    R.ZSTD_freeCCtx.argtypes = [vp]
    R.ZSTD_CCtx_setParameter.restype = _sz
    R.ZSTD_CCtx_setParameter.argtypes = [vp, ci, ci]
    R.ZSTD_compress2.restype = _sz
    R.ZSTD_compress2.argtypes = [vp, vp, _sz, vp, _sz]
    R.ZSTD_compressCCtx.restype = _sz
    R.ZSTD_compressCCtx.argtypes = [vp, vp, _sz, vp, _sz, ci]
    R.ZSTD_createCDict.restype = vp
    R.ZSTD_createCDict.argtypes = [ctypes.c_char_p, _sz, ci]
    R.ZSTD_freeCDict.argtypes = [vp]
    R.refdrv_frames.restype = _sz
    R.refdrv_frames.argtypes = [vp, vp, vp, vp, _sz, _sz, vp, _sz, ci]
    R.refdrv_records_cdict.restype = _sz
    R.refdrv_records_cdict.argtypes = [vp, vp, vp, _sz, _sz, _sz, vp, _sz]
    return R


class Pool:
    """Persistent worker threads: created once, released together for every timed pass (the ctypes calls drop the GIL)."""

    def __init__(self, n):
        self.n, self.fn, self.stop = n, None, False
        self.go, self.done = threading.Barrier(n + 1), threading.Barrier(n + 1)
        self.threads = [threading.Thread(target=self._loop, args=(i,), daemon=True) for i in range(n)]
        for t in self.threads:
            t.start()

    def _loop(self, i):
        while True:
            self.go.wait()
            if self.stop:
                return
            self.fn(i)
            self.done.wait()

    def run(self, fn):
        self.fn = fn
        t0 = time.perf_counter()
        self.go.wait()
        self.done.wait()
        return time.perf_counter() - t0

    def close(self):
        self.stop = True
        self.go.wait()


class RefRunner:
    """The reference's own CPU implementation of a workload with `threads` host threads; contexts, destination buffers
    and threads live across passes.  run() -> (seconds, compressed bytes) of one pass over the whole workload (or over
    its first `frames` frames)."""

    def __init__(self, wl, threads, frames=None):
        R = self.R = ref_lib()
        self.wl, self.threads = wl, threads
        n = wl.nframes if frames is None else min(frames, wl.nframes)
        self.hbuf = (ctypes.c_char * max(wl.size, 1)).from_buffer_copy(wl.src)
        self.addr = ctypes.addressof(self.hbuf)
        self.pool = Pool(threads)
        self.modes = {}
        self.bytes = sum(wl.sizes[i] for i in range(n))
        if wl.dict is not None:                                   # config 5: a digested dictionary, records spread over the threads
            self.cdict = R.ZSTD_createCDict(wl.dict, len(wl.dict), wl.level)
            per = (n + threads - 1) // threads
            self.parts = [(i * per, max(0, min(per, n - i * per))) for i in range(threads)]
            self.ctxs = [R.ZSTD_createCCtx() for _ in range(threads)]
            self.caps = [R.ZSTD_compressBound(wl.sizes[0]) * max(c, 1) for _, c in self.parts]
            self.dsts = [ctypes.create_string_buffer(max(c, 1)) for c in self.caps]
            self.out = [0] * threads
            rec = wl.sizes[0]

            def work(i):
                f, c = self.parts[i]
                if c:
                    self.out[i] = R.refdrv_records_cdict(self.ctxs[i], self.cdict, self.addr, rec, f, c, self.dsts[i], self.caps[i])
            self.modes[f"ZSTD_compress_usingCDict per record, {threads} threads"] = work
        elif n >= threads // 2:                                   # many frames: whole frames spread over the threads
            per = (n + threads - 1) // threads
            self.parts = [(i * per, max(0, min(per, n - i * per))) for i in range(threads)]
            self.ctxs = [R.ZSTD_createCCtx() for _ in range(threads)]
            self.caps = [sum(R.ZSTD_compressBound(wl.sizes[j]) for j in range(f, f + c)) for f, c in self.parts]
            self.dsts = [ctypes.create_string_buffer(max(c, 1)) for c in self.caps]
            self.out = [0] * threads

            def work(i):
                f, c = self.parts[i]
                if c:
                    self.out[i] = R.refdrv_frames(self.ctxs[i], self.addr, wl.offs, wl.sizes, f, c, self.dsts[i], self.caps[i], wl.level)
            self.modes[f"ZSTD_compressCCtx per frame, frames spread over {threads} threads"] = work
        else:
            # one (or a few) big frames: the two stock ways to use every host thread — ZSTDMT (nbWorkers) keeps the frame,
            # `threads` independent slices are the decomposition SURVEY.md 8d names
            size = wl.sizes[0]
            self.mt = R.ZSTD_createCCtx()
            R.ZSTD_CCtx_setParameter(self.mt, 100, wl.level)
            if threads > 1:
                R.ZSTD_CCtx_setParameter(self.mt, 400, threads)
            self.mtcap = R.ZSTD_compressBound(size)
            self.mtdst = ctypes.create_string_buffer(self.mtcap)
            self.mtout = [0]

            def work_mt(i):
                if i == 0:
                    self.mtout[0] = R.ZSTD_compress2(self.mt, self.mtdst, self.mtcap, self.addr, size)
            self.modes[f"ZSTD_compress2 nbWorkers={threads} (one frame)"] = work_mt
            per = (size + threads - 1) // threads
            self.ctxs = [R.ZSTD_createCCtx() for _ in range(threads)]
            self.caps = [R.ZSTD_compressBound(max(0, min(per, size - i * per))) for i in range(threads)]
            self.dsts = [ctypes.create_string_buffer(max(c, 1)) for c in self.caps]
            self.out = [0] * threads

            def work_sl(i):
                lo = i * per
                if lo < size:
                    self.out[i] = R.ZSTD_compressCCtx(self.ctxs[i], self.dsts[i], self.caps[i], self.addr + lo, min(per, size - lo), wl.level)
            self.modes[f"{threads} independent slices, one ZSTD_compressCCtx thread each"] = work_sl

    def run(self, mode):
        dt = self.pool.run(self.modes[mode])
        csize = self.mtout[0] if mode.startswith("ZSTD_compress2") else sum(self.out)
        return dt, csize

    def close(self):
        self.pool.close()


def time_reference(wl, threads, steps, warmup, frames=None):
    """best stock mode: (GB/s, seconds per pass, mode, compressed bytes, {mode: GB/s})"""
    r = RefRunner(wl, threads, frames)
    res = {}
    for mode in r.modes:
        for _ in range(max(2, warmup)):                           # first passes pay first-touch page faults of the buffers
            r.run(mode)
        tot, cs = 0.0, 0
        for _ in range(steps):
            dt, cs = r.run(mode)
            tot += dt
        res[mode] = (r.bytes * steps / tot / 1e9, tot / steps, cs)
    r.close()
    best = max(res, key=lambda m: res[m][0])
    return res[best][0], res[best][1], best, res[best][2], {m: round(v[0], 3) for m, v in res.items()}, r.bytes


def run_reference(args):
    """--impl reference: the reference's own CPU implementation with all host threads (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import zref
    if not zref.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libzstd_ref.so missing (reference not built on this box)"}))
        return
    cores = os.cpu_count() or 1
    wl = Workload(args.config, 0, 1, args.scale)             # the whole job of the N-GPU run at strong scaling; one shard at weak scaling
    v, per_pass, mode, csize, allmodes, nbytes = time_reference(wl, cores, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(per_pass * 1e3, 3), "higher_is_better": True, "scaling": wl.scaling,
            "vs_baseline": None, "dtype": "u8", "data": wl.data,
            "config": {"workload": wl.desc, "baseline_config": args.config, "host": host_description(), "threads": cores,
                       "modes_gbs": allmodes, "used": mode, "compressed_bytes": csize,
                       "note": "persistent worker threads, contexts and buffers; one pass = the workload of ONE rank at weak scaling, the whole job at strong scaling"},
            "cpu_baseline": {"value": round(v, 4), "unit": "GB/s", "cores": cores, "kind": "reference",
                             "sample": f"{nbytes} bytes per step on {host_description()}; {mode}"},
            "e2e": {"value": round(v, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- our arm
DUMP_SAMPLES = 4 << 20          # compressed bytes kept by --dump-outputs: 16 MiB as float32 + 32 MiB of float64 positions


def dump_outputs(dirname, frames: bytes, frame_sizes):
    """What the timed path returned in its last step, as .npy files that two builds can be compared by: the compressed
    size of every frame, and the compressed bytes (all of them, or a fixed seeded sample of DUMP_SAMPLES positions
    with those positions alongside)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    b = np.frombuffer(frames, dtype=np.uint8)
    if b.size > DUMP_SAMPLES:
        pos = np.sort(np.random.default_rng(0).integers(0, b.size, DUMP_SAMPLES))
        np.save(os.path.join(dirname, "compressed_sample_positions.npy"), pos.astype(np.float64))
        b = b[pos]
    np.save(os.path.join(dirname, "compressed_bytes.npy"), b.astype(np.float32))
    np.save(os.path.join(dirname, "frame_sizes.npy"), np.asarray(frame_sizes, dtype=np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import zstd_b200
    import zref
    from zstd_b200.sharding import gather_compressed, wait_all

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (zstd_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl = Workload(args.config, rank, world, args.scale)
    size = wl.size
    L = zstd_b200.lib()
    ctx = zstd_b200.ZSTD_CCtx(device=local)
    cdict = zstd_b200.ZSTD_CDict(wl.dict, wl.level) if wl.dict is not None else None
    cap = sum(zstd_b200.ZSTD_compressBound(wl.sizes[i]) for i in range(wl.nframes)) + 64
    d_src = torch.frombuffer(bytearray(wl.src), dtype=torch.uint8).cuda()
    # two destination buffers: the gather of step k reads one while step k+1 writes the other.  On rank 0 each is big
    # enough for every rank's bytes: its own frames are compressed straight to the front of the gathered buffer.
    caps = [cap]
    if world > 1:
        t = torch.tensor([cap], dtype=torch.int64, device="cuda")
        allc = torch.empty(world, dtype=torch.int64, device="cuda")
        dist.all_gather_into_tensor(allc, t)
        caps = [int(x) for x in allc.tolist()]
    d_dst = [torch.empty(sum(caps) if rank == 0 else cap, dtype=torch.uint8, device="cuda") for _ in range(2 if world > 1 else 1)]
    csz = (_sz * wl.nframes)()

    def compress(dst_ptr, dst_cap, src_ptr, device_memory):
        if cdict is not None:
            r = L.ZSTDB200_compressFrames_usingCDict(ctx._h, dst_ptr, dst_cap, src_ptr, wl.offs, wl.sizes, wl.nframes, cdict._h, csz, device_memory, None)
        elif wl.nframes == 1 and not device_memory:
            r = L.ZSTD_compressCCtx(ctx._h, dst_ptr, dst_cap, src_ptr, size, wl.level)       # the reference-facing entry point
        else:
            r = L.ZSTDB200_compressFrames(ctx._h, dst_ptr, dst_cap, src_ptr, wl.offs, wl.sizes, wl.nframes, None, 0, csz, wl.level, device_memory, None)
        assert not L.ZSTD_isError(r), L.ZSTD_getErrorName(r)
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pending = [[], []]
    last = {"sizes": None, "gathered": None}

    def step_device(k):
        b = k & 1 if world > 1 else 0
        wait_all(pending[b]); pending[b] = []                    # this buffer's previous gather must be over
        n = compress(d_dst[b].data_ptr(), cap, d_src.data_ptr(), 1)
        if world > 1:
            sizes, gathered, works = gather_compressed(d_dst[b][:n], dst=0, out=d_dst[b] if rank == 0 else None, async_op=True)
            pending[b] = works
            last["sizes"], last["gathered"] = sizes, gathered
        return n

    def drain():
        for b in range(2):
            wait_all(pending[b]); pending[b] = []

    # ---- device-resident throughput (`value`) ----
    csize = 0
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                     # nvidia-smi needs a moment to start: launch it before the warm-up
    for k in range(args.warmup):
        csize = step_device(k)
    drain()
    barrier()
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stats = []
    t0 = time.perf_counter()
    ev0.record()
    for k in range(args.steps):
        csize = step_device(k)
        stats.append(ctx.stats())
    drain()                                                 # the last gathers end inside the timed region
    ev1.record()
    barrier()
    wall = time.perf_counter() - t0
    sampler.unmark()
    ms = ev0.elapsed_time(ev1)
    launches = sum(s.launches for s in stats)
    frame_sizes = list(csz)
    # what rank 0 holds after the last gather must be every rank's frames, in rank order: checked below, outside the clock
    gathered_bytes = bytes(last["gathered"].cpu().numpy()) if (world > 1 and rank == 0) else None
    gathered_sizes = last["sizes"]
    got_dev = bytes(d_dst[(args.steps - 1) & 1 if world > 1 else 0][:csize].cpu().numpy())

    # per-kernel CUDA-event times come from a serial-mode context (one wave, one stream): in the default
    # mode waves on several streams overlap and a kernel's start->end no longer measures that kernel alone
    kern = None
    if rank == 0:
        os.environ["ZSTDB200_SERIAL"] = "1"
        sctx = zstd_b200.ZSTD_CCtx(device=local)
        del os.environ["ZSTDB200_SERIAL"]
        sstats = []
        for i in range(2 + 3):
            if cdict is not None:
                r = L.ZSTDB200_compressFrames_usingCDict(sctx._h, d_dst[0].data_ptr(), cap, d_src.data_ptr(), wl.offs, wl.sizes, wl.nframes, cdict._h, csz, 1, None)
            else:
                r = L.ZSTDB200_compressFrames(sctx._h, d_dst[0].data_ptr(), cap, d_src.data_ptr(), wl.offs, wl.sizes, wl.nframes, None, 0, csz, wl.level, 1, None)
            assert not L.ZSTD_isError(r)
            if i >= 2:
                sstats.append(sctx.stats())
        kern = {k: sum(getattr(s, k) for s in sstats) / len(sstats) for k in ("kernel_ms", "cand_ms", "parse_ms", "literals_ms", "sequences_ms", "stitch_ms")}
        sctx.close()
    torch.cuda.synchronize()

    # ---- end to end through the C ABI with pinned HOST buffers (a context of its own, as an application that only
    # ever passes host pointers would have); config 2 / 4: ZSTD_compressCCtx, the reference's own entry point ----
    ctx.close()
    ctx = zstd_b200.ZSTD_CCtx(device=local)
    h_src = torch.frombuffer(bytearray(wl.src), dtype=torch.uint8).pin_memory()
    h_dst = torch.empty(cap, dtype=torch.uint8).pin_memory()
    ce = 0
    for _ in range(max(3, args.warmup)):
        ce = compress(h_dst.data_ptr(), cap, h_src.data_ptr(), 0)
    barrier()
    sampler.mark()
    te0 = time.perf_counter()
    for _ in range(args.steps):
        ce = compress(h_dst.data_ptr(), cap, h_src.data_ptr(), 0)
    barrier()
    e2e_s = time.perf_counter() - te0
    sampler.unmark()
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([ms, e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_s = float(t[0]), float(t[1])
    tot = torch.tensor([ce, size], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(tot)
    d2h_total, h2d_total = int(tot[0]), int(tot[1])

    # ---- GPU decompression of what was produced (outside the timed region, in a process of its own so that nothing it
    # does can hold up the compression line): rank 0's input is compressed again there, goes back through
    # ZSTDB200_decompressDevice and must equal the input, compared on the device ----
    decode = None
    if rank == 0 and wl.dict is None and args.config in (2, 4) and not args.no_decode:
        try:
            p50 = 50 if args.config == 2 else 90
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_decode.py"), "--json", str(size), str(p50), str(wl.level), str(local)],
                               capture_output=True, text=True, timeout=240)
            decode = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 and r.stdout.strip() else {"error": (r.stderr or "no output")[-300:]}
            if "compressed_bytes" in decode:
                decode["same_frame_as_timed"] = decode["compressed_bytes"] == csize
        except Exception as ex:                                  # reported, never fatal for the compression line
            decode = {"error": str(ex)[:300]}

    # ---- parity of what was timed (outside the timed region) ----
    assert bytes(h_dst[:ce].numpy()) == got_dev, "host-path and device-path frames differ"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, got_dev, frame_sizes)
    digest = hashlib.sha256(wl.src).hexdigest()
    digests = [digest]
    if world > 1:
        digests = [None] * world if rank == 0 else None
        dist.gather_object(digest, digests, dst=0)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ok_rt = None
    if zref.have_ref():
        if wl.dict is None:
            ok_rt = zref.ref_decompress(got_dev, size) == wl.src
        else:
            ok_rt = True
            # a sample of records through the reference's dictionary decoder
            offs_c, acc = [], 0
            for c in frame_sizes:
                offs_c.append(acc); acc += c
            for i in range(0, wl.nframes, max(1, wl.nframes // 512)):
                o, n = wl.frames[i]
                ok_rt &= zref.ref_decompress_using_dict(got_dev[offs_c[i]:offs_c[i] + frame_sizes[i]], wl.dict, n) == wl.src[o:o + n]
    gather_ok = None
    if world > 1 and zref.have_ref():
        # rank 0 decodes the gathered concatenation: every rank's part must reproduce that rank's input (by SHA-256)
        gather_ok, pos = sum(gathered_sizes) == len(gathered_bytes), 0
        for r in range(world):
            part = gathered_bytes[pos:pos + gathered_sizes[r]]
            pos += gathered_sizes[r]
            if wl.dict is None:
                dec = zref.ref_decompress(part, wl.total_input)      # upper bound on a rank's share
                gather_ok &= hashlib.sha256(dec).hexdigest() == digests[r]
            else:
                gather_ok &= len(part) > 0
        if wl.dict is not None:
            gather_ok &= gathered_bytes[:gathered_sizes[0]] == got_dev
    hbm, peak_src = peaks()
    value = wl.total_input * args.steps / (ms / 1e3) / 1e9
    e2e = wl.total_input * args.steps / e2e_s / 1e9
    dom = max(("cand_ms", "parse_ms", "literals_ms", "sequences_ms", "stitch_ms"), key=lambda k: kern[k])
    achieved = (size + csize) / (kern[dom] / 1e3) / 1e9
    # DRAM bytes of that kernel per launch: from the committed ncu capture of this workload (not measured live)
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            tj = json.load(f)
        k = tj["kernels"][dom.replace("_ms", "")]
        if args.config == 2 and args.scale == 1.0:
            traffic, traffic_src = k["dram_read_bytes"] + k["dram_write_bytes"], "profiles/r2_traffic.json (ncu --set full, same workload)"
    except Exception:
        pass
    # CPU baseline on this box: the reference on a bounded sample of the same workload (rank 0's share)
    cpu, ref_csize, ref_bytes = None, None, None
    if zref.have_ref() and not args.no_cpu:
        cores = os.cpu_count() or 1
        sample_frames = None if wl.nframes == 1 else max(cores, min(wl.nframes, (2 * GiB) // max(wl.sizes[0], 1)))
        v, per_pass, mode, ref_csize, allmodes, ref_bytes = time_reference(wl, cores, 2, 2, sample_frames)
        cpu = {"value": round(v, 4), "unit": "GB/s", "cores": cores, "kind": "reference",
               "sample": f"{ref_bytes} input bytes of rank 0's share per pass, 2 timed passes after 2 warm-up passes, {host_description()}; {mode}; all modes GB/s: {allmodes}",
               "ref_compressed_bytes": ref_csize}
    ours_for_delta = csize if (ref_bytes == size) else (sum(frame_sizes[:sample_frames]) if ref_bytes else None)
    line = {"metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None,
            "dtype": "u8", "data": wl.data,
            "config": {"workload": wl.desc, "baseline_config": args.config, "level": wl.level,
                       "l2": f"{size} input bytes per GPU per step > 126 MB L2 (no reuse between steps)" if size > 126 * MiB else "input smaller than L2",
                       "compressed_bytes_rank0": csize, "roundtrip_ok": ok_rt, "gathered_decodes_ok": gather_ok,
                       "size_delta_vs_ref": (round((ours_for_delta - ref_csize) / ref_csize, 5) if (ref_csize and ours_for_delta) else None)},
            "kernel_ms": dict({k: round(v, 3) for k, v in kern.items()}, mode="serial (ZSTDB200_SERIAL=1): one wave on one stream, CUDA events around each kernel, rank 0's share"),
            "roofline": {"bound": "hbm", "kernel": dom.replace("_ms", ""), "achieved": round(achieved, 1), "peak": hbm, "unit": "GB/s",
                         "frac": round(achieved / hbm, 4), "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes": size + csize, "read_only_frac": round(size / (kern[dom] / 1e3) / 1e9 / hbm, 4)},
            "cpu_baseline": cpu,
            "e2e": {"value": round(e2e, 3), "unit": "GB/s", "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_total,
                    "api": "ZSTD_compressCCtx(host pinned src/dst)" if (wl.nframes == 1) else ("ZSTDB200_compressFrames_usingCDict" if cdict is not None else "ZSTDB200_compressFrames") + "(host pinned src/dst)"},
            "decode": decode, "gpu_launches": launches, "clocks": clocks, "wall_s": round(wall, 3)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json workload (default 2: the one the metric is quoted on)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (development only; 1.0 = the BASELINE size)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-decode", action="store_true", help="skip the GPU decompression round trip (configs 2 and 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
