#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 zstd batch codec.

Workload (BASELINE.json configs[1]): multi_decompress_to_buffer over 262144 independent 4 KiB
level-3 frames (1 GiB uncompressed) per GPU.  One step = one pass of the hot path over that batch.

  value : uncompressed GB/s with the batch resident in HBM (device-resident C-ABI call), CUDA-event timed
  e2e   : the same through the public API (ZstdDecompressor.multi_decompress_to_buffer) with HOST buffers:
          pinned input -> H2D -> kernels -> D2H into a pinned result, copies inside the timed region
  roofline : algorithmic bytes (U + C + 32 B index per frame) / the dominant kernel's mean launch time
  cpu_baseline : the unmodified reference codec (oracle/_ref) through the reference's batch orchestration
                 on this box's host cores

`--impl reference` times only that CPU arm.  Under torchrun (N > 1) every rank runs the same batch on
its own GPU (weak scaling, no data-path collective); time = max over ranks.
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
import corpus  # noqa: E402

N_FRAMES = 262144
FRAME = 4096
METRIC = "uncompressed GB/s (compress+decompress)"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def host_threads():
    """Threads the CPU arms may really use: the scheduler affinity of this process, cut by the cgroup CPU quota.
    os.cpu_count() is the machine's count and says nothing about the lease (BASELINE.md 3.3)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    use = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return use, {"os_cpu_count": os.cpu_count(), "sched_getaffinity": aff, "cgroup_cpu_quota": quota, "threads_used": use}


def pin_to_gpu_numa(local, world, info):
    """With several ranks on one box every rank's pinned buffers and copy threads should sit on the NUMA node of its GPU
    (round 1: end-to-end scaling 0.59 / 0.50 at 4 / 8 GPUs with unpinned ranks).  The GPU's local CPUs come from sysfs."""
    if world <= 1 or os.environ.get("ZB_BENCH_NO_PIN"):
        return
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-"); cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["numa_pin"] = {"pci": bdf, "local_cpulist": txt, "cpus": len(allowed)}
    except Exception as e:
        info["numa_pin"] = {"error": repr(e)}


def pick_threads(run, info):
    """The CPU arm gets whichever thread count is FASTER on this lease: the quota-sized pool or one thread per visible
    core (under a CFS quota a short burst on all cores can beat the quota-sized pool).  run(threads) -> seconds."""
    cands = sorted({info["threads_used"], info["sched_getaffinity"]})
    best_t, best = cands[0], None
    tried = {}
    for t in cands:
        run(t)
        dt = min(run(t), run(t))
        tried[t] = dt
        if best is None or dt < best:
            best, best_t = dt, t
    info["threads_tried_s"] = {str(k): v for k, v in tried.items()}
    info["threads_used"] = best_t
    return best_t


# The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, for one) write to fd 1 from C, so
# fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved original stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


def make_batch(n_frames, threads):
    """Synthetic input: n frames of S-text compressed by the UNMODIFIED reference codec at level 3
    (this is the workload generator, outside every timed region)."""
    from oracle import RefZstd
    ref = RefZstd()
    blob, off, ln = corpus.text_segments(n_frames, FRAME)
    cblob, clens = ref.batch(True, blob, off, ln, level=3, threads=threads)
    coff = np.concatenate([[0], np.cumsum(clens)[:-1]]).astype(np.uint64)
    return ref, blob, cblob, coff, clens.astype(np.uint64)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.p = None

    def __enter__(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None
        return self

    def _read(self):
        for line in self.p.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.p:
            time.sleep(0.15)
            self.p.terminate()
            try:
                self.p.wait(timeout=2)
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_FRAMES = 2048


def dump_outputs(dirname, ctx, res, n_frames, rank):
    """What a caller of the timed path receives from one step: the decoded bytes and the (offset, length) of every frame in
    them.  The bytes of a fixed, seeded sample of DUMP_FRAMES frames are written (float32, 32 MiB), the segment table in
    full (float64, exact for offsets below 2**53), so that two builds can be compared output for output."""
    import ctypes as C
    L = ctx.L
    seg = np.ctypeslib.as_array(C.cast(L.zb200_result_segments(res), C.POINTER(C.c_uint64)), shape=(n_frames, 2)).copy()
    data = np.empty(int(L.zb200_result_size(res)), dtype=np.uint8)
    ctx.check(L.zb200_memcpy_d2h(ctx.h, data.ctypes.data, L.zb200_result_data(res), len(data)), "d2h")
    pick = np.sort(np.random.default_rng(0).choice(n_frames, min(n_frames, DUMP_FRAMES), replace=False))
    sample = np.concatenate([data[int(seg[i, 0]):int(seg[i, 0] + seg[i, 1])] for i in pick])
    suffix = "" if rank == 0 else "_rank%d" % rank
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "decompressed_sample%s.npy" % suffix), sample.astype(np.float32))
    np.save(os.path.join(dirname, "sample_frames%s.npy" % suffix), pick.astype(np.float64))
    np.save(os.path.join(dirname, "segments%s.npy" % suffix), seg.astype(np.float64))


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads, host_info = host_threads()
    ref, blob, cblob, coff, clens = make_batch(N_FRAMES, host_info["sched_getaffinity"])
    sizes = np.full(N_FRAMES, FRAME, dtype=np.uint64)

    def one(t):
        t0 = time.perf_counter(); ref.batch(False, cblob, coff, clens, dst_len=sizes, threads=t, gather=False); return time.perf_counter() - t0
    threads = pick_threads(one, host_info)
    for _ in range(args.warmup):
        ref.batch(False, cblob, coff, clens, dst_len=sizes, threads=threads, gather=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.batch(False, cblob, coff, clens, dst_len=sizes, threads=threads, gather=False)
    dt = (time.perf_counter() - t0) / args.steps
    gbs = len(blob) / dt / 1e9
    emit({
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "multi_decompress_to_buffer: %d x 4 KiB independent level-3 frames (S-text), host CPU" % N_FRAMES,
                   "threads": threads, "host": host_info},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "reference",
                         "sample": "the full %d-frame batch per step (oracle/_ref libzstd 1.5.7 -O3, reference batch orchestration)" % N_FRAMES},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def run_dictionary_arm(zstd, ref, cores, device):
    """BASELINE.json configs[3]: 1,048,576 x ~1 KiB JSON-like records with a trained dictionary, compress + decompress
    through the public API (host buffers), the unmodified reference on the host cores beside it.  The records are
    16384 distinct ones repeated (every record is an independent frame, so repeats do not help either codec)."""
    n_unique, n = 16384, int(os.environ.get("ZB_BENCH_DICT_RECORDS", "1048576"))
    recs = corpus.json_records(n_unique + 2000)
    dct = ref.train_dictionary(112640, recs[:2000])
    recs = recs[2000:]
    one = np.frombuffer(b"".join(recs), dtype=np.uint8)
    ln1 = np.array([len(r) for r in recs], dtype=np.uint64)
    reps = max(1, n // n_unique)
    n = reps * n_unique
    blob = np.tile(one, reps)
    ln = np.tile(ln1, reps)
    off = np.concatenate([[0], np.cumsum(ln)[:-1]]).astype(np.uint64)
    U = int(ln.sum())
    rc, rl = ref.batch(True, blob, off, ln, level=3, threads=cores, dict_data=dct)
    rl = rl.astype(np.uint64)
    ro = np.concatenate([[0], np.cumsum(rl)[:-1]]).astype(np.uint64)
    tc = td = 1e9
    for _ in range(2):
        t0 = time.perf_counter(); ref.batch(True, blob, off, ln, level=3, threads=cores, dict_data=dct, gather=False); tc = min(tc, time.perf_counter() - t0)
        t0 = time.perf_counter(); ref.batch(False, rc, ro, rl, dst_len=ln, threads=cores, dict_data=dct, gather=False); td = min(td, time.perf_counter() - t0)
    d = zstd.ZstdCompressionDict(dct)
    pin = zstd.PinnedBuffer(len(blob), device=device); np.frombuffer(pin, dtype=np.uint8)[:] = blob
    bws = zstd.BufferWithSegments(pin, np.stack([off, ln], axis=1).astype(np.uint64).tobytes())
    cctx = zstd.ZstdCompressor(level=3, dict_data=d)
    dctx = zstd.ZstdDecompressor(dict_data=d)
    res = cctx.multi_compress_to_buffer(bws)
    csz = res.size()
    back = dctx.multi_decompress_to_buffer(res)          # our frames regenerate (sampled) ...
    step = max(1, n // 4099)
    ok = all(back[i].tobytes() == recs[i % n_unique] for i in range(0, n, step))
    del back
    # ... and the reference decoder regenerates them all
    datas, segs, base = [], [], 0
    for b_ in (res._buffers if hasattr(res, "_buffers") else [res]):
        d_ = np.frombuffer(b_.tobytes(), dtype=np.uint8)
        g_ = np.frombuffer(b_._segments, dtype=np.uint64).reshape(-1, 2).copy()
        g_[:, 0] += np.uint64(base)
        datas.append(d_); segs.append(g_); base += len(d_)
    seg = np.concatenate(segs)
    rb, _ = ref.batch(False, np.concatenate(datas), np.ascontiguousarray(seg[:, 0]), np.ascontiguousarray(seg[:, 1]),
                      dst_len=ln, threads=cores, dict_data=dct)
    ok_ref = bool(np.array_equal(rb, blob))
    del rb
    tg = tgd = 1e9
    for _ in range(3):
        t0 = time.perf_counter(); r2 = cctx.multi_compress_to_buffer(bws); _ = r2[n - 1].tobytes(); tg = min(tg, time.perf_counter() - t0); del r2
    pin2 = zstd.PinnedBuffer(len(rc), device=device); np.frombuffer(pin2, dtype=np.uint8)[:] = rc
    fbws = zstd.BufferWithSegments(pin2, np.stack([ro, rl], axis=1).astype(np.uint64).tobytes())
    o2 = dctx.multi_decompress_to_buffer(fbws); ok_dec = o2[n - 1].tobytes() == recs[(n - 1) % n_unique]; del o2
    for _ in range(3):
        t0 = time.perf_counter(); o2 = dctx.multi_decompress_to_buffer(fbws); _ = o2[n - 1].tobytes(); tgd = min(tgd, time.perf_counter() - t0); del o2
    return {
        "workload": "%d x ~%d B JSON-like records (%d distinct), trained %d-byte dictionary, level 3; public API with host buffers"
                    % (n, U // n, n_unique, len(dct)),
        "compress_e2e": {"value": U / tg / 1e9, "unit": "GB/s", "ms": tg * 1e3},
        "decompress_e2e": {"value": U / tgd / 1e9, "unit": "GB/s", "ms": tgd * 1e3},
        "ratio": U / csz, "reference_ratio": U / float(rl.sum()), "size_vs_reference_pct": 100.0 * (csz / float(rl.sum()) - 1.0),
        "roundtrip": {"own_decoder_sampled": bool(ok), "reference_decoder_all": ok_ref, "reference_frames_on_gpu": bool(ok_dec)},
        "cpu_baseline": {"compress": U / tc / 1e9, "decompress": U / td / 1e9, "unit": "GB/s", "cores": cores, "kind": "reference",
                         "sample": "the same batch, best of 2"},
    }


def run_large_frame_arm(zstd, ref):
    """BASELINE.json configs[4] on a bounded sample: ONE frame of 128 KiB blocks (level 3, cross-block matches, repeated
    tables) read through ZstdDecompressor.stream_reader; the block-parallel path decodes the entropy stage a lane per
    block and executes block after block in shared memory.  The reference's decoder is single-threaded on one frame."""
    import io
    mb = int(os.environ.get("ZB_BENCH_FRAME_MB", "256"))
    t = corpus.text_corpus(8 << 20)
    data = np.tile(t, (mb << 20) // len(t) + 1)[:mb << 20].tobytes()
    frame = ref.compress(data, level=3)
    import ctypes as C
    Z = ref.Z
    dc = Z.ZSTD_createDCtx()
    outbuf = np.empty(len(data), dtype=np.uint8); outbuf[:] = 0          # pages touched before the clock starts
    tcpu = 1e9
    for _ in range(2):
        t0 = time.perf_counter()
        got = Z.ZSTD_decompressDCtx(dc, C.c_void_p(outbuf.ctypes.data), len(data), frame, len(frame))
        tcpu = min(tcpu, time.perf_counter() - t0)
    Z.ZSTD_freeDCtx(dc)
    assert got == len(data) and outbuf.tobytes() == data
    del outbuf
    d = zstd.ZstdDecompressor(max_window_size=1 << 31)
    best = 1e9
    for _ in range(3):
        t0 = time.perf_counter()
        chunks = []
        with d.stream_reader(io.BytesIO(frame)) as r:
            while True:
                c = r.read(8 << 20)
                if not c:
                    break
                chunks.append(c)
        best = min(best, time.perf_counter() - t0)
        mv = memoryview(data); pos = 0                 # verified outside the timed region
        for c in chunks:
            assert c == mv[pos:pos + len(c)]; pos += len(c)
        assert pos == len(data)
        del chunks
    t0 = time.perf_counter(); out = d.decompress(frame); tdec = time.perf_counter() - t0
    assert out == data
    return {"workload": "stream_reader over ONE %d MiB frame of %d x 128 KiB blocks (level 3, reference-compressed, %.1f MiB)"
                        % (mb, (len(data) + 131071) // 131072, len(frame) / 2**20),
            "stream_reader": {"value": len(data) / best / 1e9, "unit": "GB/s", "s": best, "verified": "every chunk compared with the input"},
            "decompress": {"value": len(data) / tdec / 1e9, "unit": "GB/s", "s": tdec},
            "cpu_baseline": {"value": len(data) / tcpu / 1e9, "unit": "GB/s", "cores": 1, "kind": "reference",
                             "sample": "ZSTD_decompressDCtx of the same frame (one frame is one thread's work in the reference)"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--frames", type=int, default=N_FRAMES)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step decoded to DIR/*.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import ctypes as C
    import torch
    import torch.distributed as dist
    import python_zstandard_b200 as zstd
    from python_zstandard_b200 import _native

    torch.cuda.set_device(local)
    zstd.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_frames = args.frames
    cores, host_info = host_threads()
    orig_affinity = os.sched_getaffinity(0)
    threads = max(1, host_info["sched_getaffinity"] // world)
    ref, blob, cblob, coff, clens = make_batch(n_frames, threads)
    U, Cb = int(len(blob)), int(len(cblob))
    if rank == 0:
        sizes0 = np.full(n_frames, FRAME, dtype=np.uint64)

        def one_dec(t):
            t0 = time.perf_counter(); ref.batch(False, cblob, coff, clens, dst_len=sizes0, threads=t, gather=False); return time.perf_counter() - t0
        cores = pick_threads(one_dec, host_info)
    pin_to_gpu_numa(local, world, host_info)          # before the codec context (pinned pools, worker threads) exists
    log("[rank %d] batch: %d frames, U=%d B, C=%d B, ratio %.3f" % (rank, n_frames, U, Cb, U / Cb))
    segs = np.stack([coff, clens], axis=1).astype(np.uint64)

    ctx = _native.Context.get(local)
    L = ctx.L
    stream = torch.cuda.ExternalStream(L.zb200_ctx_stream(ctx.h), device=torch.device("cuda", local))

    # ---------------- device-resident arm: `value`
    d_src = torch.empty(Cb + 256, dtype=torch.uint8, device="cuda")
    d_src[:Cb].copy_(torch.from_numpy(cblob))
    d_segs = torch.from_numpy(segs.view(np.int64).copy()).cuda()
    torch.cuda.synchronize()

    def step_device():
        res = C.c_void_p()
        rc = L.zb200_decompress_batch(ctx.h, d_src.data_ptr(), d_segs.data_ptr(), n_frames, None, None,
                                      _native.SRC_DEVICE | _native.DST_DEVICE, C.byref(res))
        ctx.check(rc, "zb200_decompress_batch")
        return res

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # correctness gate before any number is recorded: byte-equal to the original
    res = step_device()
    if L.zb200_result_first_error(res, None, None, None, None):
        raise SystemExit("decode error in the benchmark batch")
    out = np.empty(U, dtype=np.uint8)
    ctx.check(L.zb200_memcpy_d2h(ctx.h, out.ctypes.data, L.zb200_result_data(res), U), "d2h")
    L.zb200_result_free(res)
    if not np.array_equal(out, blob):
        raise SystemExit("benchmark batch decoded to different bytes")
    del out

    for _ in range(args.warmup):
        L.zb200_result_free(step_device())
    ctx.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last_res = None
    barrier()
    with ClockSampler(local) as clk:
        e0.record(stream)
        for i in range(args.steps):
            res = step_device()
            if args.dump_outputs and i + 1 == args.steps:
                last_res = res
            else:
                L.zb200_result_free(res)
        e1.record(stream)
        barrier()
    dev_ms = e0.elapsed_time(e1) / args.steps
    if last_res is not None:
        dump_outputs(args.dump_outputs, ctx, last_res, n_frames, rank)
        L.zb200_result_free(last_res)
    prof = ctx.profile_read()
    ctx.profile(False)
    scratch = int(L.zb200_last_scratch_bytes(ctx.h))

    # ---------------- end-to-end arm through the public API with host buffers
    pin = zstd.PinnedBuffer(Cb, device=local)
    np.frombuffer(pin, dtype=np.uint8)[:] = cblob
    bws = zstd.BufferWithSegments(pin, segs.tobytes())
    dctx = zstd.ZstdDecompressor()
    for _ in range(args.warmup):
        r = dctx.multi_decompress_to_buffer(bws)
        del r
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = dctx.multi_decompress_to_buffer(bws)
        last = r[n_frames - 1].tobytes()          # touch the result on the host
        del r
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    assert last == blob[-FRAME:].tobytes()

    # ---------------- the same call with DEVICE buffers (SURVEY section 8(f)-2): DeviceBufferWithSegments in, DeviceBufferWithSegments
    # out through the public Python API -- what a GPU-resident caller (torch tensors) sees; only the segment table crosses PCIe
    dbuf = zstd.DeviceBufferWithSegments(d_src[:Cb], segs.tobytes())
    for _ in range(args.warmup):
        r = dctx.multi_decompress_to_buffer(dbuf)
        del r
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = dctx.multi_decompress_to_buffer(dbuf)
        if _ + 1 < args.steps:
            del r
    barrier()
    dev_api_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    assert r[n_frames - 1].tobytes() == blob[-FRAME:].tobytes()
    del r
    if os.environ.get("ZB_BENCH_PROFILE_DEVICE_API"):
        import cProfile, pstats, io as _io
        pr_ = cProfile.Profile(); pr_.enable(); r = dctx.multi_decompress_to_buffer(dbuf); del r; pr_.disable()
        so_ = _io.StringIO(); pstats.Stats(pr_, stream=so_).sort_stats("cumulative").print_stats(12); log(so_.getvalue())

    # ---------------- secondary arm: multi_compress_to_buffer on 128 KiB Silesia-mix segments (configs[2], scaled)
    # BASELINE.json configs[2] in full: 65536 x 128 KiB, ONE batch cut by segment index over the ranks (strong scaling:
    # every GPU gets 65536 / N segments, no data-path collective).  ZB_BENCH_COMPRESS_SEGMENTS shrinks it for experiments.
    cn_total = int(os.environ.get("ZB_BENCH_COMPRESS_SEGMENTS", "65536"))
    cn = cn_total // world
    cblob_in, coff_in, cln_in = corpus.silesia_mix(cn, 131072, seed=3 + rank)
    csegs = np.stack([coff_in, cln_in], axis=1).astype(np.uint64)
    d_cin = torch.empty(len(cblob_in) + 256, dtype=torch.uint8, device="cuda")
    d_cin[:len(cblob_in)].copy_(torch.from_numpy(cblob_in))
    d_csegs = torch.from_numpy(csegs.view(np.int64).copy()).cuda()
    cparams = zstd.compressor.CParams(3, 0, 1, 0)

    def step_compress():
        r_ = C.c_void_p()
        rc_ = L.zb200_compress_batch(ctx.h, d_cin.data_ptr(), d_csegs.data_ptr(), cn, C.byref(cparams), None,
                                     _native.SRC_DEVICE | _native.DST_DEVICE, C.byref(r_))
        ctx.check(rc_, "zb200_compress_batch")
        return r_

    r0 = step_compress()
    csz = int(L.zb200_result_size(r0))
    comp_bytes = np.empty(csz, dtype=np.uint8)
    ctx.check(L.zb200_memcpy_d2h(ctx.h, comp_bytes.ctypes.data, L.zb200_result_data(r0), csz), "d2h")
    comp_segs = np.ctypeslib.as_array(C.cast(L.zb200_result_segments(r0), C.POINTER(C.c_uint64)), shape=(cn, 2)).copy()
    L.zb200_result_free(r0)
    # correctness gate: the reference decoder regenerates the input bit-exact
    rb, _ = ref.batch(False, comp_bytes, np.ascontiguousarray(comp_segs[:, 0]), np.ascontiguousarray(comp_segs[:, 1]),
                      threads=threads)
    if not np.array_equal(rb, cblob_in):
        raise SystemExit("compressed batch does not round-trip through the reference decoder")
    for _ in range(2):
        L.zb200_result_free(step_compress())
    ce0, ce1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    csteps = args.steps
    barrier()
    ce0.record(stream)
    for _ in range(csteps):
        L.zb200_result_free(step_compress())
    ce1.record(stream)
    barrier()
    comp_ms = ce0.elapsed_time(ce1) / csteps
    cpin = zstd.PinnedBuffer(len(cblob_in), device=local)
    np.frombuffer(cpin, dtype=np.uint8)[:] = cblob_in
    cbws = zstd.BufferWithSegments(cpin, csegs.tobytes())
    cctx = zstd.ZstdCompressor(level=3)
    cctx.multi_compress_to_buffer(cbws)
    barrier()
    t0 = time.perf_counter()
    for _ in range(csteps):
        rr = cctx.multi_compress_to_buffer(cbws)
        _ = rr[cn - 1].tobytes()
        del rr
    barrier()
    comp_e2e_ms = (time.perf_counter() - t0) * 1e3 / csteps
    ctx.profile(True)
    L.zb200_result_free(step_compress())
    comp_prof = ctx.profile_read()
    comp_kernel = L.zb200_last_compress_kernel(ctx.h).decode()
    ctx.profile(False)
    del d_cin, cpin, cbws, cctx

    times = torch.tensor([dev_ms, e2e_ms, comp_ms, comp_e2e_ms, dev_api_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, comp_ms, comp_e2e_ms, dev_api_ms = (float(times[i]) for i in range(5))

    # ---------------- one call, one batch, N devices: the in-process partition (threads -> devices) of the public API
    sharded = None
    if world > 1:
        barrier()
        if rank == 0 and torch.cuda.device_count() >= world:
            dsh = zstd.ZstdDecompressor()
            r = dsh.multi_decompress_to_buffer(bws, threads=world); del r
            ts = []
            for _ in range(max(3, args.steps // 2)):
                t0 = time.perf_counter()
                r = dsh.multi_decompress_to_buffer(bws, threads=world)
                lastb = r[n_frames - 1].tobytes(); del r
                ts.append(time.perf_counter() - t0)
            assert lastb == blob[-FRAME:].tobytes()
            sharded = {"api": "ZstdDecompressor.multi_decompress_to_buffer(threads=%d): one process, the batch cut by segment "
                              "index over %d devices, host buffers" % (world, world),
                       "value": U / min(ts) / 1e9, "unit": "GB/s", "ms_per_step": min(ts) * 1e3, "devices": world}
        barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    os.sched_setaffinity(0, orig_affinity)             # the CPU arms below get every core of the lease again
    dict_info = None
    try:
        dict_info = run_dictionary_arm(zstd, ref, cores, local)
    except Exception as e:          # the arm is secondary: report, do not lose the headline line
        dict_info = {"error": repr(e)}
    try:
        frame_info = run_large_frame_arm(zstd, ref)
    except Exception as e:
        frame_info = {"error": repr(e)}

    # ---------------- roofline of the dominant kernel
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    alg_bytes = U + Cb + 32 * n_frames
    kernels = {k: {"ms_per_launch": v[0] / v[1], "launches": v[1]} for k, v in prof.items()}
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_launch"])
    achieved = alg_bytes / (kernels[dom]["ms_per_launch"] * 1e-3) / 1e9
    traffic = None          # DRAM bytes per step: the SUM over the step's kernels (one ncu --set full capture, profiles/traffic.json)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = sum(int(tj[k]) for k in tj if k.startswith("zb_") and not k.startswith("zb_compress"))
    except Exception:
        pass
    # the library times spans, some of which hold two kernels: placement = zb_place_reduce + zb_place_scan, execute =
    # zb_execute_tile + zb_execute (frames above the 4 KiB tile; exits at once when there are none)
    per_span = {"zb_place_frames": 2, "zb_execute": 2}
    launches = sum(v["launches"] * per_span.get(k, 1) for k, v in kernels.items())

    # ---------------- CPU baseline: the unmodified reference on this box's cores, same batch
    sizes = np.full(n_frames, FRAME, dtype=np.uint64)

    ref.batch(False, cblob, coff, clens, dst_len=sizes, threads=cores, gather=False)
    best = 1e9
    for _ in range(3):
        t0 = time.perf_counter()
        ref.batch(False, cblob, coff, clens, dst_len=sizes, threads=cores, gather=False)
        best = min(best, time.perf_counter() - t0)
    t0 = time.perf_counter()
    sub = min(n_frames, 16384)
    ref.batch(False, cblob, coff[:sub].copy(), clens[:sub].copy(), dst_len=sizes[:sub].copy(), threads=1, gather=False)
    one_core = sub * FRAME / (time.perf_counter() - t0) / 1e9

    tcb = 1e9
    for _ in range(3):
        t0 = time.perf_counter()
        refc_total = ref.batch(True, cblob_in, coff_in, cln_in, level=3, threads=cores, gather=False)
        tcb = min(tcb, time.perf_counter() - t0)
    ck = {k: {"ms_per_launch": v[0] / v[1], "launches": v[1]} for k, v in (comp_prof or {}).items()}
    cdom = max(ck, key=lambda k: ck[k]["ms_per_launch"]) if ck else None
    c_alg = len(cblob_in) + csz + 32 * cn
    compress_info = {
        "workload": "multi_compress_to_buffer: %d x 128 KiB Silesia-mix segments in all (BASELINE configs[2]), cut by segment "
                    "index over %d GPU(s): %d per GPU, level-3 class" % (cn * world, world, cn),
        "scaling": "strong", "segments_total": cn * world, "segments_per_gpu": cn,
        "value": world * len(cblob_in) / (comp_ms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": comp_ms,
        "e2e": {"value": world * len(cblob_in) / (comp_e2e_ms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": comp_e2e_ms,
                "h2d_bytes_per_step": len(cblob_in) + 16 * cn, "d2h_bytes_per_step": csz + 16 * cn},
        "kernels": ck,
        "roofline": None if not cdom else {"bound": "hbm", "kernel": (comp_kernel if cdom == "zb_compress_blocks" else cdom), "achieved": c_alg / (ck[cdom]["ms_per_launch"] * 1e-3) / 1e9,
                                           "peak": peak, "unit": "GB/s", "frac": c_alg / (ck[cdom]["ms_per_launch"] * 1e-3) / 1e9 / peak,
                                           "algorithmic_bytes_per_launch": c_alg,
                                           "note": "rank 0's shard; shared-memory and issue bound (one CTA per SM, block resident in shared memory)"},
        "ratio": len(cblob_in) / csz, "reference_level3_ratio": len(cblob_in) / refc_total,
        "size_vs_reference_pct": 100.0 * (csz / refc_total - 1.0),
        "roundtrip": "reference decoder regenerates the input bit-exact",
        "cpu_baseline": {"value": len(cblob_in) / tcb / 1e9, "unit": "GB/s", "cores": cores, "kind": "reference",
                         "sample": "rank 0's shard (%d segments), best of 3, ZSTD_compressStream2(e_end) per segment on %d threads" % (cn, cores)},
    }
    emit({
        "metric": METRIC, "value": world * U / (dev_ms * 1e-3) / 1e9, "unit": "GB/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "multi_decompress_to_buffer: %d x 4 KiB independent level-3 frames per GPU "
                               "(S-text, reference-compressed, ratio %.2f)" % (n_frames, U / Cb),
                   "l2": "inputs (%d MB compressed + %d MB output per step) exceed the 126 MB L2; no flush needed"
                         % (Cb >> 20, U >> 20),
                   "sharding": "independent frames, one process per GPU, every GPU decodes its own batch of this size (weak scaling, "
                               "no data-path collective); `compress` below is ONE batch cut over the GPUs, `sharded` one call over N devices"},
        "e2e": {"value": world * U / (e2e_ms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": Cb + 16 * n_frames, "d2h_bytes_per_step": U + 16 * n_frames,
                "api": "ZstdDecompressor.multi_decompress_to_buffer(BufferWithSegments in pinned host memory)"},
        "device_api": {"value": world * U / (dev_api_ms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": dev_api_ms,
                       "h2d_bytes_per_step": 16 * n_frames, "d2h_bytes_per_step": 0,
                       "api": "ZstdDecompressor.multi_decompress_to_buffer(DeviceBufferWithSegments) -> DeviceBufferWithSegments: the "
                              "public Python call for GPU-resident callers (wall clock, result checked)"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes,
                     "note": "latency/issue-bound bitstream work; fraction of HBM copy bandwidth"},
        "kernels": kernels,
        "compress": compress_info,
        "dictionary": dict_info,
        "large_frame": frame_info,
        "sharded": sharded,
        "host": host_info,
        "scratch_bytes_per_step": scratch,
        "cpu_baseline": {"value": U / best / 1e9, "unit": "GB/s", "cores": cores, "kind": "reference",
                         "one_core_GBps": one_core,
                         "sample": "the same %d-frame batch, best of 3 (oracle/_ref libzstd 1.5.7 -O3 via the "
                                   "reference batch orchestration restated in oracle/ref_batch.c)" % n_frames},
        "clocks": clk.summary(),
    })
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
