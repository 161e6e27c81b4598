#!/usr/bin/env python
"""bench.py — the hot-path benchmark (BASELINE.json metric: compress+decompress MB/s, % HBM roofline).

A "step" is one pass of the hot path over one batch of synthetic input: compress, then decompress, 1024 independent
chunks of 2^18 u64 (BASELINE config 2: classic mode, consecutive delta order 1; C2(i) data).  Per rank, N ranks = weak
scaling (8 ranks = config 4's 8192 chunks).  MB = 10^6 uncompressed bytes (pco_cli/src/bench/mod.rs:233-241).

  value     resident: inputs already in HBM, device buffers in and out, through the C-ABI (*_ex, flags DEVICE).
  e2e       same calls with pinned HOST buffers (H2D of the inputs and D2H of the results inside the timed region), streamed in chunk groups by
            2 + 2 host threads; e2e.single_call = one call pair over the whole array; e2e.reference_abi = the reference's 3-function ABI as is.
  roofline  fused_narrow_kernel (the decompress kernel on this data): (U + C) bytes / its CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs;
            roofline.call / roofline.compress = the same bytes over the whole decompress / compress call.
  cpu_baseline / --impl reference: oracle/ (C++ restatement of pco 1.0.3; the Rust reference cannot be built here)
            on the host cores - one worker process per host thread - on a bounded sample of the same chunks.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHUNK_N = 1 << 18
N_CHUNKS = 1024
METRIC = "compress+decompress MB/s per chunk (u64, 2^18 elems)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunks", type=int, default=N_CHUNKS, help="chunks per rank (default: BASELINE config 2)")
    ap.add_argument("--cpu-sample-chunks", type=int, default=1024, help="chunks of the CPU arm per step, spread over one worker process per host thread (about 12 s of core time)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--abi3-chunks", type=int, default=256, help="chunks of the three-function-ABI leg (no side index, no chunk offsets: the decompressor finds the chunks by speculation, host_api.cu speculative_walk_rounds)")
    ap.add_argument("--e2e-groups", type=int, default=16, help="chunk groups the streamed e2e leg cuts the array into")
    ap.add_argument("--e2e-threads", type=int, default=2, help="host threads per direction in the streamed e2e leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-index-free", action="store_true", help="skip the pco_b200_decompress_chunks timing (not part of `value`)")
    ap.add_argument("--results-csv", default=None, help="also merge this run into a CSV with the reference bench tool's schema and codec naming (pcodec_b200/benchfmt.py)")
    ap.add_argument("--no-gather-pages", action="store_true", help="N > 1: exchange only the per-chunk sizes; the default also gathers the compressed pages on the device (every rank ends up with the whole file)")
    ap.add_argument("--gather-ctas", type=int, default=0, help="CTAs of the page-gather copy kernel (it runs beside the next step's kernels on a high-priority stream); 0 = 16 per rank of the job, at most 64 (profiles/r02_zz3_gather_sweep.txt)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned to its caller (rank 0) as DIR/<name>.npy: seeded samples of the decompressed "
                         "numbers (float64), of the compressed file and of its side index (bytes as float32), and every chunk's compressed size (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs the GPU arm (--impl ours)")
    return args


# Sizes of the --dump-outputs samples: 16 + 16 + 4 MiB as written, under 64 MiB with the per-chunk sizes.  Positions come from
# DUMP_SEED and the array's length alone, so two builds that return the same outputs write the same files.
DUMP_SEED = 20251017
DUMP_NUMS, DUMP_FILE_BYTES, DUMP_INDEX_BYTES = 1 << 21, 1 << 22, 1 << 20


def dump_positions(length, k):
    """Sorted positions of the dump's sample of an array of `length` elements: all of them when there are at most `k`."""
    if length <= k:
        return np.arange(length, dtype=np.int64)
    return np.sort(np.random.default_rng([DUMP_SEED, length]).integers(0, length, size=k, dtype=np.int64))


def dump_outputs(out_dir, d_out, d_comp, n_comp, d_index, n_index, chunk_offs):
    """Writes the last timed step's outputs.  The numbers of this workload stay below 2^53, so float64 holds them exactly."""
    import torch

    os.makedirs(out_dir, exist_ok=True)

    def sample(t, length, k):
        return t[torch.from_numpy(dump_positions(length, k)).to(t.device)].cpu()

    np.save(os.path.join(out_dir, "decompressed.npy"), sample(d_out, d_out.numel(), DUMP_NUMS).numpy().view(np.uint64).astype(np.float64))
    np.save(os.path.join(out_dir, "compressed.npy"), sample(d_comp, n_comp, DUMP_FILE_BYTES).numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "index.npy"), sample(d_index, n_index, DUMP_INDEX_BYTES).numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "chunk_compressed_bytes.npy"), np.diff(np.asarray(chunk_offs, dtype=np.float64)))


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores (the one place bench.py may execute oracle/)
# ------------------------------------------------------------------------------------------------
# One worker PROCESS per host thread, each compressing and decompressing its own chunks with the oracle
# (oracle/c_api.cpp pco_oracle_bench_roundtrip, one native thread).  Processes, not threads: the port allocates MiB-sized
# scratch per chunk and threads of one process serialise in the kernel's address-space lock (8 threads: 1.6x one thread for
# compress), and a Python thread pool around per-chunk ctypes calls adds GIL-held buffer copies on top.  Measured on the
# authoring box: 8 processes = 8x one.
_W = {}
CPU_RUN_TIMEOUT_S = 120  # one timed pass of the pool; far above the ~1 s it takes


def host_threads():
    """Host threads this process may really use: the affinity mask, capped by a cgroup CPU quota when one is set."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def _cpu_worker_init(counter, barrier, chunks_per_worker):
    from oracle import pyoracle
    from pcodec_b200 import datagen

    with counter.get_lock():
        wid = counter.value
        counter.value += 1
    cfg = pyoracle.make_config(level=8, mode=pyoracle.MODE_CLASSIC, delta=pyoracle.DELTA_CONSECUTIVE, delta_order=1)
    nums = np.concatenate([datagen.c2_u64_cumsum_geometric(CHUNK_N, seed=wid * chunks_per_worker + i) for i in range(chunks_per_worker)])
    pyoracle.bench_roundtrip(nums[:CHUNK_N], 1, CHUNK_N, cfg, 1)  # load the library, touch the allocator
    _W.update(nums=nums, cfg=cfg, k=chunks_per_worker, barrier=barrier)


def _cpu_worker_run(_):
    from oracle import pyoracle

    _W["barrier"].wait(timeout=180)  # every worker takes exactly one task and they start together (a lost worker breaks the barrier, it does not hang)
    tc, td, cbytes = pyoracle.bench_roundtrip(_W["nums"], _W["k"], CHUNK_N, _W["cfg"], 1)  # raises if a chunk does not round-trip
    return tc, td, cbytes


class CpuArm:
    """`workers` processes with `chunks_per_worker` C2(i) chunks each; run() = one timed compress + decompress of all of them."""

    def __init__(self, workers, chunks_per_worker):
        import multiprocessing as mp

        from oracle import pyoracle

        pyoracle.build()  # once, here: the workers must find the library up to date instead of racing to rebuild it
        ctx = mp.get_context("spawn")  # the GPU arm's process holds a CUDA context and helper threads: no fork
        self.workers, self.k = workers, chunks_per_worker
        self.pool = ctx.Pool(workers, initializer=_cpu_worker_init, initargs=(ctx.Value("i", 0), ctx.Barrier(workers), chunks_per_worker))

    def run(self):
        """Returns (MB/s round trip, compress MB/s, decompress MB/s, compressed bytes): bytes of all workers over the slowest
        worker's time (they run concurrently from a common barrier)."""
        # map_async + timeout: a pool whose workers die at start-up is respawned forever and a plain map() would never return
        try:
            res = self.pool.map_async(_cpu_worker_run, range(self.workers), chunksize=1).get(timeout=CPU_RUN_TIMEOUT_S + 2 * self.k)
        except Exception:
            self.broken = True
            raise
        mb = self.workers * self.k * CHUNK_N * 8 / 1e6
        tc, td = max(r[0] for r in res), max(r[1] for r in res)
        return mb / max(r[0] + r[1] for r in res), mb / tc, mb / td, sum(r[2] for r in res)

    def close(self):
        if getattr(self, "broken", False):
            self.pool.terminate()
        else:
            self.pool.close()
        self.pool.join()


def cpu_roundtrip(n_chunks, threads, repeats=1):
    """Compress + decompress about `n_chunks` C2(i) chunks on `threads` host threads (one worker process each, at least one
    chunk per worker).  Returns (MB/s round trip, compress MB/s, decompress MB/s, compressed bytes, chunks actually run)."""
    workers = max(1, threads)
    k = max(1, n_chunks // workers)
    arm = CpuArm(workers, k)
    try:
        best = None
        for _ in range(repeats):
            cur = arm.run()
            if best is None or cur[0] > best[0]:
                best = cur
    finally:
        arm.close()
    return best + (workers * k,)


def run_reference_arm(args, rank):
    """--impl reference: the reference's own CPU path of the same workload.  pco is Rust and there is no cargo/rustc in the
    image (SURVEY.md §0), so this runs the oracle port and says so (cpu_baseline.kind = "port")."""
    if rank != 0:
        return
    vals, err = None, None
    for threads in sorted({host_threads(), min(host_threads(), 8), 1}, reverse=True):
        # all host threads; if a pool of that size cannot be brought up on this host, a smaller one still gives a line (and says so)
        k = max(1, args.cpu_sample_chunks // threads)
        sample = threads * k
        try:
            arm = CpuArm(threads, k)
            try:
                for _ in range(args.warmup):
                    arm.run()
                vals, t0 = [], time.perf_counter()
                for _ in range(args.steps):
                    vals.append(arm.run())
                ms = (time.perf_counter() - t0) * 1e3 / max(args.steps, 1)
            finally:
                arm.close()
            break
        except Exception as ex:  # noqa: BLE001
            vals, err = None, f"{threads} workers: {type(ex).__name__}: {ex}"
    if vals is None:
        print(json.dumps({"impl": "reference", "unavailable": f"CPU port could not be run: {err}"}))
        return
    v = float(np.median([x[0] for x in vals]))
    try:
        one = cpu_roundtrip(4, 1)  # BASELINE.md section 2: one thread and all host cores in the same run
    except Exception:  # noqa: BLE001
        one = (None, None, None, 0, 0)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "C2: 2^18-element u64 chunks, classic, consecutive delta order 1, level 8 (cumsum of geometric(0.001))",
                   "chunks_per_step": sample, "chunk_n": CHUNK_N},
        "cpu_baseline": {"value": v, "unit": "MB/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} chunks of 2^18 u64 per step, {k} per worker process, one process per host thread; C++ restatement of pco 1.0.3 (oracle/), not the Rust crate",
                         "compress_mb_s": float(np.median([x[1] for x in vals])), "decompress_mb_s": float(np.median([x[2] for x in vals])),
                         "single_core": {"value": one[0], "compress_mb_s": one[1], "decompress_mb_s": one[2], "sample": f"{one[4]} chunks, one process"},
                         **({"note": f"fewer workers than host threads ({host_threads()}) after: {err}"} if err else {})},
        "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu_index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm, smax, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                smax = max(smax, float(s[1]))
                for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons), "samples": len(sm)}


def parse_profile(L):
    buf = C.create_string_buffer(4096)
    L.pco_b200_profile_last(buf, C.c_size_t(4096))
    out = {}
    for item in buf.value.decode().split(";"):
        if "=" in item:
            k, v = item.split("=")
            out[k] = out.get(k, 0.0) + float(v)
    return out


def run_gpu_arm(args, rank, world):
    import torch

    from pcodec_b200 import ChunkConfig, DeltaSpec, ModeSpec, _lib, datagen

    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        # stdout carries exactly one JSON line: keep NCCL's version banner (NCCL_DEBUG=VERSION prints it to stdout) off it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    if not L.pco_b200_device_available():
        raise RuntimeError("libcpcodec.so found no usable CUDA device: " + L.pco_b200_last_error_message().decode())

    n_chunks = args.chunks
    n = n_chunks * CHUNK_N
    U = n * 8
    cfg = ChunkConfig(compression_level=8, mode_spec=ModeSpec.classic(), delta_spec=DeltaSpec.try_consecutive(1))._to_c()
    # the SAME arrays as the CPU arm (--impl reference / cpu_baseline): chunk c of rank r is datagen.c2_u64_cumsum_geometric(seed =
    # r * n_chunks + c), generated on the host (a few seconds, outside every timed region) and staged through pinned memory
    pinned_ok = not args.no_e2e
    try:
        h_nums = torch.empty(n, dtype=torch.int64, pin_memory=pinned_ok)
    except Exception:  # noqa: BLE001  (a crowded host can refuse 2 GiB of pinned memory: the e2e leg is skipped, the line survives)
        pinned_ok = False
        h_nums = torch.empty(n, dtype=torch.int64)
    h_np = h_nums.numpy().view(np.uint64)
    from concurrent.futures import ThreadPoolExecutor

    def _gen(c):
        h_np[c * CHUNK_N:(c + 1) * CHUNK_N] = datagen.c2_u64_cumsum_geometric(CHUNK_N, seed=rank * n_chunks + c)

    with ThreadPoolExecutor(max(1, min(8, host_threads()))) as ex:
        list(ex.map(_gen, range(n_chunks)))
    nums = h_nums.to(dev)
    cap = L.pco_standalone_guarantee_file_size(n, 2)
    icap = L.pco_b200_index_size_bound(n, n_chunks)
    gather_on = world > 1 and not args.no_gather_pages
    n_bufs = 2 if gather_on else 1  # the page gather of step k reads buffer k % 2 while step k + 1 compresses into the other
    d_comps = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(n_bufs)]
    d_indexes = [torch.empty(icap, dtype=torch.uint8, device=dev) for _ in range(n_bufs)]
    d_comp, d_index = d_comps[0], d_indexes[0]
    step_no = [0]
    d_out = torch.empty(n, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    SRC, DST, IDX = 1, 2, 4
    n_written, ilen = C.c_size_t(), C.c_size_t()
    prog = _lib._CProgress()

    def compress_resident():
        nonlocal d_comp, d_index
        d_comp, d_index = d_comps[step_no[0] % n_bufs], d_indexes[step_no[0] % n_bufs]
        if gather_on and push_done[step_no[0] % n_bufs] is not None:
            push_done[step_no[0] % n_bufs].synchronize()  # the gather of two steps ago has read this buffer
        rc = L.pco_b200_compress_ex(C.c_void_p(nums.data_ptr()), C.c_size_t(n), C.c_ubyte(2), C.byref(cfg), C.c_int(0), C.c_void_p(d_comp.data_ptr()),
                                    C.c_size_t(cap), C.byref(n_written), C.c_void_p(d_index.data_ptr()), C.c_size_t(icap), C.byref(ilen),
                                    C.c_uint32(SRC | DST | IDX), sp)
        _lib.check(rc)

    def decompress_resident():
        rc = L.pco_b200_decompress_ex(C.c_void_p(d_comp.data_ptr()), n_written, C.c_ubyte(2), C.c_void_p(d_out.data_ptr()), C.c_size_t(n), C.byref(prog),
                                      C.c_void_p(d_index.data_ptr()), ilen, C.c_uint32(SRC | DST | IDX), sp)
        _lib.check(rc)
        assert prog.n_processed == n and prog.finished

    # ---- the exchange step of the sharded path (SURVEY.md 8e): rank r holds chunks r, r + N, r + 2N, ... of the logical file.
    # Default: the GPUs gather the pages themselves (pcodec_b200/csrc/gather_kernels.cuh) - per-chunk sizes are all-gathered as a
    # device tensor (NCCL, no host copy), a scan kernel turns them into file offsets and a copy kernel stores this rank's chunks into
    # EVERY rank's file buffer over NVLink.  The gather of step k runs on a side stream beside decompress(k) and compress(k + 1).
    # --no-gather-pages: only the per-rank compressed sizes are exchanged (a sharded writer's file offsets), pages stay sharded.
    push_done = [None, None]
    gather_events = []
    # the gather's few CTAs must not queue behind the 1024-CTA grids of the step it overlaps: high priority
    side = torch.cuda.Stream(device=dev, priority=-1) if world > 1 else None
    gather_ctas = args.gather_ctas if args.gather_ctas > 0 else min(16 * world, 64)
    pg = None
    sizes_dev = all_sizes_dev = file_len_dev = None
    first_chunk_off = [0]
    if gather_on:
        from pcodec_b200 import sharded

        file_cap = L.pco_standalone_guarantee_file_size(world * n, 2) + 64
        pg = sharded.DevicePageGather(file_cap, world, rank)
        sizes_dev = torch.zeros(n_chunks, dtype=torch.int64, device=dev)
        all_sizes_dev = torch.zeros(world * n_chunks, dtype=torch.int64, device=dev)
        file_len_dev = torch.zeros(1, dtype=torch.int64, device=dev)

    def gather_pages():
        if world == 1:
            return
        import torch.distributed as dist

        k = step_no[0]
        step_no[0] += 1
        side.wait_stream(stream)
        with torch.cuda.stream(side):
            if gather_on:
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record(side)
                pg.chunk_sizes(d_index.data_ptr(), ilen.value, sizes_dev.data_ptr(), n_chunks, side.cuda_stream)
                dist.all_gather_into_tensor(all_sizes_dev, sizes_dev)
                pg.gather(d_comp.data_ptr() + first_chunk_off[0], all_sizes_dev.data_ptr(), n_chunks, world * n, file_len_dev.data_ptr(), side.cuda_stream,
                          max_ctas=gather_ctas)
                g1.record(side)
                push_done[k % n_bufs] = g1
                gather_events.append((g0, g1))
            else:
                sizes = torch.zeros(world, dtype=torch.int64, device=dev)
                dist.all_gather_into_tensor(sizes, torch.tensor([n_written.value], dtype=torch.int64, device=dev))

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also verifies the bit-exact round trip)
    L.pco_b200_profile_enable(1)
    if gather_on:  # where the first chunk starts in a rank's own file (behind its standalone header): constant for this workload
        import struct as _st

        compress_resident()
        ih0 = bytes(d_index[:64].cpu().numpy())
        first_chunk_off[0] = _st.unpack_from("<Q", bytes(d_index[_st.unpack_from("<Q", ih0, 32)[0]:_st.unpack_from("<Q", ih0, 32)[0] + 8].cpu().numpy()), 0)[0]
    for w in range(max(args.warmup, 3)):
        compress_resident()
        gather_pages()
        decompress_resident()
    torch.cuda.synchronize()
    assert torch.equal(d_out, nums), "GPU round trip is not bit-exact"
    Cbytes, Ibytes = n_written.value, ilen.value
    gather_info = None
    if gather_on:
        import torch.distributed as dist

        pg.wait(side.cuda_stream)
        dist.barrier()
        torch.cuda.synchronize()
        flen = int(file_len_dev.item())
        ft = pg.file_tensor()
        # every rank holds the same file (checksum of 8-byte words all-gathered), its own first and last chunk sit at their offsets
        words = ft[: flen // 8 * 8].view(torch.int64)
        chk = torch.stack([words.sum(), words[::7].sum(), torch.tensor(flen, device=dev)])
        allchk = torch.zeros(world * 3, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allchk, chk)
        assert bool((allchk.view(world, 3) == chk).all()), "the ranks' gathered files differ"
        hdr = bytes(ft[:4].cpu().numpy())
        assert hdr == b"pco!" and int(ft[flen - 1].item()) == 0, "gathered file: header / terminator"
        own_sizes = all_sizes_dev.view(world, n_chunks)
        off0 = 4 + 1 + 1 + (6 + (world * n).bit_length() + 7) // 8 + 2 + int(own_sizes[:rank, 0].sum().item())
        sz0 = int(own_sizes[rank, 0].item())
        assert torch.equal(ft[off0:off0 + sz0], d_comp[first_chunk_off[0]:first_chunk_off[0] + sz0]), "gathered file: this rank's first chunk is not where it belongs"
        gather_info = {"file_bytes": flen, "nvlink_bytes_out_per_gpu": int((world - 1) * (Cbytes - first_chunk_off[0] - 1)), "checked": "all ranks hold the same file (checksums), own chunk at its offset"}
    # byte parity of the measured file with the oracle on a sample of its chunks (outside every timed region): the bytes of
    # chunk c in the GPU's file must be the oracle's chunk bytes for the same numbers and ChunkConfig
    import struct

    def index_chunks(d_index, file_len):
        """(chunk count, the index's 32-byte chunk records, every chunk's start offset in the file followed by the terminator's)."""
        ih = bytes(d_index[:64].cpu().numpy())
        n_idx_chunks, chunks_off = struct.unpack_from("<Q", ih, 8)[0], struct.unpack_from("<Q", ih, 32)[0]
        recs = bytes(d_index[chunks_off:chunks_off + 32 * n_idx_chunks].cpu().numpy())
        return n_idx_chunks, recs, [struct.unpack_from("<Q", recs, 32 * i)[0] for i in range(n_idx_chunks)] + [file_len - 1]  # the terminator byte ends the file

    n_idx_chunks, recs, chunk_offs = index_chunks(d_index, Cbytes)
    parity = {"checked_chunks": 0, "against": "oracle/ (C++ restatement of pco 1.0.3), same numbers and ChunkConfig"}
    try:
        from oracle import pyoracle

        ocfg = pyoracle.make_config(level=8, mode=pyoracle.MODE_CLASSIC, delta=pyoracle.DELTA_CONSECUTIVE, delta_order=1)
        sample = sorted({0, 1, n_chunks // 3, n_chunks // 2, n_chunks - 2, n_chunks - 1} & set(range(n_chunks)))
        for c in sample:
            want = pyoracle.simple_compress(h_np[c * CHUNK_N:(c + 1) * CHUNK_N], ocfg)
            hdr_len = 12  # standalone header of a 2^18-number file (SURVEY.md Appendix A KAT 1); the chunk follows, then the terminator
            got = bytes(d_comp[chunk_offs[c]:chunk_offs[c + 1]].cpu().numpy())
            assert got == want[hdr_len:-1], f"chunk {c}: GPU bytes differ from the oracle's"
            parity["checked_chunks"] += 1
        parity["chunks"] = sample
    except ImportError as ex:  # the checker is test infrastructure: its absence is reported, not fatal
        parity["error"] = str(ex)

    # ---- timed region: resident
    sampler = ClockSampler(local_rank)
    if rank == 0:  # only rank 0's samples go into the line; N nvidia-smi pollers would only add host noise
        sampler.start()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    t_c, t_d, t_g, prof_c, prof_d = [], [], [], [], []
    gather_events.clear()
    barrier()
    ev_all0, ev_all1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev_all0.record(stream)
    for ev in evs:
        # no device-wide synchronisation inside the timed region: the page gather of step k (side stream) runs beside decompress(k) AND
        # compress(k + 1); the library calls synchronise their own stream, the per-step spans are read after the closing barrier
        ev[0].record(stream)
        compress_resident()
        ev[1].record(stream)
        prof_c.append(parse_profile(L))
        gather_pages()
        ev[2].record(stream)
        decompress_resident()
        ev[3].record(stream)
        prof_d.append(parse_profile(L))
    if side is not None:
        stream.wait_stream(side)  # the last step's gather belongs to the timed region
    ev_all1.record(stream)
    barrier()
    for ev in evs:
        t_c.append(ev[0].elapsed_time(ev[1]))
        t_g.append(ev[1].elapsed_time(ev[2]))
        t_d.append(ev[2].elapsed_time(ev[3]))
    total_ms = ev_all0.elapsed_time(ev_all1)
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / max(args.steps, 1)
    if args.dump_outputs and rank == 0:  # before the index-free leg below decodes into d_out again
        dump_outputs(args.dump_outputs, d_out, d_comp, n_written.value, d_index, ilen.value, index_chunks(d_index, n_written.value)[2])
    if gather_on and gather_info is not None:
        gather_info["device_ms"] = float(np.mean([a.elapsed_time(b) for a, b in gather_events])) if gather_events else None
        gather_info["ctas"] = gather_ctas
        gather_info["what"] = "sizes all-gather + scan + copy kernel on a high-priority side stream (overlaps decompress of the same step and compress of the next)"
    value = world * U / 1e6 / (ms_per_step / 1e3)

    # ---- the index-free path (not part of `value`): the same chunks decoded from their byte offsets alone
    # (pco_b200_decompress_chunks: one tANS walk per chunk builds the per-batch index on the device, all chunks in parallel)
    chunks_free = None
    if hasattr(L, "pco_b200_decompress_chunks") and not args.no_index_free:
        offs = np.array(chunk_offs[:n_idx_chunks], dtype=np.uint64)
        cns = np.array([struct.unpack_from("<I", recs, 32 * i + 8)[0] for i in range(n_idx_chunks)], dtype=np.uint32)
        nw_free = C.c_size_t()

        def decompress_chunks():
            rc = L.pco_b200_decompress_chunks(C.c_void_p(d_comp.data_ptr()), n_written, C.c_ubyte(2), offs.ctypes.data_as(C.c_void_p), cns.ctypes.data_as(C.c_void_p),
                                              C.c_size_t(n_idx_chunks), C.c_void_p(d_out.data_ptr()), C.c_size_t(n), C.byref(nw_free), C.c_uint32(SRC | DST), sp)
            _lib.check(rc)

        d_out.zero_()
        decompress_chunks()
        torch.cuda.synchronize()
        assert nw_free.value == n and torch.equal(d_out, nums), "index-free decompress is not bit-exact"
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(3):
            decompress_chunks()
        f1.record(stream)
        torch.cuda.synchronize()
        free_ms = f0.elapsed_time(f1) / 3
        chunks_free = {"decompress_mb_s": U / 1e6 / (free_ms / 1e3), "ms": free_ms, "kernel_ms": parse_profile(L),
                       "api": "pco_b200_decompress_chunks (chunk byte offsets only, no side index), buffers resident in HBM",
                       "roofline": {"bound": "hbm", "achieved": (U + Cbytes) / 1e9 / (free_ms / 1e3), "unit": "GB/s", "algorithmic_bytes": U + Cbytes,
                                    "basis": "the whole call (walk + decode), U + C"}}

    # ---- e2e: the same calls with pinned host buffers (H2D / D2H inside the timed region)
    e2e = None
    e2e_ok = 0 if args.no_e2e else 1
    if e2e_ok and not pinned_ok:
        e2e_ok = 0
        e2e = {"value": None, "unit": "MB/s", "error": "pinned host buffers: the input staging buffer could not be pinned"}
        if world > 1:  # the other ranks' collective below needs every rank
            import torch.distributed as dist

            dist.all_reduce(torch.tensor([0], dtype=torch.int64, device=dev), op=dist.ReduceOp.MIN)
    if e2e_ok:
        # the pinned staging buffers (2 x U + compressed + index per rank) can fail on a crowded host: every rank then
        # skips the e2e leg together instead of losing the whole line (the collectives below need all ranks)
        G = max(1, min(args.e2e_groups, n_chunks))
        bounds = [n_chunks * g // G for g in range(G + 1)]
        g_n = [(bounds[g + 1] - bounds[g]) * CHUNK_N for g in range(G)]
        g_cap = [L.pco_standalone_guarantee_file_size(g_n[g], 2) for g in range(G)]
        g_icap = [L.pco_b200_index_size_bound(g_n[g], bounds[g + 1] - bounds[g]) for g in range(G)]
        g_coff = np.concatenate([[0], np.cumsum(g_cap)]).astype(np.int64)
        g_ioff = np.concatenate([[0], np.cumsum([(x + 63) // 64 * 64 for x in g_icap])]).astype(np.int64)
        try:
            h_comp = torch.empty(max(cap, int(g_coff[-1])), dtype=torch.uint8, pin_memory=True)  # whole-file and per-group layouts share it
            h_index = torch.empty(max(icap, int(g_ioff[-1])), dtype=torch.uint8, pin_memory=True)
            h_out = torch.empty(n, dtype=torch.int64, pin_memory=True)
        except Exception as ex:  # noqa: BLE001
            e2e_ok = 0
            e2e = {"value": None, "unit": "MB/s", "error": f"pinned host buffers: {ex}"}
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([e2e_ok], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            if int(t.item()) == 0 and e2e_ok:
                e2e = {"value": None, "unit": "MB/s", "error": "pinned host buffers failed on another rank"}
            e2e_ok = int(t.item())
    if e2e_ok:
        nw2, il2 = C.c_size_t(), C.c_size_t()
        L.pco_b200_profile_enable(0)  # the per-kernel spans above are done; the e2e legs run without the profiler's events

        def e2e_single_call():
            rc = L.pco_b200_compress_ex(C.c_void_p(h_nums.data_ptr()), C.c_size_t(n), C.c_ubyte(2), C.byref(cfg), C.c_int(0), C.c_void_p(h_comp.data_ptr()),
                                        C.c_size_t(cap), C.byref(nw2), C.c_void_p(h_index.data_ptr()), C.c_size_t(icap), C.byref(il2), C.c_uint32(0), sp)
            _lib.check(rc)
            rc = L.pco_b200_decompress_ex(C.c_void_p(h_comp.data_ptr()), nw2, C.c_ubyte(2), C.c_void_p(h_out.data_ptr()), C.c_size_t(n), C.byref(prog),
                                          C.c_void_p(h_index.data_ptr()), il2, C.c_uint32(0), sp)
            _lib.check(rc)

        # The streaming use of the same two calls: the array goes through in groups of chunks, one host thread compresses group
        # g + 1 (H2D of its numbers dominates) while another decompresses group g (D2H of its numbers dominates), each on its own
        # stream with its own per-thread library context - both PCIe directions are busy.  Every group is a standalone file.
        h_comp_g, h_index_g = h_comp, h_index
        g_nw = [C.c_size_t() for _ in range(G)]
        g_il = [C.c_size_t() for _ in range(G)]
        import queue

        # two persistent worker threads (the library keeps its scratch per calling thread: a worker that lived for one pass would allocate
        # all of it again on every pass)
        class _Worker(threading.Thread):
            def __init__(self, fn):
                super().__init__(daemon=True)
                self.fn, self.jobs, self.done = fn, queue.Queue(), queue.Queue()
                self.start()

            def run(self):
                torch.cuda.set_device(local_rank)
                while True:
                    job = self.jobs.get()
                    if job is None:
                        L.pco_b200_thread_release()
                        return
                    try:
                        self.fn(job)
                        self.done.put(None)
                    except Exception as ex:  # noqa: BLE001
                        self.done.put(ex)

        P = max(1, min(args.e2e_threads, G))  # host threads per direction: producer p compresses groups p, p + P, ..., consumer p decompresses them
        streams = [torch.cuda.Stream(device=dev) for _ in range(2 * P)]
        handoffs = [queue.Queue() for _ in range(P)]
        trace = []  # (call, group, start, end) of the last streamed pass: shows how far the two directions overlap

        def make_produce(p):
            def produce(_):
                try:
                    sa = C.c_void_p(streams[p].cuda_stream)
                    for g in range(p, G, P):
                        t_a = time.perf_counter()
                        rc = L.pco_b200_compress_ex(C.c_void_p(h_nums.data_ptr() + 8 * bounds[g] * CHUNK_N), C.c_size_t(g_n[g]), C.c_ubyte(2), C.byref(cfg), C.c_int(0),
                                                    C.c_void_p(h_comp_g.data_ptr() + int(g_coff[g])), C.c_size_t(g_cap[g]), C.byref(g_nw[g]),
                                                    C.c_void_p(h_index_g.data_ptr() + int(g_ioff[g])), C.c_size_t(g_icap[g]), C.byref(g_il[g]), C.c_uint32(0), sa)
                        _lib.check(rc)
                        trace.append(("c", g, t_a, time.perf_counter()))
                        handoffs[p].put(g)
                finally:
                    handoffs[p].put(None)

            return produce

        def make_consume(p):
            def consume(_):
                sb = C.c_void_p(streams[P + p].cuda_stream)
                pr = _lib._CProgress()
                while True:
                    g = handoffs[p].get()
                    if g is None:
                        return
                    t_b = time.perf_counter()
                    rc = L.pco_b200_decompress_ex(C.c_void_p(h_comp_g.data_ptr() + int(g_coff[g])), g_nw[g], C.c_ubyte(2),
                                                  C.c_void_p(h_out.data_ptr() + 8 * bounds[g] * CHUNK_N), C.c_size_t(g_n[g]), C.byref(pr),
                                                  C.c_void_p(h_index_g.data_ptr() + int(g_ioff[g])), g_il[g], C.c_uint32(0), sb)
                    _lib.check(rc)
                    trace.append(("d", g, t_b, time.perf_counter()))
                    assert pr.n_processed == g_n[g] and pr.finished

            return consume

        workers = [_Worker(make_produce(p)) for p in range(P)] + [_Worker(make_consume(p)) for p in range(P)]

        def e2e_pipelined():
            trace.clear()
            for w in workers:
                w.jobs.put(1)
            errs = [w.done.get() for w in workers]
            for ex in errs:
                if ex is not None:
                    raise ex

        pass_wall = []  # host wall clock of every timed pass (ms)

        def timed(fn, reps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                t_p = time.perf_counter()
                fn()  # every call returns with its results in host memory (the library synchronises its stream)
                stream.synchronize()
                pass_wall.append(round((time.perf_counter() - t_p) * 1e3, 2))
            e1.record(stream)
            barrier()
            ms = e0.elapsed_time(e1) / reps
            if world > 1:
                import torch.distributed as dist

                t = torch.tensor([ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return ms

        e2e_single_call()
        assert torch.equal(h_out, h_nums), "e2e round trip is not bit-exact"
        h_out.zero_()
        e2e_pipelined()
        assert torch.equal(h_out, h_nums), "pipelined e2e round trip is not bit-exact"
        e2e_pipelined()  # second warm-up: both threads' contexts have their scratch
        e2e_ms = timed(e2e_pipelined, max(1, args.steps))
        streamed_wall = list(pass_wall)
        single_ms = timed(e2e_single_call, max(1, min(args.steps, 3)))
        t_first = min(t[2] for t in trace) if trace else 0.0
        e2e_trace = [[t[0], t[1], round((t[2] - t_first) * 1e3, 2), round((t[3] - t_first) * 1e3, 2)] for t in sorted(trace, key=lambda t: t[2])]
        for w in workers:
            w.jobs.put(None)
        for w in workers:
            w.join(timeout=30)
        cg, ig = sum(x.value for x in g_nw), sum(x.value for x in g_il)
        e2e = {"value": world * U / 1e6 / (e2e_ms / 1e3), "unit": "MB/s", "h2d_bytes_per_step": int(U + cg + ig),
               "d2h_bytes_per_step": int(cg + ig + U), "ms_per_step": e2e_ms, "steps": max(1, args.steps),
               "api": f"pco_b200_compress_ex + pco_b200_decompress_ex (C-ABI), pinned host buffers, streamed in {G} groups of chunks by {P} + {P} host threads: "
                      "compress of later groups runs beside decompress of earlier ones (per-thread library contexts, one stream each; every group is a standalone file; "
                      "big copies of one direction take turns, 32 MB slices)",
               "trace_ms": e2e_trace, "pass_wall_ms": streamed_wall,
               "single_call": {"value": world * U / 1e6 / (single_ms / 1e3), "ms_per_step": single_ms,
                               "api": "one pco_b200_compress_ex + one pco_b200_decompress_ex over the whole array (H2D, kernels, D2H back to back)"}}
    # ---- the reference's own three-function C ABI, unmodified (pco_c/include/cpcodec_generated.h:33-64): default config (Auto mode, Auto
    # delta, resolved per chunk), host buffers, no side index and no chunk offsets - the decompressor has to find every chunk boundary by
    # walking the stream (chunk lengths are not in the format), one chunk after the other.  A bounded sample of the workload.
    abi3 = None
    if not args.no_e2e and rank == 0:
        try:
            k3 = max(1, min(args.abi3_chunks, n_chunks))
            n3 = k3 * CHUNK_N
            src3 = h_np[:n3]
            cap3 = L.pco_standalone_guarantee_file_size(n3, 2)
            dst3 = np.empty(cap3, dtype=np.uint8)
            out3 = np.empty(n3, dtype=np.uint64)
            nw3, nd3 = C.c_size_t(), C.c_size_t()

            def abi3_step():
                rc = L.pco_standalone_simple_compress_into(src3.ctypes.data_as(C.c_void_p), C.c_size_t(n3), C.c_ubyte(2), None, dst3.ctypes.data_as(C.c_void_p), C.c_size_t(cap3), C.byref(nw3))
                assert rc == 0, f"pco_standalone_simple_compress_into: {rc}"
                t_mid = time.perf_counter()
                rc = L.pco_standalone_simple_decompress_into(dst3.ctypes.data_as(C.c_void_p), nw3, C.c_ubyte(2), out3.ctypes.data_as(C.c_void_p), C.c_size_t(n3), C.byref(nd3))
                assert rc == 0 and nd3.value == n3, f"pco_standalone_simple_decompress_into: {rc}"
                return t_mid

            abi3_step()
            assert np.array_equal(out3, src3), "3-function ABI round trip is not bit-exact"
            t0 = time.perf_counter()
            t_mid = abi3_step()
            t1 = time.perf_counter()
            abi3 = {"value": n3 * 8 / 1e6 / (t1 - t0), "unit": "MB/s", "compress_mb_s": n3 * 8 / 1e6 / (t_mid - t0), "decompress_mb_s": n3 * 8 / 1e6 / (t1 - t_mid),
                    "sample": f"{k3} chunks of 2^18 u64 in one standalone file, pageable host buffers, wall clock",
                    "api": "pco_standalone_simple_compress_into(config = NULL) + pco_standalone_simple_decompress_into: the reference's C ABI as is"}
        except Exception as ex:  # noqa: BLE001
            abi3 = {"value": None, "error": f"{type(ex).__name__}: {ex}"}
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=2)

    if rank != 0:
        return
    # ---- roofline of the decompress kernels: algorithmic bytes / CUDA-event duration
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    # the decompress path is two kernels: symwalk_kernel (tANS symbol walk) + decode_kernel (offsets, un-delta, join)
    dk_ms = float(np.mean([p.get("fused_narrow_kernel", 0.0) + p.get("decode_kernel", 0.0) + p.get("symwalk_kernel", 0.0) for p in prof_d]))
    dec_spans = {}
    for p in prof_d:
        for k, v in p.items():
            dec_spans.setdefault(k, []).append(v)
    dec_spans = {k: float(np.mean(v)) for k, v in dec_spans.items()}
    alg_bytes = U + Cbytes  # SURVEY.md 8(d): C read + U written; the side index (Ibytes more) is metadata, not algorithmic traffic
    achieved = alg_bytes / 1e9 / (dk_ms / 1e3) if dk_ms > 0 else None
    call_ms = float(np.mean(t_d))
    achieved_call = alg_bytes / 1e9 / (call_ms / 1e3)
    # DRAM traffic of the same two kernels from the committed `ncu --set full` capture (dram__bytes_read.sum +
    # dram__bytes_write.sum per launch, same workload); never measured under this run
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath) and n_chunks == N_CHUNKS:
        tj = json.load(open(tpath))
        traffic, traffic_src = int(sum(tj["dram_bytes_per_launch"].values())), tj["source"]
    comp_spans = {}
    for p in prof_c:
        for k, v in p.items():
            comp_spans.setdefault(k, []).append(v)
    comp_spans = {k: float(np.mean(v)) for k, v in comp_spans.items()}

    cpu = None
    if not args.no_cpu_baseline and world == 1:  # the CPU arm beside the GPU number: rank 0 at N = 1 only
        threads = host_threads()
        try:  # a CPU-side failure must not cost the GPU line
            v = cpu_roundtrip(max(threads, args.cpu_sample_chunks), threads)
            one = cpu_roundtrip(4, 1)  # BASELINE.md section 2: one thread and all host cores in the same run
            cpu = {"value": v[0], "unit": "MB/s", "cores": threads, "kind": "port",
                   "sample": f"{v[4]} chunks of 2^18 u64 (same generator), one worker process per host thread; C++ restatement of pco 1.0.3 (oracle/), not the Rust crate",
                   "compress_mb_s": v[1], "decompress_mb_s": v[2],
                   "single_core": {"value": one[0], "compress_mb_s": one[1], "decompress_mb_s": one[2], "sample": f"{one[4]} chunks, one process"}}
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": "MB/s", "cores": threads, "kind": "port", "sample": "failed", "error": f"{type(ex).__name__}: {ex}"}

    line = {
        "metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": f"C2: {n_chunks} chunks x 2^18 u64 per GPU, classic mode, consecutive delta order 1, level 8 (cumsum of geometric(0.001)); "
                               "step = compress + decompress of every chunk, buffers resident in HBM",
                   "chunks_per_gpu": n_chunks, "chunk_n": CHUNK_N, "l2": "inputs (2 GiB per GPU) exceed the 126 MB L2",
                   "multi_gpu": (("independent chunk shards per rank (chunk c on rank c mod N); every step the compressed PAGES ARE GATHERED on the device: NCCL all-gather of the per-chunk "
                                  "sizes (device tensor), scan kernel, then each rank stores its chunks into every rank's file buffer over NVLink (P2P stores into cudaIpc-mapped peer memory) - "
                                  "all ranks end up with the whole standalone file; the gather of step k overlaps decompress(k) and compress(k+1)") if gather_on else
                                 "independent chunk shards per rank; one NCCL all-gather per step of the per-rank compressed sizes (file offsets of the shards); pages stay sharded") if world > 1 else "single GPU",
                   "side_index": "decompress uses the per-batch side index emitted by the compressor (bytes counted in the roofline)"},
        "compress_mb_s": world * U / 1e6 / (float(np.mean(t_c)) / 1e3), "decompress_mb_s": world * U / 1e6 / (float(np.mean(t_d)) / 1e3),
        "gather_ms": float(np.mean(t_g)), "gather": gather_info, "compressed_bytes_per_gpu": Cbytes, "index_bytes_per_gpu": Ibytes, "ratio": U / Cbytes,
        "kernel_ms": {**dec_spans, **comp_spans},
        "roofline": {"bound": "hbm", "kernel": "fused_narrow_kernel (tANS walk + offsets + un-delta + join of every chunk in one launch)", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": alg_bytes,
                     "kernel_ms": dk_ms, "peak_source": peak_src,
                     "call": {"ms": call_ms, "achieved": achieved_call, "frac": achieved_call / peak, "what": "the whole pco_b200_decompress_ex call (device buffers), same bytes"},
                     "compress": {"ms": float(np.mean(t_c)), "achieved": alg_bytes / 1e9 / (float(np.mean(t_c)) / 1e3), "frac": alg_bytes / 1e9 / (float(np.mean(t_c)) / 1e3) / peak,
                                  "what": "the whole pco_b200_compress_ex call: U read + C written"}},
        "parity": parity,
        "index_free_decompress": ({**chunks_free, "roofline": {**chunks_free["roofline"], "peak": peak, "frac": chunks_free["roofline"]["achieved"] / peak}} if chunks_free else None),
        "cpu_baseline": cpu, "e2e": ({**e2e, "reference_abi": abi3} if e2e else e2e), "clocks": sampler.summary(),
        # per step (profiles/r02_zz_launches.csv): compress = init_chunks, split_count, publish (flags readback), plan_solve, fallback, bin_lut,
        # ans_encode, layout, chunk_offsets, pack, header_footer, emit_index; decompress = fused_narrow_kernel + publish (statuses readback)
        "gpu_launches": 14 + (3 if gather_on else 0),  # + chunk_sizes_kernel, gather_offsets_kernel, push_pages_kernel of the page gather
    }
    print(json.dumps(line))
    if args.results_csv:
        # the same run in the reference bench tool's format (docs/benchmark_results/*.csv): seconds per pass over the whole job
        from pcodec_b200 import benchfmt

        benchfmt.merge_results_csv(args.results_csv, [dict(
            input=f"c2_u64_cumsum_geometric_{world * n_chunks}x2^18", codec=benchfmt.PcoCodec(level=8, delta=DeltaSpec.try_consecutive(1), mode=ModeSpec.classic()),
            compress_dt=float(np.mean(t_c)) / 1e3, decompress_dt=float(np.mean(t_d)) / 1e3, compressed_size=world * Cbytes, uncompressed_size=world * U)])


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    run_gpu_arm(args, rank, world)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
