"""What stream-ordered decompress (pco_b200_decompress_async, pcodec.device) costs beside pco_b200_decompress_ex on the same device-resident
file: call time on the stream (CUDA events, the two alternated), per-kernel device time (torch.profiler, a run of its own), host time per
enqueue, and CUDA-graph replay time.  C2: 1024 x 2^18 u64 (datagen.c2_u64_torch, Classic, consecutive order 1: every chunk goes through the
fused kernel, the general pair only launches); C3: f64 decimal sinusoid (FloatMult 0.01, order 2: every chunk takes the general pair).

    python profiles/tools/async_decompress_probe.py --out async_probe.txt
"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from pcodec_b200 import ChunkConfig, DeltaSpec, ModeSpec, _lib, datagen, device  # noqa: E402


def gpu_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name()} (nvidia-smi: {e})"


class Case:
    def __init__(self, name, f):
        self.name, self.f = name, f
        self.L = _lib.lib()
        self.byte = device.dtype_byte(f.dtype)
        self.out = torch.empty(f.n, dtype=f.dtype, device="cuda")
        self.ws = torch.empty(device.workspace_bytes(f), dtype=torch.uint8, device="cuda")
        self.res = torch.zeros(24, dtype=torch.uint8, device="cuda")
        self.prog = _lib._CProgress()
        device.prepare(f)

    def sync_call(self):
        f = self.f
        rc = self.L.pco_b200_decompress_ex(C.c_void_p(f.data.data_ptr()), C.c_size_t(f.data.numel()), C.c_ubyte(self.byte), C.c_void_p(self.out.data_ptr()),
                                           C.c_size_t(f.n), C.byref(self.prog), C.c_void_p(f.index.data_ptr()), C.c_size_t(f.index.numel()), C.c_uint32(7),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream))
        _lib.check(rc)

    def async_call(self):
        f = self.f
        rc = self.L.pco_b200_decompress_async(f.data.data_ptr(), f.data.numel(), self.byte, f.index.data_ptr(), f.index.numel(), f.n_chunks, f.n,
                                              self.out.data_ptr(), f.n, self.ws.data_ptr(), self.ws.numel(), self.res.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream)
        _lib.check(rc)

    def async_ok(self):
        r = device._CAsyncResult.from_buffer_copy(self.res.cpu().numpy().tobytes())
        return r.status == 0 and r.n_total == self.f.n and r.finished == 1


def time_calls(fn, reps):
    """ms per call from CUDA events around `reps` back-to-back calls on the current stream (ends in a synchronise)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_times(fn, reps):
    """us per call of every kernel the calls launch (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.name.split("(")[0].split("<")[0].replace("void ", "").replace("pcob200::", "")
        out[name] = out.get(name, 0.0) + ev.device_time / reps
    return out


def host_enqueue_us(fn, reps):
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        a = time.perf_counter()
        fn()
        t.append((time.perf_counter() - a) * 1e6)
    torch.cuda.synchronize()
    return statistics.median(t), min(t)


def probe(case, lines, reps):
    f = case.f
    gb = f.n * torch.empty(0, dtype=f.dtype).element_size() / 1e9
    lines.append(f"== {case.name}: {f.n} numbers ({gb:.3f} GB), "
                 f"{f.n_chunks} chunks, file {f.data.numel() / 1e6:.1f} MB, workspace {case.ws.numel() / 1e6:.1f} MB")
    # outputs agree
    case.sync_call()
    torch.cuda.synchronize()
    ref = case.out.clone()
    case.out.zero_()
    case.async_call()
    torch.cuda.synchronize()
    assert case.async_ok() and torch.equal(case.out, ref), "async output differs from decompress_ex"
    for fn in (case.sync_call, case.async_call):  # warm-up
        time_calls(fn, 3)
    s_ms, a_ms = [], []
    for _ in range(5):  # alternated
        s_ms.append(time_calls(case.sync_call, reps))
        a_ms.append(time_calls(case.async_call, reps))
    lines.append(f"call time on the stream, ms per call (median of 5 x {reps}; min..max): decompress_ex {statistics.median(s_ms):.4f} "
                 f"({min(s_ms):.4f}..{max(s_ms):.4f})  decompress_async {statistics.median(a_ms):.4f} ({min(a_ms):.4f}..{max(a_ms):.4f})")
    # graph replay
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            case.async_call()
    torch.cuda.current_stream().wait_stream(s)
    case.out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert case.async_ok() and torch.equal(case.out, ref), "graph replay output differs"
    time_calls(g.replay, 3)
    r_ms = [time_calls(g.replay, reps) for _ in range(5)]
    a2 = [time_calls(case.async_call, reps) for _ in range(5)]
    lines.append(f"graph replay, ms per replay (median of 5 x {reps}): {statistics.median(r_ms):.4f} ({min(r_ms):.4f}..{max(r_ms):.4f}); "
                 f"eager decompress_async in the same window {statistics.median(a2):.4f}")
    # host time per enqueue (stream kept busy by a sleep so no call waits on a full launch queue)
    torch.cuda._sleep(int(1e8))
    med, lo = host_enqueue_us(case.async_call, 50)
    lines.append(f"host time per pco_b200_decompress_async enqueue: median {med:.1f} us, min {lo:.1f} us (ctypes call, 6 launches)")
    torch.cuda._sleep(int(1e8))
    med2, lo2 = host_enqueue_us(lambda: device.decompress(f, case.out, case.ws), 50)
    lines.append(f"host time per pcodec.device.decompress (prepare + result buffer + event): median {med2:.1f} us, min {lo2:.1f} us")
    med3, lo3 = host_enqueue_us(case.sync_call, 20)
    lines.append(f"host time per pco_b200_decompress_ex (returns after the work): median {med3:.1f} us, min {lo3:.1f} us")
    # per-kernel device time
    for label, fn in (("decompress_ex", case.sync_call), ("decompress_async", case.async_call)):
        kt = kernel_times(fn, reps)
        lines.append(f"kernels of {label}, us per call: " + ", ".join(f"{k} {v:.1f}" for k, v in sorted(kt.items(), key=lambda kv: -kv[1])))
        if label == "decompress_async":
            fused = sum(v for k, v in kt.items() if k.startswith("fused_narrow_kernel"))
            pair = sum(v for k, v in kt.items() if k.startswith(("symwalk_kernel", "decode_kernel")))
            extra = sum(v for k, v in kt.items() if k.startswith(("async_validate_kernel", "async_outcome_kernel")))
            lines.append(f"general pair (symwalk + decode<1> + decode<2>) {pair:.1f} us = {100 * pair / max(fused, 1e-9):.2f} % of the fused kernel's {fused:.1f} us; "
                         f"validate + outcome {extra:.1f} us")
    torch.cuda.synchronize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--chunks", type=int, default=1024)
    ap.add_argument("--c3-chunks", type=int, default=256)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    torch.cuda.init()
    lines = [f"GPU: {gpu_line()}  torch {torch.__version__}"]
    t = datagen.c2_u64_torch(args.chunks).view(torch.uint64)
    cfg = ChunkConfig(compression_level=8, mode_spec=ModeSpec.classic(), delta_spec=DeltaSpec.try_consecutive(1))
    f = device.compress(t, cfg)
    del t
    probe(Case(f"C2 u64, {args.chunks} x 2^18, Classic order 1", f), lines, args.reps)
    del f
    torch.cuda.empty_cache()
    x = torch.from_numpy(datagen.c3_f64_decimal_sinusoid(args.c3_chunks * datagen.CHUNK_N)).cuda()
    cfg3 = ChunkConfig(compression_level=8, mode_spec=ModeSpec.try_float_mult(0.01), delta_spec=DeltaSpec.try_consecutive(2))
    f3 = device.compress(x, cfg3)
    del x
    probe(Case(f"C3 f64, {args.c3_chunks} x 2^18, FloatMult 0.01 order 2", f3), lines, max(5, args.reps // 2))
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text)


if __name__ == "__main__":
    main()
