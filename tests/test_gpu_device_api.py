"""GPU tests of pcodec.device: compress a CUDA tensor into a device-resident file, decompress it with pco_b200_decompress_async on the
current stream (no host round trip), bit-exact against the original numbers, standalone.simple_compress and the oracle; the outcome of
broken files matches pco_b200_decompress_ex; the call does not wait for the device and replays from a CUDA graph."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TORCH_OF = {np.dtype(np.uint8): torch.uint8, np.dtype(np.int8): torch.int8, np.dtype(np.uint16): torch.uint16, np.dtype(np.int16): torch.int16,
            np.dtype(np.float16): torch.float16, np.dtype(np.uint32): torch.uint32, np.dtype(np.int32): torch.int32, np.dtype(np.float32): torch.float32,
            np.dtype(np.uint64): torch.uint64, np.dtype(np.int64): torch.int64, np.dtype(np.float64): torch.float64}
ALL_DTYPES = [np.uint8, np.int8, np.uint16, np.int16, np.float16, np.uint32, np.int32, np.float32, np.uint64, np.int64, np.float64]


def _signed(dt):
    return np.dtype(f"i{np.dtype(dt).itemsize}")


def to_dev(x, device="cuda"):
    x = np.ascontiguousarray(x)
    return torch.from_numpy(x.view(_signed(x.dtype)).copy()).to(device).view(TORCH_OF[x.dtype])


def to_host(t, np_dtype):
    return t.view(TORCH_OF[np.dtype(_signed(np_dtype))]).cpu().numpy().view(np_dtype)


def _walk(dtype, n, seed, scale=0.05):
    rng = np.random.default_rng(seed)
    if np.dtype(dtype).kind == "f":
        x = np.cumsum(rng.normal(size=n)).astype(dtype)
        if n > 5:
            x[3], x[4], x[5] = np.nan, -np.inf, -0.0
        return x
    steps = rng.geometric(scale, size=n).astype(np.int64) - int(1 / scale) // 2
    return np.cumsum(steps).astype(np.uint64).astype(np.dtype(dtype).str.replace("i", "u")).view(dtype)


def _cfgs(oracle, mode="classic", order=0, max_page_n=0, **kw):
    """Matching (product ChunkConfig, oracle config) pair."""
    from pcodec_b200 import ChunkConfig, DeltaSpec, ModeSpec, PagingSpec

    ms = {"classic": ModeSpec.classic(), "float_mult": ModeSpec.try_float_mult(kw.get("base", 0.01)), "int_mult": ModeSpec.try_int_mult(kw.get("ibase", 8)),
          "float_quant": ModeSpec.try_float_quant(kw.get("k", 13))}[mode]
    om = {"classic": oracle.MODE_CLASSIC, "float_mult": oracle.MODE_FLOAT_MULT, "int_mult": oracle.MODE_INT_MULT, "float_quant": oracle.MODE_FLOAT_QUANT}[mode]
    ours = ChunkConfig(mode_spec=ms, delta_spec=DeltaSpec.try_consecutive(order), paging_spec=PagingSpec.equal_pages_up_to(max_page_n or (1 << 18)), enable_8_bit=True)
    theirs = oracle.make_config(mode=om, delta=oracle.DELTA_CONSECUTIVE, delta_order=order, float_mult_base=kw.get("base", 0.01), int_mult_base=kw.get("ibase", 8),
                                float_quant_k=kw.get("k", 13), max_page_n=max_page_n)
    return ours, theirs


def sync_decompress(f, dst, src_len=None):
    """pco_b200_decompress_ex on the same device buffers: (error kind or None, last error message)."""
    from pcodec_b200 import _lib, device

    L = _lib.lib()
    prog = _lib._CProgress()
    rc = L.pco_b200_decompress_ex(C.c_void_p(f.data.data_ptr()), C.c_size_t(f.data.numel() if src_len is None else src_len), C.c_ubyte(device.dtype_byte(f.dtype)),
                                  C.c_void_p(dst.data_ptr()), C.c_size_t(dst.numel()), C.byref(prog), C.c_void_p(f.index.data_ptr()), C.c_size_t(f.index.numel()),
                                  C.c_uint32(7), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return (None if rc == 0 else _lib.ERROR_KINDS[rc]), L.pco_b200_last_error_message().decode()


def async_outcome(f, dst):
    from pcodec_b200 import PcoError, device

    _, st = device.decompress(f, dst)
    try:
        st.check()
        return None, st
    except PcoError as e:
        return e.kind, st


def _roundtrip(oracle, nums, mode, order, max_page_n, **kw):
    from pcodec_b200 import device, standalone

    ours_cfg, their_cfg = _cfgs(oracle, mode, order, max_page_n, **kw)
    t = to_dev(nums)
    f = device.compress(t, ours_cfg)
    assert f.n == nums.size and f.shape == nums.shape and f.dtype == t.dtype
    b = f.to_bytes()
    assert b == standalone.simple_compress(nums, ours_cfg)
    assert b == oracle.simple_compress(nums, their_cfg)
    out, st = device.decompress(f)
    st.check()
    assert st.n_total == nums.size and st.finished
    np.testing.assert_array_equal(to_host(out, nums.dtype).view(_signed(nums.dtype)), nums.view(_signed(nums.dtype)))


@pytest.mark.parametrize("dtype", ALL_DTYPES)
@pytest.mark.parametrize("order", [0, 1, 7])
def test_classic_round_trip(oracle, dtype, order):
    for n in (1, 257, 70001):
        _roundtrip(oracle, _walk(dtype, n, seed=n + order), "classic", order, 1 << 14)


@pytest.mark.parametrize("dtype", [np.uint16, np.int16, np.uint32, np.int32, np.uint64, np.int64])
def test_int_mult_round_trip(oracle, dtype):
    rng = np.random.default_rng(1)
    info = np.iinfo(dtype)
    nums = (rng.integers(0, min(info.max // 8, 1 << 20), size=30001) * 8 + 3).astype(dtype)
    _roundtrip(oracle, nums, "int_mult", 1, 1 << 13, ibase=8)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("mode", ["float_mult", "float_quant"])
def test_float_modes_round_trip(oracle, dtype, mode):
    n = 40001
    if mode == "float_mult":
        x = (np.round(1e5 * np.cos(2 * np.pi * np.arange(n) / (n / 103))) * 0.01).astype(dtype)
        x[5], x[6], x[7] = np.nan, np.inf, dtype(-0.0)
        _roundtrip(oracle, x, mode, 2, 1 << 13, base=0.01)
    else:
        x = np.random.default_rng(2).normal(size=n).astype(np.float16).astype(dtype)
        _roundtrip(oracle, x, mode, 0, 1 << 13, k=13 if dtype == np.float32 else 42)


@pytest.mark.parametrize("dtype", [np.uint64, np.float64, np.uint32])
def test_full_size_chunks(oracle, dtype):
    n = 2 * (1 << 18) + 3  # two chunks of 2^18 + 1 and 2^18 + 2 numbers (default paging)
    _roundtrip(oracle, _walk(dtype, n, seed=3), "classic", 1, 0)


def test_mixed_fused_and_general_chunks(oracle):
    """Narrow chunks (fused kernel) between wide ones (symwalk + decode_kernel): both launch unconditionally and each chunk is decoded
    once; the sync path's class counts show the file really mixes them."""
    from pcodec_b200 import _lib, device

    rng = np.random.default_rng(7)
    page = 1 << 14
    parts = [_walk(np.uint64, page, 1), rng.integers(0, 2**63, size=page, dtype=np.uint64) * 2 + 1, _walk(np.uint64, page, 2),
             rng.integers(0, 2**63, size=page + 11, dtype=np.uint64)]
    nums = np.concatenate(parts)
    _roundtrip(oracle, nums, "classic", 1, page)
    ours_cfg, _ = _cfgs(oracle, "classic", 1, page)
    f = device.compress(to_dev(nums), ours_cfg)
    dst = torch.empty(f.n, dtype=torch.uint64, device="cuda")
    assert sync_decompress(f, dst)[0] is None
    counts = (C.c_uint * 8)()
    assert _lib.lib().pco_b200_profile_chunk_classes(counts) == f.n_chunks
    assert counts[1] + counts[2] > 0 and counts[3] + counts[4] + counts[5] > 0, list(counts)
    # and a two-var file, where every chunk takes the general pair
    x = (np.round(1e5 * np.cos(2 * np.pi * np.arange(50000) / 400.0)) * 0.01)
    _roundtrip(oracle, x, "float_mult", 2, 1 << 13, base=0.01)


def _canary_out(f, extra=64):
    buf = torch.empty(f.n + extra, dtype=f.dtype, device="cuda")
    buf.view(torch.uint8).fill_(0x5A)
    return buf


def _assert_same_outcome(f, n):
    """Same kind (and failing chunk) from both paths, the same numbers in [0, n), an untouched canary behind dst.  The files are Classic
    u32, whose chunks all go through the fused kernel, so a failing file leaves the same numbers behind on both paths too."""
    a, b = _canary_out(f), _canary_out(f)
    canary = a[f.n:].clone()
    kind_async, st = async_outcome(f, a[:f.n])
    kind_sync, msg = sync_decompress(f, b[:n])
    assert torch.equal(a[f.n:], canary)
    if kind_async == "Unsupported":  # the sync path hands such chunks to the single-thread decoder, which this path does not have
        return kind_async
    assert kind_async == kind_sync, (kind_async, kind_sync, msg)
    if kind_async is not None and st.first_bad_chunk != 0xFFFFFFFF:
        m = re.search(r"chunk (\d+)", msg)
        assert m and int(m.group(1)) == st.first_bad_chunk, (msg, st.first_bad_chunk)
    assert torch.equal(a[:n].view(torch.uint8), b[:n].view(torch.uint8))
    return kind_async


@pytest.fixture(scope="module")
def u32_file(oracle):
    from pcodec_b200 import device

    nums = _walk(np.uint32, 20000, 4)
    ours_cfg, _ = _cfgs(oracle, "classic", 1, 4096)
    return nums, device.compress(to_dev(nums), ours_cfg)


def test_wrong_index_magic(u32_file):
    from pcodec_b200 import device

    _, f = u32_file
    idx = f.index.clone()
    idx[0] ^= 0xFF
    g = device.DeviceFile(f.data, idx, f.dtype, f.shape, f.n, f.n_chunks)
    assert _assert_same_outcome(g, f.n) == "InvalidArgument"


def test_declared_n_total_that_disagrees_with_the_index(u32_file):
    """The index says n numbers; a caller that declares n - 1 gets InvalidArgument and not a number written (the synchronous path,
    which reads n_total from the index itself, decodes the file)."""
    from pcodec_b200 import device

    _, f = u32_file
    g = device.DeviceFile(f.data, f.index, f.dtype, (f.n - 1,), f.n - 1, f.n_chunks)
    out = _canary_out(g)
    before = out.clone()
    kind, st = async_outcome(g, out[:g.n])
    assert kind == "InvalidArgument" and st.first_bad_chunk == 0xFFFFFFFF
    assert torch.equal(out, before)
    g = device.DeviceFile(f.data, f.index, f.dtype, f.shape, f.n, f.n_chunks + 1)
    with pytest.raises(device.PcoError):  # a chunk count the index does not have (here: one its table is too short for)
        device.decompress(g)[1].check()


def test_shortened_src_len(u32_file):
    from pcodec_b200 import device

    _, f = u32_file
    for cut in (1, 100):
        g = device.DeviceFile(f.data[:-cut], f.index, f.dtype, f.shape, f.n, f.n_chunks)
        assert _assert_same_outcome(g, f.n) == "InvalidArgument"
    g = device.DeviceFile(f.data[:3], f.index, f.dtype, f.shape, f.n, f.n_chunks)
    assert _assert_same_outcome(g, f.n) == "InsufficientData"  # the header itself is cut short


def _chunk_offsets(f):
    idx = f.index.cpu().numpy()
    return [int(idx[64 + 32 * c:72 + 32 * c].view(np.uint64)[0]) for c in range(f.n_chunks)]


def test_bit_flipped_chunks(u32_file):
    """Flips in the chunk headers (type byte, count, chunk meta: mostly caught) and in the chunk bodies (mostly decoded into other
    numbers, which must then be the synchronous path's numbers)."""
    from pcodec_b200 import device

    nums, f = u32_file
    data = f.data.cpu()
    rng = np.random.default_rng(0)
    heads = np.concatenate([np.arange(8 * o, 8 * (o + 24)) for o in _chunk_offsets(f)])
    bits = np.concatenate([rng.choice(heads, size=40, replace=False), rng.choice(np.arange(8 * 16, data.numel() * 8), size=40, replace=False)])
    kinds = []
    for bit in bits:
        d = data.clone()
        d[bit // 8] ^= 1 << (bit % 8)
        g = device.DeviceFile(d.cuda(), f.index, f.dtype, f.shape, f.n, f.n_chunks)
        kinds.append(_assert_same_outcome(g, f.n))
    assert set(kinds) - {None, "Unsupported"}, kinds  # some flips were caught


def test_decompress_does_not_wait_for_the_device(u32_file):
    from pcodec_b200 import device

    nums, f = u32_file
    device.prepare(f)
    stream = torch.cuda.current_stream()
    torch.cuda._sleep(int(2e8))  # ~0.1 s of spinning ahead of the decompress on the same stream
    out, st = device.decompress(f)
    assert not stream.query()
    st.check()
    np.testing.assert_array_equal(to_host(out, np.uint32), nums)


def test_cuda_graph_capture_and_replay(u32_file):
    from pcodec_b200 import PcoError, device

    nums, f = u32_file
    data = f.data.clone()
    g_file = device.DeviceFile(data, f.index, f.dtype, f.shape, f.n, f.n_chunks)
    pos = _chunk_offsets(f)[2]  # the type byte of chunk 2: a flip there is Corruption in chunk 2
    dst = torch.empty(f.n, dtype=f.dtype, device="cuda")
    bad = data.clone()
    bad[pos] ^= 0x24
    assert sync_decompress(device.DeviceFile(bad, f.index, f.dtype, f.shape, f.n, f.n_chunks), dst)[0] == "Corruption"
    device.prepare(g_file)
    out = torch.empty(f.n, dtype=f.dtype, device="cuda")
    ws = torch.empty(device.workspace_bytes(g_file), dtype=torch.uint8, device="cuda")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _, st = device.decompress(g_file, out, ws)
    graph.replay()
    st.check()
    np.testing.assert_array_equal(to_host(out, np.uint32), nums)
    orig = int(data[pos])
    data[pos] = orig ^ 0x24
    graph.replay()
    with pytest.raises(PcoError) as e:
        st.check()
    assert e.value.kind == "Corruption" and st.first_bad_chunk == 2
    data[pos] = orig
    out.zero_()
    graph.replay()
    st.check()
    np.testing.assert_array_equal(to_host(out, np.uint32), nums)


def test_two_streams_one_thread(oracle):
    from pcodec_b200 import device

    a, b = _walk(np.uint64, 300000, 11), _walk(np.float32, 200001, 12)
    fa = device.compress(to_dev(a), _cfgs(oracle, "classic", 1, 1 << 14)[0])
    fb = device.compress(to_dev(b), _cfgs(oracle, "classic", 0, 1 << 14)[0])
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream())
    s2.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s1):
        torch.cuda._sleep(int(5e7))
        oa, sa = device.decompress(fa)
    with torch.cuda.stream(s2):
        ob, sb = device.decompress(fb)
    sb.check()
    sa.check()
    np.testing.assert_array_equal(to_host(oa, np.uint64), a)
    np.testing.assert_array_equal(to_host(ob, np.float32).view(np.int32), b.view(np.int32))


def test_from_bytes_of_an_oracle_file(oracle):
    from pcodec_b200 import device

    nums = _walk(np.int64, 50001, 13)
    data = oracle.simple_compress(nums, oracle.make_config(mode=oracle.MODE_CLASSIC, delta=oracle.DELTA_CONSECUTIVE, delta_order=2, max_page_n=1 << 13))
    f = device.DeviceFile.from_bytes(data, torch.int64)
    assert f.n == nums.size and f.n_chunks == 7 and f.to_bytes() == data
    out, st = device.decompress(f)
    st.check()
    np.testing.assert_array_equal(out.cpu().numpy(), nums)


def test_second_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device")
    from pcodec_b200 import device

    nums = _walk(np.uint64, 100000, 14)
    t = to_dev(nums, "cuda:1")
    f = device.compress(t)
    assert f.device == torch.device("cuda:1") and f.index.device == torch.device("cuda:1")
    out, st = device.decompress(f)
    st.check()
    assert out.device == torch.device("cuda:1")
    np.testing.assert_array_equal(to_host(out, np.uint64), nums)


def test_empty_and_non_contiguous_tensors():
    from pcodec_b200 import device

    f = device.compress(torch.empty(0, dtype=torch.int32, device="cuda"))
    out, st = device.decompress(f)
    assert out.numel() == 0 and st.check().finished
    t = torch.arange(3000, dtype=torch.int64, device="cuda").reshape(30, 100).t()  # non-contiguous: copied once
    f = device.compress(t)
    out, st = device.decompress(f)
    st.check()
    assert out.shape == (100, 30) and torch.equal(out, t.contiguous())
