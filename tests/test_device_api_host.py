"""CPU checks of the stream-ordered decompress ABI (pco_b200_decompress_async) and of pcodec.device's dtype mapping: the symbols are
exported, argument errors come back at enqueue without a device, and the workspace grows with the file."""
import ctypes as C

import pytest
import torch

from pcodec_b200 import _lib, device

INVALID_ARGUMENT, INVALID_TYPE, CUDA = 3, 5, 6
SYMBOLS = ("pco_b200_decompress_async", "pco_b200_decompress_async_workspace_size", "pco_b200_decompress_async_prepare")


def _L():
    return device._L()


def _call(src=0x1000, src_len=100, dtype=2, index=0x2000, index_len=64 + 32 * 4, n_chunks=4, n_total=1000, dst=0x3000, dst_len=1000,
          ws=0x4000, ws_len=None, result=0x5000):
    L = _L()
    if ws_len is None:
        ws_len = L.pco_b200_decompress_async_workspace_size(n_total, n_chunks, 2)
    return L.pco_b200_decompress_async(src, src_len, dtype, index, index_len, n_chunks, n_total, dst, dst_len, ws, ws_len, result, None)


def test_async_symbols_are_exported():
    L = _lib.lib()
    for s in SYMBOLS:
        assert hasattr(L, s), s
    assert C.sizeof(device._CAsyncResult) == 24


def test_without_a_device_the_calls_return_cuda():
    if _L().pco_b200_device_available():
        pytest.skip("a CUDA device is present")
    assert _call() == CUDA
    assert _L().pco_b200_decompress_async_prepare(2) == CUDA


@pytest.mark.parametrize("change, expect", [
    ({"src": None}, INVALID_ARGUMENT),
    ({"index": None}, INVALID_ARGUMENT),
    ({"dst": None}, INVALID_ARGUMENT),
    ({"ws": None}, INVALID_ARGUMENT),
    ({"result": None}, INVALID_ARGUMENT),
    ({"n_chunks": 0}, INVALID_ARGUMENT),
    ({"dst_len": 999}, INVALID_ARGUMENT),
    ({"index_len": 63}, INVALID_ARGUMENT),
    ({"index_len": 64 + 32 * 3}, INVALID_ARGUMENT),
    ({"index": 0x2004}, INVALID_ARGUMENT),
    ({"ws_len": 1024}, INVALID_ARGUMENT),
    ({"dtype": 0}, INVALID_TYPE),
    ({"dtype": 12}, INVALID_TYPE),
])
def test_enqueue_time_argument_errors(change, expect):
    """Caught on the host before any device work, so they are the same with or without a GPU (the pointers are never touched)."""
    kw = dict(change)
    if "ws_len" not in kw and "n_chunks" in kw:
        kw["ws_len"] = 1 << 30
    assert _call(**kw) == expect
    assert _L().pco_b200_last_error_message()


def test_workspace_too_small_by_one_byte():
    need = _L().pco_b200_decompress_async_workspace_size(1000, 4, 2)
    assert _call(ws_len=need - 1) == INVALID_ARGUMENT


def test_workspace_size_is_monotone():
    f = _L().pco_b200_decompress_async_workspace_size
    assert f(1000, 4, 99) == 0
    for dt in (2, 5, 10):
        prev = 0
        for n in (0, 1, 255, 256, 257, 1 << 18, (1 << 18) + 1, 1 << 28):
            row = [f(n, k, dt) for k in (1, 2, 7, 64, 1024, 1 << 20)]
            assert all(a <= b for a, b in zip(row, row[1:])), (n, row)
            assert row[0] >= prev
            prev = row[0]
    # the general pair's rows: about 2 bytes of symbols and 1/32 of offsets per number
    assert f(1 << 28, 1024, 2) >= 2 * (1 << 28)


@pytest.mark.parametrize("dtype, byte", [
    (torch.uint8, 10), (torch.int8, 11), (torch.int16, 8), (torch.uint16, 7), (torch.int32, 3), (torch.uint32, 1),
    (torch.int64, 4), (torch.uint64, 2), (torch.float16, 9), (torch.float32, 5), (torch.float64, 6),
])
def test_torch_dtype_mapping(dtype, byte):
    assert device.dtype_byte(dtype) == byte
    assert _lib.BYTE_TO_NP[byte].itemsize == torch.empty(0, dtype=dtype).element_size()


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.bool, torch.complex64, torch.complex128])
def test_dtypes_without_a_pco_type_are_rejected_before_device_work(dtype):
    t = torch.zeros(16, dtype=dtype)  # a host tensor: the dtype is refused before the device is even looked at
    with pytest.raises(TypeError):
        device.compress(t)
    with pytest.raises(TypeError):
        device.dtype_byte(dtype)
    with pytest.raises(TypeError):
        device.DeviceFile.from_bytes(b"pco!", dtype)


def test_compress_wants_a_cuda_tensor():
    with pytest.raises(ValueError):
        device.compress(torch.arange(10, dtype=torch.int64))


def test_pcodec_device_is_the_same_module():
    import pcodec.device

    assert pcodec.device.compress is device.compress and pcodec.device.decompress is device.decompress
