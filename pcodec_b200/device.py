"""Device-resident files for PyTorch: compress a CUDA tensor into a file in HBM, and decompress it back asynchronously on the current
stream, CUDA-graph capturable (pco_b200_compress_ex with every buffer on the device, pco_b200_decompress_async).

    f = device.compress(t)                  # synchronous: the file's size comes back to the host
    out, status = device.decompress(f)      # enqueued on torch.cuda.current_stream(); returns at once
    ...                                     # more work on the same stream and thread
    status.check()                          # waits, raises PcoError with the kind pco_b200_decompress_ex would give

Capture: call `prepare(f)` once outside the capture, preallocate `out` and `workspace` (`workspace_bytes(f)`), capture
`decompress(f, out, workspace)`, replay; `status.check()` after a replay reports that replay.  The file's bytes and index stay where
they were at capture time and may be rewritten in place between replays.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, standalone
from ._lib import ChunkConfig, PcoError  # noqa: F401

__all__ = ["DeviceFile", "AsyncStatus", "compress", "decompress", "prepare", "workspace_bytes", "dtype_byte", "TORCH_TO_BYTE", "PcoError"]

# torch dtype -> pco number type byte (pco_c/include/cpcodec.h:10-20).  bfloat16, bool and complex have no pco type.
TORCH_TO_BYTE = {
    torch.uint8: 10, torch.int8: 11, torch.int16: 8, torch.uint16: 7, torch.int32: 3, torch.uint32: 1,
    torch.int64: 4, torch.uint64: 2, torch.float16: 9, torch.float32: 5, torch.float64: 6,
}
SRC_ON_DEVICE, DST_ON_DEVICE, INDEX_ON_DEVICE = 1, 2, 4
_INDEX_HEADER_BYTES = 64  # IndexHeader: magic, version, n_chunks, n_total, file_len, chunks_offset, end_byte, reserved[2]


class _CAsyncResult(C.Structure):
    _fields_ = [("status", C.c_uint32), ("first_bad_chunk", C.c_uint32), ("n_total", C.c_uint64), ("finished", C.c_uint32),
                ("reserved", C.c_uint32)]


_RESULT_BYTES = C.sizeof(_CAsyncResult)
_ready = False


def _L():
    global _ready
    L = _lib.lib()
    if not _ready:
        L.pco_b200_decompress_async_workspace_size.restype = C.c_size_t
        L.pco_b200_decompress_async_workspace_size.argtypes = [C.c_size_t, C.c_size_t, C.c_ubyte]
        L.pco_b200_decompress_async_prepare.argtypes = [C.c_ubyte]
        L.pco_b200_decompress_async.argtypes = [C.c_void_p, C.c_size_t, C.c_ubyte, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t,
                                                C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        _ready = True
    return L


def dtype_byte(dtype):
    """The pco number type byte of a torch dtype; TypeError for dtypes pco has no type for (bfloat16, bool, complex, ...)."""
    if dtype not in TORCH_TO_BYTE:
        raise TypeError(f"pco has no number type for {dtype}")
    return TORCH_TO_BYTE[dtype]


def _index_header(index):
    """(n_chunks, n_total) from the first bytes of a side index (a uint8 tensor or bytes)."""
    if isinstance(index, torch.Tensor):
        head = index[:_INDEX_HEADER_BYTES].cpu().numpy().tobytes()
    else:
        head = bytes(index[:_INDEX_HEADER_BYTES])
    if len(head) < _INDEX_HEADER_BYTES:
        raise PcoError("InvalidArgument", "side index is shorter than its header")
    w = np.frombuffer(head, dtype=np.uint64)
    return int(w[1]), int(w[2])


class DeviceFile:
    """A standalone .pco file and its side index, both uint8 CUDA tensors on one device.  `data` holds exactly the file's bytes (the
    same as standalone.simple_compress writes for the same numbers and config); `n` numbers of `dtype` in `n_chunks` chunks, which
    decompress into a tensor of `shape`."""

    def __init__(self, data, index, dtype, shape, n, n_chunks):
        self.data, self.index, self.dtype, self.shape, self.n, self.n_chunks = data, index, dtype, tuple(shape), int(n), int(n_chunks)

    @property
    def device(self):
        return self.data.device

    @classmethod
    def from_bytes(cls, b, dtype, device=None):
        """A file written elsewhere (standalone.simple_compress, the reference's pco) moved to the device.  Its side index is built by
        pco_b200_build_index; a device dtype is a torch dtype."""
        np_dtype = _lib.BYTE_TO_NP[dtype_byte(dtype)]
        index = standalone.build_index(b, np_dtype)
        n_chunks, n_total = _index_header(index)
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        data = torch.frombuffer(bytearray(b), dtype=torch.uint8).to(dev) if len(b) else torch.empty(0, dtype=torch.uint8, device=dev)
        idx = torch.frombuffer(bytearray(index), dtype=torch.uint8).to(dev)
        return cls(data, idx, dtype, (n_total,), n_total, n_chunks)

    def to_bytes(self):
        """The file's bytes on the host, for standalone.simple_decompress, the reference or storage."""
        return self.data.cpu().numpy().tobytes()

    def __repr__(self):
        return f"DeviceFile(n={self.n}, dtype={self.dtype}, shape={self.shape}, n_chunks={self.n_chunks}, bytes={self.data.numel()}, device={self.device})"


def compress(t, config=None):
    """Compresses a CUDA tensor into a DeviceFile on the same device (pco_b200_compress_ex, every buffer in HBM, on
    torch.cuda.current_stream(t.device)).  Synchronous: it returns once the file is written, because the file's size comes back to
    the host.  A non-contiguous tensor is copied once.  `config` is a ChunkConfig (None: pco's default, as standalone.simple_compress)."""
    byte = dtype_byte(t.dtype)
    if not t.is_cuda:
        raise ValueError("device.compress takes a CUDA tensor; standalone.simple_compress takes host arrays")
    L = _L()
    shape = tuple(t.shape)
    t = t.contiguous()
    n = t.numel()
    cfg = (config or ChunkConfig())._to_c()
    cap = L.pco_standalone_guarantee_file_size(n, byte)
    icap = L.pco_b200_index_size_bound(n, max(n >> 8, 64))
    if cfg.paging_spec == 1 or (cfg.max_page_n and cfg.max_page_n < (1 << 18)):
        # the guarantee above assumes default paging; small pages add a per-chunk meta allowance (as standalone.simple_compress)
        n_pages = int(cfg.n_exact_pages) if cfg.paging_spec == 1 else -(-n // max(cfg.max_page_n, 1))
        cap += n_pages * 160
        icap += n_pages * 64
    with torch.cuda.device(t.device):
        stream = torch.cuda.current_stream(t.device)
        data = torch.empty(cap, dtype=torch.uint8, device=t.device)
        # an empty tensor's index is a bare header that the library writes from the host: give it a host buffer
        index = torch.empty(icap, dtype=torch.uint8, device=t.device if n else "cpu")
        flags = SRC_ON_DEVICE | DST_ON_DEVICE | (INDEX_ON_DEVICE if n else 0)
        n_written, ilen = C.c_size_t(), C.c_size_t()
        rc = L.pco_b200_compress_ex(C.c_void_p(t.data_ptr()), C.c_size_t(n), C.c_ubyte(byte), C.byref(cfg), C.c_int(0),
                                    C.c_void_p(data.data_ptr()), C.c_size_t(cap), C.byref(n_written), C.c_void_p(index.data_ptr()),
                                    C.c_size_t(icap), C.byref(ilen), C.c_uint32(flags), C.c_void_p(stream.cuda_stream))
        _lib.check(rc)
        data = data.narrow(0, 0, n_written.value)
        index = index.narrow(0, 0, ilen.value).to(t.device)
        n_chunks, n_total = _index_header(index)
    return DeviceFile(data, index, t.dtype, shape, n_total, n_chunks)


def workspace_bytes(f):
    """Bytes of scratch a decompress of `f` needs (pco_b200_decompress_async_workspace_size)."""
    return int(_L().pco_b200_decompress_async_workspace_size(f.n, f.n_chunks, dtype_byte(f.dtype)))


def prepare(f):
    """The calling thread's one-time set-up for decompressing `f`'s dtype on `f`'s device; call it before capturing a decompress."""
    with torch.cuda.device(f.device):
        _lib.check(_L().pco_b200_decompress_async_prepare(dtype_byte(f.dtype)))


class AsyncStatus:
    """What a decompress found, once the stream has reached it.  check() waits for it; after a graph replay it reports that replay."""

    def __init__(self, result, device, event, n):
        self._result, self._device, self._event, self._n = result, device, event, n
        self.status = self.first_bad_chunk = self.n_total = self.finished = None

    def check(self):
        """Waits for the decompress and raises PcoError (the kind pco_b200_decompress_ex gives for the same file) if it failed;
        returns self with `n_total` and `finished` filled in."""
        if self._result is None:  # an empty file: nothing was enqueued
            self.status, self.first_bad_chunk, self.n_total, self.finished = 0, 0xFFFFFFFF, self._n, True
            return self
        if self._event is not None:
            self._event.synchronize()
        else:  # captured: the replay ran on whichever stream replayed the graph
            torch.cuda.synchronize(self._device)
        r = _CAsyncResult.from_buffer_copy(self._result.cpu().numpy().tobytes())
        self.status, self.first_bad_chunk, self.n_total, self.finished = int(r.status), int(r.first_bad_chunk), int(r.n_total), bool(r.finished)
        if self.status != 0:
            kind = _lib.ERROR_KINDS.get(self.status, f"code {self.status}")
            where = f"chunk {self.first_bad_chunk}" if self.first_bad_chunk != 0xFFFFFFFF else "the file header or the side index"
            raise PcoError(kind, f"device decompress failed in {where}")
        return self

    def ok(self):
        try:
            self.check()
        except PcoError:
            return False
        return True


def decompress(f, out=None, workspace=None):
    """Decompresses a DeviceFile into `out` (allocated when None: f.shape, f.dtype, on f's device) without waiting for the device:
    every kernel is enqueued on torch.cuda.current_stream(f.device) and the call returns.  Returns (out, AsyncStatus).  `workspace`
    is a uint8 CUDA tensor of at least workspace_bytes(f) (allocated when None) that no other decompress uses at the same time.
    Capturable in a CUDA graph once prepare(f) has run on this thread."""
    byte = dtype_byte(f.dtype)
    dev = f.device
    L = _L()
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        if out is None:
            out = torch.empty(f.shape, dtype=f.dtype, device=dev)
        elif out.device != dev or out.dtype != f.dtype or not out.is_contiguous() or out.numel() < f.n:
            raise ValueError(f"out must be a contiguous {f.dtype} tensor of at least {f.n} numbers on {dev}")
        if f.n_chunks == 0:  # an empty file has no chunk to decode
            return out, AsyncStatus(None, dev, None, f.n)
        need = workspace_bytes(f)
        if workspace is None:
            workspace = torch.empty(need, dtype=torch.uint8, device=dev)
        elif workspace.device != dev or not workspace.is_contiguous() or workspace.numel() * workspace.element_size() < need:
            raise ValueError(f"workspace must be a contiguous CUDA tensor of at least {need} bytes on {dev}")
        result = torch.empty(_RESULT_BYTES, dtype=torch.uint8, device=dev)
        capturing = torch.cuda.is_current_stream_capturing()
        if not capturing:
            _lib.check(L.pco_b200_decompress_async_prepare(byte))
        rc = L.pco_b200_decompress_async(f.data.data_ptr(), f.data.numel(), byte, f.index.data_ptr(), f.index.numel(), f.n_chunks, f.n,
                                         out.data_ptr(), out.numel(), workspace.data_ptr(), workspace.numel() * workspace.element_size(),
                                         result.data_ptr(), stream.cuda_stream)
        _lib.check(rc)
        event = None
        if not capturing:
            # the caller may free any of these while the stream still reads them: the allocator must not reuse them before it has
            for buf in (f.data, f.index, out, workspace):
                buf.record_stream(stream)
            event = torch.cuda.Event()
            event.record(stream)
    return out, AsyncStatus(result, dev, event, f.n)
