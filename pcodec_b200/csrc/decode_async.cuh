// Device side of pco_b200_decompress_async (host_api.cu): what the synchronous path decides on the host - the standalone header, the
// side index's header, the per-chunk statuses - decided on the device, so that the call needs no readback between its kernels.
//   async_validate_kernel   the checks of parse_standalone_header and of the side index; opens or closes the gate (AsyncGate) that
//                           the decode kernels read in their prologue, and writes the result when it closes it;
//   fused_narrow_kernel, symwalk_kernel, decode_kernel<L, 1 / 2>   as on the synchronous path (every launch gated);
//   async_outcome_kernel    reduces the statuses and class bytes to the result.
#pragma once
#include "../../include/pco_b200.h"
#include "decode_kernels.cuh"

namespace pcob200 {

static_assert(sizeof(PcoB200AsyncResult) == 24, "PcoB200AsyncResult layout");
static_assert(sizeof(AsyncGate) == 32, "AsyncGate layout");

// parse_standalone_header (host_common.hpp) over the first `avail` (<= 32) bytes: the same checks in the same order, a device status
// instead of a message.
__device__ inline uint32_t parse_standalone_header_dev(const uint8_t* b, uint64_t avail, uint64_t file_len, uint32_t* uniform_type, uint32_t* format_major) {
  auto byte_at = [&](uint64_t i) -> uint32_t { return (i < file_len && i < avail) ? b[i] : 0u; };
  if (!(4 <= file_len && 4 <= avail)) return ST_INSUFFICIENT_DATA;
  if (b[0] != 112 || b[1] != 99 || b[2] != 111 || b[3] != 33) return ST_CORRUPTION;  // "pco!"
  uint64_t pos = 4;
  const uint32_t ver = byte_at(pos);
  uint32_t uniform = 0;
  if (ver >= 2) {
    pos += 1;
    if (ver >= 3) {
      const uint32_t t = byte_at(pos);
      pos += 1;
      if (t != 0) {
        if (!nt_valid(t)) return ST_CORRUPTION;
        uniform = t;
      }
    }
    // varint: 6 bits (power - 1), then `power` bits; only its length and its padding bits are checked
    const uint32_t power = 1 + (byte_at(pos) & 63);
    const uint32_t total_bits = 6 + power;
    const uint32_t nbytes = (total_bits + 7) / 8;
    if (pos + nbytes > file_len) return ST_INSUFFICIENT_DATA;
    const uint32_t pad = nbytes * 8 - total_bits;
    if (pad && (byte_at(pos + nbytes - 1) >> (8 - pad)) != 0) return ST_CORRUPTION;
    pos += nbytes;
  }
  if (pos > file_len) return ST_INSUFFICIENT_DATA;
  if (ver > 3) return ST_CORRUPTION;
  const uint32_t major = byte_at(pos);
  pos += 1;
  if (major >= 4) pos += 1;
  if (major > 4) return ST_CORRUPTION;
  if (pos > file_len) return ST_INSUFFICIENT_DATA;
  *uniform_type = uniform;
  *format_major = major;
  return ST_OK;
}

// status_to_error (host_common.hpp) without the message
__device__ __forceinline__ uint32_t status_to_error_code(uint32_t st) {
  switch (st) {
    case ST_OK: return PCO_B200_OK;
    case ST_INSUFFICIENT_DATA: return PCO_B200_INSUFFICIENT_DATA;
    case ST_INVALID_ARGUMENT: return PCO_B200_INVALID_ARGUMENT;
    case ST_UNSUPPORTED: return PCO_B200_UNSUPPORTED;
    default: return PCO_B200_CORRUPTION;
  }
}

// C(n, j) for n <= 256, j < MAX_ORDER: the product n (n - 1) ... (n - j + 1) stays below 2^48, so the division is exact and the value
// is the one ensure_device builds by Pascal additions.
__device__ __forceinline__ uint64_t binom_small(uint32_t n, uint32_t j) {
  uint64_t num = 1, den = 1;
  for (uint32_t i = 0; i < j; i++) {
    num *= uint64_t(n >= i ? n - i : 0);
    den *= i + 1;
  }
  return num / den;
}

// One CTA of 32 threads.  Writes the binomials decode_kernel reads (the workspace carries them, so that a captured graph depends on no
// buffer of the calling thread's context), then thread 0 decides the gate.
__global__ void __launch_bounds__(32) async_validate_kernel(const uint8_t* __restrict__ src, uint64_t src_len, uint32_t dtype, const uint8_t* __restrict__ index,
                                                            uint64_t index_len, uint64_t n_chunks, uint64_t n_total, AsyncGate* __restrict__ gate,
                                                            Binoms* __restrict__ binoms, PcoB200AsyncResult* __restrict__ result) {
  const uint32_t tid = threadIdx.x;
  for (uint32_t j = 0; j < MAX_ORDER; j++) binoms->lane8[tid][j] = binom_small(8 * tid, j);
  if (tid < MAX_ORDER) binoms->full[tid] = binom_small(256, tid);
  if (tid != 0) return;
  uint8_t head[32];
  const uint64_t avail = src_len < 32 ? src_len : 32;
  for (uint32_t i = 0; i < 32; i++) head[i] = i < avail ? src[i] : 0;
  uint32_t uniform = 0, major = 0;
  uint32_t st = parse_standalone_header_dev(head, avail, src_len, &uniform, &major);
  if (st == ST_OK && uniform != 0 && uniform != dtype) st = ST_CORRUPTION;  // every chunk's type byte would fail against it
  const IndexHeader ih = *reinterpret_cast<const IndexHeader*>(index);     // index_len >= sizeof(IndexHeader): checked at enqueue
  if (st == ST_OK) {
    // the host checks of decompress_fast, then the caller's declared shape
    if (ih.magic != INDEX_MAGIC || ih.version != 1 || ih.file_len != src_len || ih.chunks_offset > index_len ||
        ih.n_chunks > (index_len - ih.chunks_offset) / sizeof(IndexChunk) || ih.n_chunks > 0xffffffffull)
      st = ST_INVALID_ARGUMENT;
    else if (ih.n_chunks != n_chunks || ih.n_total != n_total || ih.chunks_offset != sizeof(IndexHeader))
      st = ST_INVALID_ARGUMENT;
  }
  AsyncGate g;
  g.open = st == ST_OK ? 1u : 0u;
  g.uniform_type = uniform;
  g.format_major = major;
  g.finished = ih.end_byte != 0 ? 1u : 0u;
  g.n_total = n_total;
  g.reserved = 0;
  *gate = g;
  if (st != ST_OK) {
    PcoB200AsyncResult r;
    r.status = status_to_error_code(st);
    r.first_bad_chunk = 0xffffffffu;
    r.n_total = 0;
    r.finished = 0;
    r.reserved = 0;
    *result = r;
  }
}

constexpr int OUTCOME_THREADS = 1024;

// The synchronous path reports the first failing chunk among those fused_narrow_kernel finished and only then runs the general pair,
// whose failures it reports next; the lowest index of the first group, else of the second, is the same answer.
__global__ void __launch_bounds__(OUTCOME_THREADS) async_outcome_kernel(const uint32_t* __restrict__ gate, const uint32_t* __restrict__ statuses,
                                                                        const uint8_t* __restrict__ d_cls, uint32_t n_chunks,
                                                                        PcoB200AsyncResult* __restrict__ result) {
  const AsyncGate* g = reinterpret_cast<const AsyncGate*>(gate);
  if (g->open == 0) return;
  __shared__ uint32_t first_fused_bad, first_bad;
  if (threadIdx.x == 0) first_fused_bad = first_bad = 0xffffffffu;
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < n_chunks; i += OUTCOME_THREADS) {
    if (statuses[i] == ST_OK) continue;
    atomicMin(&first_bad, i);
    if (d_cls[i] & CLS_DONE) atomicMin(&first_fused_bad, i);
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  const uint32_t k = first_fused_bad != 0xffffffffu ? first_fused_bad : first_bad;
  PcoB200AsyncResult r;
  r.status = k == 0xffffffffu ? uint32_t(PCO_B200_OK) : status_to_error_code(statuses[k]);
  r.first_bad_chunk = k;
  r.n_total = g->n_total;
  r.finished = r.status == PCO_B200_OK ? g->finished : 0u;
  r.reserved = 0;
  *result = r;
}

}  // namespace pcob200
