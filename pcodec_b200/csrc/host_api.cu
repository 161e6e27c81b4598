// libcpcodec.so — C-ABI entry points (include/cpcodec.h, include/pco_b200.h) over the sm_100a kernels.
// There is no CPU implementation of the hot path in this library: without a CUDA device every
// compute entry point fails with PCO_B200_CUDA.
#include <algorithm>

#include "compress_host.cuh"
#include "decode_kernels.cuh"
#include "decode_narrow.cuh"
#include "decode_fused.cuh"
#include "gather_kernels.cuh"
#include "decode_cold.cuh"
#include "decode_async.cuh"
#include "host_common.hpp"

namespace pcob200 {

// One Context per host thread (thread_local): its scratch buffers, events and the last call's profile belong to the calling
// thread, so calls from different threads run concurrently (e.g. compress of chunk group g + 1 while group g decompresses, each
// on its own stream) and the entry points are thread-safe the way the reference documents its own (pco_c/src/lib.rs:57-70).
// The context follows the thread's current device: a cudaSetDevice between calls drops the scratch of the previous device.
struct Context {
  int device = -1;
  bool attrs_set = false;
  bool initialized = false;
  bool device_ok = false;
  std::string device_err;
  DevBuf src, out, index, statuses, misc, dec_syms, dec_offs, dec_narrow, gather, cold, spec;
  CompressScratch enc;
  Binoms* d_binoms = nullptr;
  int sm_count = 0;
  uint32_t last_decode_chunks = 0;  // chunks of the last decode launch (their class bytes are still at d_cls)
  std::vector<uint8_t> host_cls;    // class bytes of the last fused launch as the kernel reported them (0 = decoded there)
  uint8_t* d_cls = nullptr;         // class bytes of the last decode launch (they live behind the status words in `statuses`)
  void* pinned_res = nullptr;       // page-locked landing buffer for the statuses + class bytes of a decode launch
  size_t pinned_cap = 0;
  bool last_classes_fused = false;
  uint32_t* gather_err = nullptr;   // error word of the last page gather (inside `gather`)  // every chunk of the last launch was served by fused_narrow_kernel
};

static Context& ctx() {
  static thread_local Context c;
  return c;
}

static void release_buffers(Context& c) {
  for (DevBuf* b : {&c.src, &c.out, &c.index, &c.statuses, &c.misc, &c.dec_syms, &c.dec_offs, &c.dec_narrow, &c.gather, &c.cold, &c.spec}) b->release();
  c.enc.release();
  c.gather_err = nullptr;
  c.d_cls = nullptr;
  if (c.pinned_res) cudaFreeHost(c.pinned_res);
  c.pinned_res = nullptr;
  c.pinned_cap = 0;
  if (c.d_binoms) cudaFree(c.d_binoms);
  c.d_binoms = nullptr;
}

static PcoB200Error ensure_device(Context& c) {
  if (c.initialized && c.device_ok) {
    int cur = -1;
    if (cudaGetDevice(&cur) == cudaSuccess && cur != c.device) {  // the thread moved to another device: start over there
      const int now = cur;
      cudaSetDevice(c.device);
      release_buffers(c);
      cudaSetDevice(now);
      c.initialized = false;
      c.device_ok = false;
      c.attrs_set = false;
    }
  }
  if (!c.initialized) {
    c.initialized = true;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
      c.device_err = e != cudaSuccess ? cudaGetErrorString(e) : "no CUDA device";
      cudaGetLastError();
    } else {
      cudaDeviceProp prop;
      int dev = 0;
      cudaGetDevice(&dev);
      c.device = dev;
      e = cudaGetDeviceProperties(&prop, dev);
      if (e != cudaSuccess) c.device_err = cudaGetErrorString(e);
      else if (prop.major < 10) c.device_err = std::string("device ") + prop.name + " is not sm_100";
      else {
        c.sm_count = prop.multiProcessorCount;
        // binomials mod 2^64 by Pascal additions
        Binoms hb;
        std::vector<std::vector<uint64_t>> C(257, std::vector<uint64_t>(MAX_ORDER, 0));
        for (int nn = 0; nn <= 256; nn++) {
          C[nn][0] = 1;
          for (int j = 1; j < MAX_ORDER; j++) C[nn][j] = nn == 0 ? 0 : C[nn - 1][j - 1] + C[nn - 1][j];
        }
        for (int l = 0; l < 32; l++)
          for (int j = 0; j < MAX_ORDER; j++) hb.lane8[l][j] = C[8 * l][j];
        for (int j = 0; j < MAX_ORDER; j++) hb.full[j] = C[256][j];
        e = cudaMalloc(&c.d_binoms, sizeof(Binoms));
        if (e == cudaSuccess) e = cudaMemcpy(c.d_binoms, &hb, sizeof(Binoms), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(walk_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WalkSmem<12>));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(walk_kernel<SMALL_MAX_SIZE_LOG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WalkSmem<SMALL_MAX_SIZE_LOG>));
        if (e != cudaSuccess) c.device_err = cudaGetErrorString(e);
        else c.device_ok = true;
      }
    }
  }
  if (!c.device_ok)
    return fail(PCO_B200_CUDA, "CUDA device unavailable (" + c.device_err + "); libcpcodec has no CPU fallback");
  return PCO_B200_OK;
}

template <typename Fn>
static auto dispatch_latent(uint32_t dtype, Fn&& fn) {
  switch (nt_bits(dtype)) {
    case 8: return fn(uint8_t(0));
    case 16: return fn(uint16_t(0));
    case 32: return fn(uint32_t(0));
    default: return fn(uint64_t(0));
  }
}

// Function attributes of the decode kernels, set once per thread context (the first decode launch, or pco_b200_decompress_async_prepare).
static PcoB200Error set_decode_attrs(Context& c) {
  if (c.attrs_set) return PCO_B200_OK;
  c.attrs_set = true;
  PCOB_CUDA_TRY(cudaFuncSetAttribute(symwalk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SymWalkSmem)));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(symwalk_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint64_t>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint32_t>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint16_t>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  PCOB_CUDA_TRY(cudaFuncSetAttribute(fused_narrow_kernel<uint8_t>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  return PCO_B200_OK;
}

struct DecodeOutcome {
  uint64_t n_total = 0;   // numbers in the chunks seen
  bool terminated = false;
};

// Launch the decode over `n_chunks` IndexChunk records that live on the device.
//   1. fused_narrow_kernel (decode_fused.cuh): parses and classifies every chunk and fully decodes the narrow class;
//   2. only if some chunk is of another class: symwalk_kernel + decode_kernel<L, 1 / 2> for those.
// PCOB200_FUSED=0 selects the round-1 pair symwalk_kernel + decode_narrow_kernel (kept for A/B measurements).
static PcoB200Error launch_decode(Context& c, const FileParams& fp, const uint8_t* d_index, uint64_t index_len, uint64_t chunks_offset, uint32_t n_chunks,
                                  void* d_out, uint64_t out_len, cudaStream_t stream) {
  if (n_chunks == 0) return PCO_B200_OK;
  // status words and class bytes side by side: one copy brings both back
  const size_t res_bytes = size_t(n_chunks) * (sizeof(uint32_t) + 1);
  PCOB_CUDA_TRY(c.statuses.reserve(res_bytes + 64));
  uint32_t* d_st = c.statuses.as<uint32_t>();
  uint8_t* d_cls = reinterpret_cast<uint8_t*>(d_st + n_chunks);
  c.d_cls = d_cls;
  if (c.pinned_cap < res_bytes) {
    if (c.pinned_res) cudaFreeHost(c.pinned_res);
    c.pinned_res = nullptr;
    c.pinned_cap = 0;
    PCOB_CUDA_TRY(cudaHostAlloc(&c.pinned_res, res_bytes + (res_bytes >> 1) + 4096, cudaHostAllocDefault));
    c.pinned_cap = res_bytes + (res_bytes >> 1) + 4096;
  }
  const IndexChunk* d_chunks = reinterpret_cast<const IndexChunk*>(d_index + chunks_offset);
  static const bool use_fused = [] { const char* e = std::getenv("PCOB200_FUSED"); return !(e && e[0] == '0'); }();
  const bool narrow_ok = true;  // the fused kernel serves every number width
  if (PcoB200Error e = set_decode_attrs(c)) return e;
  c.last_decode_chunks = n_chunks;
  const uint32_t* st = static_cast<const uint32_t*>(c.pinned_res);
  bool fused_ran = false;
  if (!(use_fused && narrow_ok)) PCOB_CUDA_TRY(cudaMemsetAsync(d_st, 0xff, size_t(n_chunks) * sizeof(uint32_t), stream));  // the fused kernel writes every word itself
  if (use_fused && narrow_ok) {
    fused_ran = true;
    profiler().begin("fused_narrow_kernel", stream);
    dispatch_latent(fp.dtype, [&](auto tag) {
      using L = decltype(tag);
      fused_narrow_kernel<L><<<n_chunks, FZ_THREADS, sizeof(FusedSmem), stream>>>(fp, d_chunks, d_index, index_len, d_st, d_cls, static_cast<L*>(d_out), out_len, nullptr);
      return 0;
    });
    profiler().end(stream);
    PCOB_CUDA_TRY(cudaGetLastError());
    // statuses and class bytes come back in one round trip; the general kernels only run if some chunk still needs them
    PCOB_CUDA_TRY(readback_small_sync(c.pinned_res, d_st, (res_bytes + 3) & ~size_t(3), stream));  // the buffers hold res_bytes + 64
    const uint8_t* cls = reinterpret_cast<const uint8_t*>(st + n_chunks);
    c.host_cls.assign(cls, cls + n_chunks);
    bool pending = false;
    for (uint32_t i = 0; i < n_chunks; i++) {
      if (!(cls[i] & CLS_DONE)) { pending = true; continue; }
      if (st[i] != ST_OK) return status_to_error(st[i], ("chunk " + std::to_string(i)).c_str());
    }
    c.last_classes_fused = true;
    if (!pending) return PCO_B200_OK;
  }
  c.last_classes_fused = false;
  // scratch between the two kernels: one symbol byte per latent the destination can take, one section start per batch
  const uint64_t rows = scratch_rows_total(out_len, n_chunks);
  PCOB_CUDA_TRY(c.dec_syms.reserve(rows * BATCH_N + 64));
  PCOB_CUDA_TRY(c.dec_offs.reserve(rows * sizeof(uint32_t) + 64));
  const bool old_narrow = nt_bits(fp.dtype) >= 32 && !fused_ran;  // PCOB200_FUSED=0: the round-1 narrow kernel serves 32- and 64-bit types
  if (old_narrow) PCOB_CUDA_TRY(c.dec_narrow.reserve(size_t(n_chunks) * sizeof(NarrowInfo)));
  profiler().begin("symwalk_kernel", stream);
  symwalk_kernel<<<n_chunks, SW_THREADS, sizeof(SymWalkSmem), stream>>>(fp, d_chunks, d_index, index_len, out_len, c.dec_syms.as<uint8_t>(), c.dec_offs.as<uint32_t>(),
                                                                        d_cls, old_narrow ? c.dec_narrow.as<NarrowInfo>() : nullptr, fused_ran ? 1 : 0, nullptr);
  profiler().end(stream);
  profiler().begin("decode_kernel", stream);  // the span covers every decode instantiation (a chunk runs in exactly one)
  if (old_narrow) {
    if (nt_bits(fp.dtype) == 64)
      decode_narrow_kernel<uint64_t><<<n_chunks, NW_THREADS, 0, stream>>>(fp, d_chunks, d_st, static_cast<uint64_t*>(d_out), out_len, c.dec_syms.as<uint8_t>(),
                                                                        c.dec_offs.as<uint32_t>(), d_cls, c.dec_narrow.as<NarrowInfo>());
    else
      decode_narrow_kernel<uint32_t><<<n_chunks, NW_THREADS, 0, stream>>>(fp, d_chunks, d_st, static_cast<uint32_t*>(d_out), out_len, c.dec_syms.as<uint8_t>(),
                                                                        c.dec_offs.as<uint32_t>(), d_cls, c.dec_narrow.as<NarrowInfo>());
  }
  dispatch_latent(fp.dtype, [&](auto tag) {
    using L = decltype(tag);
    decode_kernel<L, 1><<<n_chunks, DEC_THREADS, sizeof(DecodeSmem), stream>>>(fp, d_chunks, d_st, d_index, index_len, static_cast<L*>(d_out), out_len, c.d_binoms,
                                                                                c.dec_syms.as<uint8_t>(), c.dec_offs.as<uint32_t>(), d_cls, nullptr);
    decode_kernel<L, 2><<<n_chunks, DEC_THREADS, sizeof(DecodeSmem), stream>>>(fp, d_chunks, d_st, d_index, index_len, static_cast<L*>(d_out), out_len, c.d_binoms,
                                                                                c.dec_syms.as<uint8_t>(), c.dec_offs.as<uint32_t>(), d_cls, nullptr);
    return 0;
  });
  profiler().end(stream);
  PCOB_CUDA_TRY(cudaGetLastError());
  PCOB_CUDA_TRY(readback_small_sync(c.pinned_res, d_st, size_t(n_chunks) * sizeof(uint32_t), stream));
  for (uint32_t i = 0; i < n_chunks; i++)
    if (st[i] != ST_OK) return status_to_error(st[i], ("chunk " + std::to_string(i)).c_str());
  return PCO_B200_OK;
}

// Index-free decompress, the parallel part (the reference's decompressor walks chunk after chunk, standalone/decompressor.rs:150-215;
// so did this library's serial walk_kernel<<<1>>>, at one GPU thread's ~0.2 GB/s).  Chunk lengths are not in the file, but the chunks
// of a file nearly always start with the same 4 bytes - the type byte and count - 1 (docs/format.md:186-192).  So, from the first
// unread chunk at `*next_byte`:
//   1. find_chunk_starts_kernel lists every position behind it that carries the same 4 bytes (the real chunk starts of that size
//      plus, once per ~4 GB of compressed bytes, a coincidence);
//   2. walk_kernel walks ALL of them at once, one thread each, as if each were a chunk start: index entries, status, end position;
//   3. the host follows the chain from the first chunk: the chunk at p is real, it ends at e(p), and if e(p) is on the list the chunk
//      there is real too (a coincidence is never reached: no verified chunk ends on it).  The verified chunks are decoded by the
//      ordinary kernels, their output offsets being k * n.
// The loop repeats from where the chain stopped (chunks of another size - typically the file's last one - start a new pattern) and
// hands over to the serial walker as soon as a round verifies nothing: the terminator, a chunk that does not fit `dst`, a corrupt or
// truncated chunk and every other special case keep the serial path's semantics and error reporting.
// `host_src` is the file in host memory (nullptr when it only lives on the device).  PCOB200_SPECULATIVE_WALK=0 turns this off.
static PcoB200Error speculative_walk_rounds(Context& c, const FileParams& fp, const uint8_t* host_src, void* dst, uint64_t dst_len, bool dst_dev, size_t elem,
                                            cudaStream_t stream, uint64_t* next_byte, uint64_t* out_off, void** d_out_io) {
  {  // read per call: tests of the serial walk switch it off in-process
    const char* e = std::getenv("PCOB200_SPECULATIVE_WALK");
    if (e && e[0] == '0') return PCO_B200_OK;
  }
  constexpr uint32_t CAND_CAP = 1u << 16;                  // candidates listed per round
  constexpr uint64_t INDEX_BUDGET = uint64_t(768) << 20;   // bytes of index scratch per round
  for (int round = 0; round < 4096; round++) {
    const uint64_t pos = *next_byte;
    if (pos + 4 > fp.src_len) return PCO_B200_OK;
    uint8_t h4[4];
    if (host_src) std::memcpy(h4, host_src + pos, 4);
    else {
      PCOB_CUDA_TRY(cudaMemcpyAsync(h4, static_cast<const uint8_t*>(fp.src) + pos, 4, cudaMemcpyDeviceToHost, stream));
      PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    }
    if (h4[0] != fp.dtype) return PCO_B200_OK;  // the terminator (0), or a type byte the serial path will report
    const uint32_t n0 = (uint32_t(h4[1]) | (uint32_t(h4[2]) << 8) | (uint32_t(h4[3]) << 16)) + 1;
    if (*out_off + n0 > dst_len) return PCO_B200_OK;  // the serial path owns the too-small-destination semantics
    const uint32_t pattern = uint32_t(h4[0]) | (uint32_t(h4[1]) << 8) | (uint32_t(h4[2]) << 16) | (uint32_t(h4[3]) << 24);
    // scratch: count | candidate positions | chunk ends | statuses
    PCOB_CUDA_TRY(c.spec.reserve(64 + size_t(CAND_CAP) * (8 + 8 + 4)));
    uint32_t* d_count = c.spec.as<uint32_t>();
    uint64_t* d_cand = reinterpret_cast<uint64_t*>(c.spec.as<uint8_t>() + 64);
    uint64_t* d_ends = d_cand + CAND_CAP;
    uint32_t* d_stat = reinterpret_cast<uint32_t*>(d_ends + CAND_CAP);
    PCOB_CUDA_TRY(cudaMemsetAsync(d_count, 0, 4, stream));
    const uint64_t scan_end = fp.src_len - 3;  // last position + 1 whose 4 bytes lie inside the file
    const uint64_t per_block = uint64_t(FIND_THREADS) * FIND_PER_THREAD;
    const uint64_t blocks = (scan_end - pos + per_block - 1) / per_block;
    if (blocks > 0x7fffffffull) return PCO_B200_OK;
    profiler().begin("find_chunk_starts_kernel", stream);
    find_chunk_starts_kernel<<<uint32_t(blocks), FIND_THREADS, 0, stream>>>(static_cast<const uint8_t*>(fp.src), pos, scan_end, pattern, d_cand, CAND_CAP, d_count);
    profiler().end(stream);
    PCOB_CUDA_TRY(cudaGetLastError());
    uint32_t count = 0;
    PCOB_CUDA_TRY(cudaMemcpyAsync(&count, d_count, 4, cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    if (count == 0 || count > CAND_CAP) return PCO_B200_OK;  // a file full of the pattern: not worth speculating on
    std::vector<uint64_t> cand(count);
    PCOB_CUDA_TRY(cudaMemcpyAsync(cand.data(), d_cand, size_t(count) * 8, cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    std::sort(cand.begin(), cand.end());
    if (cand[0] != pos) return PCO_B200_OK;
    // walk as many candidates (in file order) as the index budget and the destination allow
    const uint32_t nb0 = n_batches_of(n0);
    const uint64_t stride = (uint64_t(MAX_VARS) * nb0 * sizeof(BatchEntry) + 15) & ~uint64_t(15);
    const uint64_t fit = (dst_len - *out_off) / n0;  // chunks of this size the destination can still take (>= 1)
    uint64_t m64 = std::min<uint64_t>(count, std::max<uint64_t>(1, INDEX_BUDGET / (stride + sizeof(IndexChunk))));
    m64 = std::min<uint64_t>(m64, fit + 8);  // a few more than fit: coincidences in front of the last chunk needed
    const uint32_t m = uint32_t(m64);
    const uint64_t chunks_offset = sizeof(IndexHeader);
    const uint64_t entries_begin = (chunks_offset + uint64_t(m) * sizeof(IndexChunk) + 15) & ~uint64_t(15);
    const uint64_t index_bytes = entries_begin + uint64_t(m) * stride;
    std::vector<IndexChunk> recs(m);
    for (uint32_t k = 0; k < m; k++) {
      recs[k].chunk_offset = cand[k];
      recs[k].n = n0;
      recs[k].n_vars = 0;
      recs[k].entries_offset = entries_begin + uint64_t(k) * stride;
      recs[k].out_offset = 0;
    }
    PCOB_CUDA_TRY(c.index.reserve(index_bytes + 64));
    uint8_t* d_index = c.index.as<uint8_t>();
    PCOB_CUDA_TRY(cudaMemcpyAsync(d_index + chunks_offset, recs.data(), size_t(m) * sizeof(IndexChunk), cudaMemcpyHostToDevice, stream));
    PCOB_CUDA_TRY(cudaMemsetAsync(d_stat, 0xff, size_t(m) * 4, stream));
    PCOB_CUDA_TRY(cudaMemsetAsync(d_ends, 0, size_t(m) * 8, stream));
    PCOB_CUDA_TRY(c.misc.reserve(sizeof(WalkResult)));
    profiler().begin("walk_kernel", stream);
    walk_kernel<SMALL_MAX_SIZE_LOG><<<m, WALK_THREADS, sizeof(WalkSmem<SMALL_MAX_SIZE_LOG>), stream>>>(
        fp, d_index, chunks_offset, m, 0, index_bytes, 0, 0, ~uint64_t(0), d_stat, c.misc.as<WalkResult>(), 0, d_ends);
    profiler().end(stream);
    PCOB_CUDA_TRY(cudaGetLastError());
    std::vector<uint32_t> st(m);
    std::vector<uint64_t> ends(m);
    PCOB_CUDA_TRY(cudaMemcpyAsync(st.data(), d_stat, size_t(m) * 4, cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaMemcpyAsync(ends.data(), d_ends, size_t(m) * 8, cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaMemcpyAsync(recs.data(), d_index + chunks_offset, size_t(m) * sizeof(IndexChunk), cudaMemcpyDeviceToHost, stream));  // n_vars as walked
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    // the chain of real chunks
    uint64_t p = pos;
    const std::vector<uint32_t> chain = follow_chunk_chain(cand.data(), st.data(), ends.data(), m, pos, n0, *out_off, dst_len, fp.src_len, &p);
    std::vector<IndexChunk> real;
    real.reserve(chain.size());
    for (uint32_t k : chain) {
      IndexChunk ic = recs[k];
      ic.out_offset = *out_off + uint64_t(real.size()) * n0;
      real.push_back(ic);
    }
    if (real.empty()) return PCO_B200_OK;
    PCOB_CUDA_TRY(cudaMemcpyAsync(d_index + chunks_offset, real.data(), real.size() * sizeof(IndexChunk), cudaMemcpyHostToDevice, stream));
    const uint64_t emit_end = *out_off + uint64_t(real.size()) * n0;
    void* d_out = dst;
    if (!dst_dev) {
      PCOB_CUDA_TRY(c.out.grow_preserve(emit_end * elem + 64, *out_off * elem, stream));
      d_out = c.out.p;
    }
    if (PcoB200Error e = launch_decode(c, fp, d_index, index_bytes, chunks_offset, uint32_t(real.size()), d_out, dst_dev ? dst_len : emit_end, stream)) return e;
    *d_out_io = d_out;
    *out_off = emit_end;
    *next_byte = p;
  }
  return PCO_B200_OK;
}


// The fast kernels behind every decompress entry point.  The walk goes on while the numbers seen fit the destination - an exact fit still
// has to find the terminator (a truncated file is an error for both of the reference's semantics) - and stops with `terminated = false`
// and n_total > dst_len at the first chunk that does not fit: pco_standalone_simple_decompress_into turns that into its "exceeds dst_cap"
// error (pco_c/src/lib.rs:98-120), pco_b200_decompress_ex into Progress{finished = false} (standalone/simple.rs:115-140).
static PcoB200Error decompress_fast(const void* compressed, size_t compressed_len, uint32_t dtype, void* dst, size_t dst_len,
                                    const void* index, size_t index_len, uint32_t flags, void* cuda_stream, DecodeOutcome* outcome) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  const bool src_dev = flags & PCO_B200_SRC_ON_DEVICE, dst_dev = flags & PCO_B200_DST_ON_DEVICE;
  const size_t elem = nt_bits(dtype) / 8;

  // 1. standalone header (host parse of the first bytes)
  uint8_t head[32] = {0};
  size_t avail = std::min<size_t>(compressed_len, sizeof(head));
  // the file header and (when it lives on the device) the side index header come back in one round trip
  const bool have_index = index != nullptr && index_len >= sizeof(IndexHeader);
  const bool idx_dev = flags & PCO_B200_INDEX_ON_DEVICE;
  IndexHeader ih;
  std::memset(&ih, 0, sizeof(ih));
  bool need_sync = false;
  if (avail) {
    if (src_dev) { PCOB_CUDA_TRY(cudaMemcpyAsync(head, compressed, avail, cudaMemcpyDeviceToHost, stream)); need_sync = true; }
    else std::memcpy(head, compressed, avail);
  }
  if (have_index) {
    if (idx_dev) { PCOB_CUDA_TRY(cudaMemcpyAsync(&ih, index, sizeof(ih), cudaMemcpyDeviceToHost, stream)); need_sync = true; }
    else std::memcpy(&ih, index, sizeof(ih));
  }
  if (need_sync) PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
  StandaloneHeader hdr;
  if (PcoB200Error e = parse_standalone_header(head, avail, compressed_len, &hdr)) return e;

  // 2. the file in HBM
  const uint8_t* d_src;
  if (src_dev) d_src = static_cast<const uint8_t*>(compressed);
  else {
    PCOB_CUDA_TRY(c.src.reserve(compressed_len + 16));
    call_trace().mark("d.begin");
    PCOB_CUDA_TRY(copy_sliced(c.src.p, compressed, compressed_len, cudaMemcpyHostToDevice, stream));
    call_trace().mark("d.h2d_submitted");
    d_src = c.src.as<uint8_t>();
  }
  FileParams fp;
  fp.src = d_src;
  fp.src_len = compressed_len;
  fp.dtype = dtype;
  fp.uniform_type = hdr.uniform_type;
  fp.format_major = hdr.format_major;

  // 3a. caller-supplied side index
  if (have_index) {
    // overflow-safe: the chunk table must lie inside the index; per-chunk fields are bounded on the device (entries inside the
    // index, chunk_offset inside the file, writes inside the destination)
    if (ih.magic != INDEX_MAGIC || ih.version != 1 || ih.file_len != compressed_len || ih.chunks_offset > index_len ||
        ih.n_chunks > (index_len - ih.chunks_offset) / sizeof(IndexChunk))
      return fail(PCO_B200_INVALID_ARGUMENT, "side index does not belong to this file");
    const uint8_t* d_idx = static_cast<const uint8_t*>(index);
    if (!idx_dev) {
      PCOB_CUDA_TRY(c.index.reserve(index_len));
      PCOB_CUDA_TRY(copy_sliced(c.index.p, index, index_len, cudaMemcpyHostToDevice, stream));
      d_idx = c.index.as<uint8_t>();
    }
    uint64_t n_emit = std::min<uint64_t>(ih.n_total, dst_len);
    void* d_out = dst;
    bool dst_in_place = false;
    if (!dst_dev) {
      // a page-locked destination is written in place by the decode kernels (every number is stored once, in 32-byte pieces that a
      // warp lays down as 1 KiB runs): no staging buffer, no copy behind the kernel (host_common.hpp, zero copy)
      void* in_place = (zero_copy_mask().load(std::memory_order_relaxed) & 2) ? mapped_host_ptr(dst) : nullptr;
      if (in_place) {
        d_out = in_place;
        dst_in_place = true;
      } else {
        PCOB_CUDA_TRY(c.out.reserve(n_emit * elem + 64));
        d_out = c.out.p;
      }
    }
    if (ih.n_chunks > 0xffffffffull) return fail(PCO_B200_INVALID_ARGUMENT, "too many chunks");
    // a host destination holds (or is staged in c.out, which holds) n_emit numbers: that is the kernels' bound, whatever the index claims
    if (PcoB200Error e = launch_decode(c, fp, d_idx, index_len, ih.chunks_offset, uint32_t(ih.n_chunks), d_out, dst_dev ? uint64_t(dst_len) : n_emit, stream)) return e;
    call_trace().mark("d.decoded");
    if (dst_in_place) {
      PCOB_CUDA_TRY(cudaStreamSynchronize(stream));  // launch_decode has read the statuses back already: the stores are in host memory
    } else if (!dst_dev && n_emit) {
      PCOB_CUDA_TRY(copy_sliced(dst, d_out, n_emit * elem, cudaMemcpyDeviceToHost, stream));
      call_trace().mark("d.d2h_submitted");
      PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    }
    call_trace().mark("d.end");
    call_trace().flush("decompress");
    outcome->n_total = ih.n_total;
    outcome->terminated = ih.end_byte != 0;
    return PCO_B200_OK;
  }

  // 3b. no index: walk the file on the device in rounds, decoding each round's chunks.
  // Chunk boundaries are not in the stream, so this is one serial tANS walk (cold path).
  const uint32_t max_chunks = uint32_t(std::min<uint64_t>(uint64_t(compressed_len) / 5 + 2, 1u << 16));
  uint64_t next_byte = hdr.first_chunk_byte;
  uint64_t out_off = 0;
  void* d_out = dst;
  // runs of same-sized chunks are found, walked and decoded in parallel; what is left (the terminator at least) goes through the serial walk
  if (PcoB200Error e = speculative_walk_rounds(c, fp, src_dev ? nullptr : static_cast<const uint8_t*>(compressed), dst, uint64_t(dst_len), dst_dev, elem, stream,
                                               &next_byte, &out_off, &d_out))
    return e;
  PCOB_CUDA_TRY(c.misc.reserve(sizeof(WalkResult)));
  WalkResult* d_res = c.misc.as<WalkResult>();
  for (;;) {
    // scratch index: header | IndexChunk[max_chunks] | entries for the batches dst can still take (+2 per chunk) x 2 vars
    const uint64_t chunks_offset = sizeof(IndexHeader);
    const uint64_t entries_begin = chunks_offset + uint64_t(max_chunks) * sizeof(IndexChunk);
    uint64_t want_batches = (dst_len > out_off ? (dst_len - out_off) / BATCH_N : 0) + 2ull * max_chunks + 2;
    want_batches = std::min<uint64_t>(want_batches, uint64_t(1) << 23);
    const uint64_t entries_bytes = want_batches * MAX_VARS * sizeof(BatchEntry) + 16ull * max_chunks + 64;
    PCOB_CUDA_TRY(c.index.reserve(entries_begin + entries_bytes));
    uint8_t* d_index = c.index.as<uint8_t>();
    profiler().begin("walk_kernel", stream);
    walk_kernel<12><<<1, WALK_THREADS, sizeof(WalkSmem<12>), stream>>>(fp, d_index, chunks_offset, max_chunks, entries_begin, entries_begin + entries_bytes,
                                                      next_byte, out_off, uint64_t(dst_len), nullptr, d_res, 1);
    profiler().end(stream);
    PCOB_CUDA_TRY(cudaGetLastError());
    WalkResult res;
    PCOB_CUDA_TRY(cudaMemcpyAsync(&res, d_res, sizeof(res), cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    const bool soft = res.status == ST_TERMINATOR || res.status == ST_INDEX_FULL || res.status == ST_DST_FULL;
    // decode what was indexed this round (the reference also emits the chunks before a failing one)
    if (res.n_chunks > 0) {
      uint64_t round_emit_end = std::min<uint64_t>(out_off + res.n_total, dst_len);
      if (!dst_dev) {
        PCOB_CUDA_TRY(c.out.grow_preserve(round_emit_end * elem + 64, std::min<uint64_t>(out_off, dst_len) * elem, stream));
        d_out = c.out.p;
      }
      if (PcoB200Error e = launch_decode(c, fp, d_index, entries_begin + entries_bytes, chunks_offset, res.n_chunks, d_out, dst_dev ? uint64_t(dst_len) : round_emit_end, stream)) return e;
    }
    out_off += res.n_total;
    next_byte = res.next_byte;
    if (!soft) return status_to_error(res.status, ("chunk " + std::to_string(res.n_chunks) + " of this walk round").c_str());
    if (res.status == ST_TERMINATOR) { outcome->terminated = true; break; }
    if (res.status == ST_DST_FULL) break;
    if (res.n_chunks == 0) return fail(PCO_B200_UNSUPPORTED, "a single chunk exceeds the device index scratch");
  }
  outcome->n_total = out_off;
  uint64_t n_emit = std::min<uint64_t>(out_off, dst_len);
  if (!dst_dev && n_emit) {
    PCOB_CUDA_TRY(copy_sliced(dst, d_out, n_emit * elem, cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
  }
  return PCO_B200_OK;
}

// The catch-all behind the fast kernels: the whole file through cold_decode_kernel (decode_cold.cuh) - one GPU thread, any valid pco.
static PcoB200Error decompress_cold(const void* compressed, size_t compressed_len, uint32_t dtype, void* dst, size_t dst_len, uint32_t flags, void* cuda_stream,
                                    DecodeOutcome* outcome) {
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  const bool src_dev = flags & PCO_B200_SRC_ON_DEVICE, dst_dev = flags & PCO_B200_DST_ON_DEVICE;
  const size_t elem = nt_bits(dtype) / 8;
  uint8_t head[32] = {0};
  const size_t avail = std::min<size_t>(compressed_len, sizeof(head));
  if (avail) {
    if (src_dev) { PCOB_CUDA_TRY(cudaMemcpyAsync(head, compressed, avail, cudaMemcpyDeviceToHost, stream)); PCOB_CUDA_TRY(cudaStreamSynchronize(stream)); }
    else std::memcpy(head, compressed, avail);
  }
  StandaloneHeader hdr;
  if (PcoB200Error e = parse_standalone_header(head, avail, compressed_len, &hdr)) return e;
  const uint8_t* d_src = static_cast<const uint8_t*>(compressed);
  if (!src_dev) {
    PCOB_CUDA_TRY(c.src.reserve(compressed_len + 16));
    PCOB_CUDA_TRY(copy_sliced(c.src.p, compressed, compressed_len, cudaMemcpyHostToDevice, stream));
    d_src = c.src.as<uint8_t>();
  }
  FileParams fp{d_src, compressed_len, dtype, hdr.uniform_type, hdr.format_major};
  void* d_out = dst;
  if (!dst_dev) {
    PCOB_CUDA_TRY(c.out.reserve(dst_len * elem + 64));
    d_out = c.out.p;
  }
  PCOB_CUDA_TRY(c.misc.reserve(256));
  ColdResult* d_res = reinterpret_cast<ColdResult*>(c.misc.as<uint8_t>() + 160);
  ColdResult res;
  for (uint32_t window_cap : {16u, COLD_MAX_WINDOW_LOG}) {  // lookback windows beyond 2^16 numbers get the large scratch on a second try
    PCOB_CUDA_TRY(c.cold.reserve(cold_scratch_bytes(window_cap)));
    profiler().begin("cold_decode_kernel", stream);
    dispatch_latent(dtype, [&](auto tag) {
      using L = decltype(tag);
      cold_decode_kernel<L><<<1, 32, 0, stream>>>(fp, hdr.first_chunk_byte, static_cast<L*>(d_out), uint64_t(dst_len), c.cold.as<uint8_t>(), window_cap, d_res);
      return 0;
    });
    profiler().end(stream);
    PCOB_CUDA_TRY(cudaGetLastError());
    PCOB_CUDA_TRY(cudaMemcpyAsync(&res, d_res, sizeof(res), cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    if (res.status != ST_UNSUPPORTED) break;
  }
  // like the walk path: the chunks before a failing one have been emitted (the reference's decoder stops where the error is)
  const uint64_t n_emit = std::min<uint64_t>(res.n_total, dst_len);
  if (!dst_dev && n_emit) {
    PCOB_CUDA_TRY(copy_sliced(dst, d_out, n_emit * elem, cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
  }
  if (res.status != ST_TERMINATOR && res.status != ST_DST_FULL) return status_to_error(res.status, ("chunk " + std::to_string(res.n_chunks)).c_str());
  outcome->n_total = res.n_total;
  outcome->terminated = res.status == ST_TERMINATOR;
  return PCO_B200_OK;
}

// Core of every decompress entry point: the fast kernels, and for streams they decline (valid pco with Dict mode, Lookback / Conv1
// deltas, tANS tables beyond 2^10 states or 256 bins, ...) the single-thread device decoder.  PCOB200_COLD_DECODE=0 keeps the refusal.
static PcoB200Error decompress_core(const void* compressed, size_t compressed_len, uint32_t dtype, void* dst, size_t dst_len,
                                    const void* index, size_t index_len, uint32_t flags, void* cuda_stream, DecodeOutcome* outcome) {
  PcoB200Error e = decompress_fast(compressed, compressed_len, dtype, dst, dst_len, index, index_len, flags, cuda_stream, outcome);
  static const bool cold_ok = [] { const char* v = std::getenv("PCOB200_COLD_DECODE"); return !(v && v[0] == '0'); }();
  if (e == PCO_B200_UNSUPPORTED && cold_ok) {
    *outcome = DecodeOutcome();
    e = decompress_cold(compressed, compressed_len, dtype, dst, dst_len, flags, cuda_stream, outcome);
  }
  return e;
}

// ---- stream-ordered decompress (pco_b200_decompress_async) ---------------------------------------------------------------------------
// The caller's workspace, from a 256-byte aligned base: gate | binomials | statuses | class bytes | the general pair's symbol rows |
// its section starts.  The rows are sized from n_total (the kernels' out_len), as scratch_rows_total does for a 64-bit chunk count.
struct AsyncLayout {
  size_t gate, binoms, statuses, cls, syms, offs, total;
};
static AsyncLayout async_layout(uint64_t n_total, uint64_t n_chunks) {
  auto up = [](uint64_t x) { return (x + 255) & ~uint64_t(255); };
  const uint64_t rows = uint64_t(MAX_VARS) * (n_total / BATCH_N + n_chunks + 1);
  AsyncLayout l;
  uint64_t o = 0;
  l.gate = o; o += up(sizeof(AsyncGate));
  l.binoms = o; o += up(sizeof(Binoms));
  l.statuses = o; o += up(n_chunks * sizeof(uint32_t));
  l.cls = o; o += up(n_chunks);
  l.syms = o; o += up(rows * BATCH_N + 64);
  l.offs = o; o += up(rows * sizeof(uint32_t) + 64);
  l.total = o + 256;  // room to align the caller's pointer
  return l;
}

// The thread context's one-time set-up (device, binomials, kernel attributes) runs synchronous CUDA calls, which a stream capture
// refuses: during a capture it has to have happened already.
static PcoB200Error async_setup(Context& c, cudaStream_t stream) {
  int cur = -1;
  const bool ready = c.initialized && c.device_ok && c.attrs_set && cudaGetDevice(&cur) == cudaSuccess && cur == c.device;
  if (!ready) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone)
      return fail(PCO_B200_CUDA, "the first pco_b200_decompress_async on a thread and device cannot be captured: call pco_b200_decompress_async_prepare before capturing");
    cudaGetLastError();
  }
  if (PcoB200Error e = ensure_device(c)) return e;
  return set_decode_attrs(c);
}

}  // namespace pcob200

using namespace pcob200;

extern "C" {

const char* pco_b200_last_error_message(void) { return last_error_ref().c_str(); }

int pco_b200_device_available(void) {
  Context& c = ctx();
  return ensure_device(c) == PCO_B200_OK ? 1 : 0;
}

// pco_c/src/lib.rs:127-139
size_t pco_standalone_guarantee_file_size(size_t n, unsigned char dtype) {
  if (!nt_valid(dtype)) return 0;
  // PagingSpec::default() = EqualPagesUpTo(2^18) (pco/src/chunk_config.rs:127-132, :134-183)
  const size_t max_page_n = size_t(1) << 18;
  size_t res = standalone_header_size();
  if (n > 0) {
    size_t n_pages = (n + max_page_n - 1) / max_page_n;
    size_t low = n / n_pages, r = n % n_pages;
    res += r * standalone_chunk_size_guarantee(nt_bits(dtype), low + 1) + (n_pages - r) * standalone_chunk_size_guarantee(nt_bits(dtype), low);
  }
  return res + 1;
}

// pco_c/src/lib.rs:98-120,178-195: full simple_decompress, then fail if it does not fit.
enum PcoError pco_standalone_simple_decompress_into(const void* compressed, size_t compressed_len, unsigned char dtype, void* dst,
                                                    size_t dst_cap, size_t* n_written) {
  if (!nt_valid(dtype)) return PcoInvalidType;
  DecodeOutcome oc;
  PcoB200Error e = decompress_core(compressed, compressed_len, dtype, dst, dst_cap, nullptr, 0, 0, nullptr, &oc);
  if (e != PCO_B200_OK) return PcoDecompressionError;
  if (oc.n_total > dst_cap) {
    fail(PCO_B200_IO, "decompressed count exceeds dst_cap");
    return PcoDecompressionError;
  }
  if (n_written) *n_written = size_t(oc.n_total);
  return PcoSuccess;
}

PcoB200Error pco_b200_decompress_ex(const void* compressed, size_t compressed_len, unsigned char dtype, void* dst, size_t dst_len,
                                    PcoB200Progress* progress, const void* index, size_t index_len, uint32_t flags, void* cuda_stream) {
  DecodeOutcome oc;
  PcoB200Error e = decompress_core(compressed, compressed_len, dtype, dst, dst_len, index, index_len, flags, cuda_stream, &oc);
  profiler().resolve();
  if (e != PCO_B200_OK) return e;
  if (progress) {
    progress->n_processed = size_t(std::min<uint64_t>(oc.n_total, dst_len));
    progress->finished = (oc.terminated && oc.n_total <= dst_len) ? 1 : 0;
  }
  return PCO_B200_OK;
}

size_t pco_b200_decompress_async_workspace_size(size_t n_total, size_t n_chunks, unsigned char dtype) {
  if (!nt_valid(dtype)) return 0;
  return size_t(async_layout(n_total, n_chunks).total);
}

PcoB200Error pco_b200_decompress_async_prepare(unsigned char dtype) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  return async_setup(ctx(), nullptr);
}

// Six launches on `cuda_stream` and nothing else: async_validate_kernel, fused_narrow_kernel, symwalk_kernel, decode_kernel<L, 1>,
// decode_kernel<L, 2>, async_outcome_kernel.  The general pair runs whatever the fused kernel left, since the host does not look: the
// chunks the fused kernel finished leave its CTAs at once through their class bytes.
PcoB200Error pco_b200_decompress_async(const void* d_src, size_t src_len, unsigned char dtype, const void* d_index, size_t index_len, size_t n_chunks,
                                       size_t n_total, void* d_dst, size_t dst_len, void* d_workspace, size_t workspace_len, PcoB200AsyncResult* d_result,
                                       void* cuda_stream) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  if (!d_src || !d_index || !d_dst || !d_workspace || !d_result) return fail(PCO_B200_INVALID_ARGUMENT, "null pointer");
  if (n_chunks == 0 || n_chunks > 0x7fffffffull) return fail(PCO_B200_INVALID_ARGUMENT, "n_chunks must be 1..2^31 - 1");
  if (dst_len < n_total) return fail(PCO_B200_INVALID_ARGUMENT, "dst holds " + std::to_string(dst_len) + " numbers, the file " + std::to_string(n_total));
  if (index_len < sizeof(IndexHeader) || (index_len - sizeof(IndexHeader)) / sizeof(IndexChunk) < n_chunks)
    return fail(PCO_B200_INVALID_ARGUMENT, "side index is shorter than its chunk table");
  if (reinterpret_cast<uintptr_t>(d_index) & 7) return fail(PCO_B200_INVALID_ARGUMENT, "side index must be 8-byte aligned");
  const AsyncLayout lay = async_layout(n_total, n_chunks);
  if (workspace_len < lay.total)
    return fail(PCO_B200_INVALID_ARGUMENT, "workspace holds " + std::to_string(workspace_len) + " bytes, the call needs " + std::to_string(lay.total));
  Context& c = ctx();
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  if (PcoB200Error e = async_setup(c, stream)) return e;
  uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(d_workspace) + 255) & ~uintptr_t(255));
  AsyncGate* gate = reinterpret_cast<AsyncGate*>(ws + lay.gate);
  const uint32_t* gate_words = reinterpret_cast<const uint32_t*>(gate);
  Binoms* binoms = reinterpret_cast<Binoms*>(ws + lay.binoms);
  uint32_t* d_st = reinterpret_cast<uint32_t*>(ws + lay.statuses);
  uint8_t* d_cls = ws + lay.cls;
  uint8_t* d_syms = ws + lay.syms;
  uint32_t* d_offs = reinterpret_cast<uint32_t*>(ws + lay.offs);
  const uint8_t* d_idx = static_cast<const uint8_t*>(d_index);
  const IndexChunk* d_chunks = reinterpret_cast<const IndexChunk*>(d_idx + sizeof(IndexHeader));  // chunks_offset is checked on the device
  const uint32_t grid = uint32_t(n_chunks);
  // uniform_type and format_major come from the gate; the kernels write no number at or beyond n_total
  FileParams fp{d_src, uint64_t(src_len), dtype, 0, 4};
  async_validate_kernel<<<1, 32, 0, stream>>>(static_cast<const uint8_t*>(d_src), src_len, dtype, d_idx, index_len, n_chunks, n_total, gate, binoms, d_result);
  dispatch_latent(dtype, [&](auto tag) {
    using L = decltype(tag);
    L* out = static_cast<L*>(d_dst);
    fused_narrow_kernel<L><<<grid, FZ_THREADS, sizeof(FusedSmem), stream>>>(fp, d_chunks, d_idx, index_len, d_st, d_cls, out, n_total, gate_words);
    symwalk_kernel<<<grid, SW_THREADS, sizeof(SymWalkSmem), stream>>>(fp, d_chunks, d_idx, index_len, n_total, d_syms, d_offs, d_cls, nullptr, 1, gate_words);
    decode_kernel<L, 1><<<grid, DEC_THREADS, sizeof(DecodeSmem), stream>>>(fp, d_chunks, d_st, d_idx, index_len, out, n_total, binoms, d_syms, d_offs, d_cls, gate_words);
    decode_kernel<L, 2><<<grid, DEC_THREADS, sizeof(DecodeSmem), stream>>>(fp, d_chunks, d_st, d_idx, index_len, out, n_total, binoms, d_syms, d_offs, d_cls, gate_words);
    return 0;
  });
  async_outcome_kernel<<<1, OUTCOME_THREADS, 0, stream>>>(gate_words, d_st, d_cls, grid, d_result);
  PCOB_CUDA_TRY(cudaGetLastError());
  return PCO_B200_OK;
}

PcoB200Error pco_b200_simple_decompress_into(const void* compressed, size_t compressed_len, unsigned char dtype, void* dst, size_t dst_len,
                                             PcoB200Progress* progress) {
  return pco_b200_decompress_ex(compressed, compressed_len, dtype, dst, dst_len, progress, nullptr, 0, 0, nullptr);
}

static PcoB200Error compress_dispatch(const void* nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig* config, bool uniform, void* dst,
                                      size_t dst_cap, size_t* n_written, void* index, size_t index_cap, size_t* index_len, uint32_t flags,
                                      void* cuda_stream) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  PcoB200ChunkConfig cfg;
  if (config) cfg = *config;
  else {
    std::memset(&cfg, 0, sizeof(cfg));  // pco::ChunkConfig::default(): level 8, Auto, Auto, EqualPagesUpTo(2^18)
    cfg.compression_level = 8;
  }
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  CompressResult res;
  PcoB200Error e = dispatch_latent(dtype, [&](auto tag) {
    using L = decltype(tag);
    return compress_typed<L>(c.enc, nums, n, dtype, cfg, uniform, dst, dst_cap, index, index_cap, flags, static_cast<cudaStream_t>(cuda_stream), &res);
  });
  profiler().resolve();
  if (e != PCO_B200_OK) return e;
  if (n_written) *n_written = size_t(res.total_bytes);
  if (index_len) *index_len = size_t(res.index_bytes);
  return PCO_B200_OK;
}

PcoB200Error pco_b200_compress_ex(const void* nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig* config, int uniform_type_header,
                                  void* dst, size_t dst_cap, size_t* n_written, void* index, size_t index_cap, size_t* index_len, uint32_t flags,
                                  void* cuda_stream) {
  return compress_dispatch(nums, n, dtype, config, uniform_type_header != 0, dst, dst_cap, n_written, index, index_cap, index_len, flags, cuda_stream);
}
PcoB200Error pco_b200_simple_compress(const void* nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig* config, void* dst, size_t dst_cap,
                                      size_t* n_written) {
  return compress_dispatch(nums, n, dtype, config, false, dst, dst_cap, n_written, nullptr, 0, nullptr, 0, nullptr);
}
PcoB200Error pco_b200_simple_compress_into(const void* nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig* config, void* dst,
                                           size_t dst_cap, size_t* n_written) {
  return compress_dispatch(nums, n, dtype, config, true, dst, dst_cap, n_written, nullptr, 0, nullptr, 0, nullptr);
}

// pco_c/src/lib.rs:76-96,146-169: Auto mode / Auto delta, enable_8_bit, uniform-type header
enum PcoError pco_standalone_simple_compress_into(const void* nums, size_t n, unsigned char dtype, const struct PcoChunkConfig* config, void* dst,
                                                  size_t dst_cap, size_t* n_written) {
  if (!nt_valid(dtype)) return PcoInvalidType;
  PcoB200ChunkConfig cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  cfg.compression_level = config ? config->compression_level : 8;
  cfg.max_page_n = config ? config->max_page_n : 0;
  cfg.mode_spec = PCO_B200_MODE_AUTO;
  cfg.delta_spec = PCO_B200_DELTA_AUTO;
  cfg.enable_8_bit = 1;
  PcoB200Error e = compress_dispatch(nums, n, dtype, &cfg, true, dst, dst_cap, n_written, nullptr, 0, nullptr, 0, nullptr);
  return e == PCO_B200_OK ? PcoSuccess : PcoCompressionError;
}

// ---------------------------------------------------------------------------
// Wrapped format (pco/src/wrapped/): one page per chunk.  A wrapped chunk = chunk meta bytes + page bytes, i.e. a
// standalone chunk without its 4-byte preamble, so the compressor handle holds one CHUNKS_ONLY chunk and the page
// decoder re-frames meta + page as a one-chunk standalone file for the same kernels.
// ---------------------------------------------------------------------------
struct PcoB200ChunkCompressor {
  // one emission per page, back to back: [type byte][page_n - 1 (24 bits)][chunk meta][page]; the pages of a chunk share
  // their bins, so every emission carries the same chunk meta
  std::vector<uint8_t> bytes;
  size_t meta_len = 0;
  size_t n = 0;
  std::vector<size_t> page_off, page_n;  // byte offset of each emission (+ one past the last), numbers per page
};

namespace {
// Byte length of a chunk meta (metadata/chunk.rs:127-189, delta_encoding.rs, chunk_latent_var.rs:55-71) read from host bytes.
// Only what the GPU path writes/reads is accepted: Classic / IntMult / FloatMult / FloatQuant, delta None / Consecutive.
PcoB200Error host_chunk_meta_len(const uint8_t* b, size_t len, uint32_t dtype, size_t* out) {
  const uint32_t lbits = nt_bits(dtype);
  uint64_t pos = 0;
  bool short_read = false;
  auto rd = [&](uint32_t nb) -> uint64_t {
    uint64_t v = 0;
    for (uint32_t i = 0; i < nb; i++) {
      const uint64_t bit = pos + i;
      if ((bit >> 3) >= len) { short_read = true; break; }
      v |= uint64_t((b[bit >> 3] >> (bit & 7)) & 1) << i;
    }
    pos += nb;
    return v;
  };
  const uint32_t mode = uint32_t(rd(4));
  uint32_t n_vars = 2;
  switch (mode) {
    case MODE_CLASSIC: n_vars = 1; break;
    case MODE_INT_MULT: case MODE_FLOAT_MULT: pos += lbits; break;
    case MODE_FLOAT_QUANT: pos += 8; break;
    default: return fail(PCO_B200_UNSUPPORTED, "wrapped chunk meta: mode outside the GPU hot path");
  }
  const uint32_t delta = uint32_t(rd(4));
  if (delta == 1) pos += 4;  // order (3 bits) + secondary_uses_delta (1 bit)
  else if (delta != 0) return fail(PCO_B200_UNSUPPORTED, "wrapped chunk meta: delta encoding outside the GPU hot path");
  for (uint32_t v = 0; v < n_vars; v++) {
    const uint32_t size_log = uint32_t(rd(4));
    const uint32_t n_bins = uint32_t(rd(15));
    pos += uint64_t(n_bins) * (size_log + lbits + offset_bits_bits(lbits));
  }
  if (short_read || (pos + 7) / 8 > len) return fail(PCO_B200_INSUFFICIENT_DATA, "chunk meta is cut short");
  *out = size_t((pos + 7) / 8);
  return PCO_B200_OK;
}
}  // namespace

PcoB200Error pco_b200_file_compressor_write_header(void* dst, size_t dst_cap, size_t* n_written) {
  if (dst_cap < 2) return fail(PCO_B200_IO, "failed to write whole buffer");
  static_cast<uint8_t*>(dst)[0] = 4;  // FormatVersion { major: 4, minor: 1 } (metadata/format_version.rs:30-34,87-91)
  static_cast<uint8_t*>(dst)[1] = 1;
  if (n_written) *n_written = 2;
  return PCO_B200_OK;
}

PcoB200Error pco_b200_file_decompressor_read_header(const void* src, size_t src_len, size_t* n_read) {
  const uint8_t* b = static_cast<const uint8_t*>(src);
  if (src_len < 1) return fail(PCO_B200_INSUFFICIENT_DATA, "empty wrapped header");
  const uint8_t major = b[0];
  if (major > 4) return fail(PCO_B200_CORRUPTION, "file's format version exceeds the max supported version");  // format_version.rs:60-72
  size_t used = 1;
  if (major >= 4) {  // the minor version byte exists from 4.0 on
    if (src_len < 2) return fail(PCO_B200_INSUFFICIENT_DATA, "wrapped header is cut short");
    used = 2;
  }
  if (major < 4) return fail(PCO_B200_UNSUPPORTED, "wrapped files older than format 4 are outside the GPU hot path");
  if (n_read) *n_read = used;
  return PCO_B200_OK;
}

PcoB200Error pco_b200_chunk_compressor_new(const void* nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig* config,
                                           PcoB200ChunkCompressor** out) {
  if (!out) return fail(PCO_B200_INVALID_ARGUMENT, "null output handle");
  *out = nullptr;
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  if (n == 0) return fail(PCO_B200_INVALID_ARGUMENT, "cannot compress empty chunk");  // chunk_compressor.rs:113-127
  PcoB200ChunkConfig cfg;
  if (config) cfg = *config;
  else { std::memset(&cfg, 0, sizeof(cfg)); cfg.compression_level = 8; }
  std::vector<uint64_t> pages;
  if (PcoB200Error e = n_per_page(cfg, n, &pages)) return e;
  auto cc = std::make_unique<PcoB200ChunkCompressor>();
  cc->n = n;
  const uint32_t lbits = nt_bits(dtype);
  size_t cap = 64;
  for (uint64_t pn : pages) cap += standalone_chunk_size_guarantee(lbits, size_t(pn)) + 8;
  cc->bytes.resize(cap);
  size_t written = 0, ilen = 0;
  std::vector<uint8_t> index(pco_b200_index_size_bound(n, pages.size()) + 64 * pages.size());
  // several pages: the pipeline runs them as the call's chunks with ONE set of bins trained on all of them
  const uint32_t flags = PCO_B200_CHUNKS_ONLY | (pages.size() > 1 ? PCO_B200_INTERNAL_SHARED_BINS : 0u);
  if (PcoB200Error e = compress_dispatch(nums, n, dtype, &cfg, false, cc->bytes.data(), cc->bytes.size(), &written, index.data(), index.size(), &ilen, flags,
                                         nullptr))
    return e;
  cc->bytes.resize(written);
  if (written < 4 || ilen < sizeof(IndexHeader)) return fail(PCO_B200_CUDA, "compressor returned a truncated chunk");
  IndexHeader ih;
  std::memcpy(&ih, index.data(), sizeof(ih));
  if (ih.n_chunks != pages.size() || ih.chunks_offset + ih.n_chunks * sizeof(IndexChunk) > ilen) return fail(PCO_B200_CUDA, "compressor returned an inconsistent page table");
  for (size_t p = 0; p < pages.size(); p++) {
    IndexChunk ic;
    std::memcpy(&ic, index.data() + ih.chunks_offset + p * sizeof(IndexChunk), sizeof(ic));
    cc->page_off.push_back(size_t(ic.chunk_offset));
    cc->page_n.push_back(size_t(pages[p]));
  }
  cc->page_off.push_back(written);
  if (PcoB200Error e = host_chunk_meta_len(cc->bytes.data() + 4, cc->page_off[1] - 4, dtype, &cc->meta_len)) return e;
  for (size_t p = 1; p < pages.size(); p++)  // shared bins: every page's emission repeats the chunk meta
    if (cc->page_off[p + 1] - cc->page_off[p] < 4 + cc->meta_len ||
        std::memcmp(cc->bytes.data() + 4, cc->bytes.data() + cc->page_off[p] + 4, cc->meta_len) != 0)
      return fail(PCO_B200_CUDA, "pages of one chunk came back with different chunk metas");
  *out = cc.release();
  return PCO_B200_OK;
}
void pco_b200_chunk_compressor_free(PcoB200ChunkCompressor* cc) { delete cc; }
size_t pco_b200_chunk_compressor_n_pages(const PcoB200ChunkCompressor* cc) { return cc ? cc->page_n.size() : 0; }
size_t pco_b200_chunk_compressor_page_n(const PcoB200ChunkCompressor* cc, size_t page_idx) {
  return (cc && page_idx < cc->page_n.size()) ? cc->page_n[page_idx] : 0;
}
size_t pco_b200_chunk_compressor_meta_size(const PcoB200ChunkCompressor* cc) { return cc ? cc->meta_len : 0; }
size_t pco_b200_chunk_compressor_page_size(const PcoB200ChunkCompressor* cc, size_t page_idx) {
  return (cc && page_idx < cc->page_n.size()) ? cc->page_off[page_idx + 1] - cc->page_off[page_idx] - 4 - cc->meta_len : 0;
}
PcoB200Error pco_b200_chunk_compressor_write_meta(const PcoB200ChunkCompressor* cc, void* dst, size_t dst_cap, size_t* n_written) {
  if (!cc) return fail(PCO_B200_INVALID_ARGUMENT, "null chunk compressor");
  if (dst_cap < cc->meta_len) return fail(PCO_B200_IO, "failed to write whole buffer");
  std::memcpy(dst, cc->bytes.data() + 4, cc->meta_len);
  if (n_written) *n_written = cc->meta_len;
  return PCO_B200_OK;
}
PcoB200Error pco_b200_chunk_compressor_write_page(const PcoB200ChunkCompressor* cc, size_t page_idx, void* dst, size_t dst_cap, size_t* n_written) {
  if (!cc) return fail(PCO_B200_INVALID_ARGUMENT, "null chunk compressor");
  if (page_idx >= cc->page_n.size())  // chunk_compressor.rs:661-666
    return fail(PCO_B200_INVALID_ARGUMENT, "page idx exceeds num pages (" + std::to_string(page_idx) + " >= " + std::to_string(cc->page_n.size()) + ")");
  const size_t begin = cc->page_off[page_idx] + 4 + cc->meta_len, len = cc->page_off[page_idx + 1] - begin;
  if (dst_cap < len) return fail(PCO_B200_IO, "failed to write whole buffer");
  std::memcpy(dst, cc->bytes.data() + begin, len);
  if (n_written) *n_written = len;
  return PCO_B200_OK;
}

PcoB200Error pco_b200_chunk_meta_size(const void* src, size_t src_len, unsigned char dtype, size_t* meta_len) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  size_t len = 0;
  if (PcoB200Error e = host_chunk_meta_len(static_cast<const uint8_t*>(src), src_len, dtype, &len)) return e;
  if (meta_len) *meta_len = len;
  return PCO_B200_OK;
}

PcoB200Error pco_b200_page_decompress(const void* chunk_meta, size_t meta_len, const void* page, size_t page_len, size_t page_n,
                                      unsigned char dtype, void* dst, size_t dst_len, PcoB200Progress* progress, size_t* bytes_read) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  if (page_n == 0 || page_n > (size_t(1) << 24)) return fail(PCO_B200_INVALID_ARGUMENT, "page n out of range");
  // PageDecompressor::read: dst must take whole batches or the rest of the page (page_decompressor.rs:200-206)
  if (dst_len % BATCH_N != 0 && dst_len < page_n)
    return fail(PCO_B200_INVALID_ARGUMENT, "num_dst's length must either be a multiple of 256 or be at least the count of numbers remaining");
  // one-chunk standalone file around the same bytes: header | type byte | n - 1 | meta | page | terminator
  std::vector<uint8_t> file = make_standalone_header(page_n, 0);
  file.push_back(dtype);
  const uint32_t nm1 = uint32_t(page_n - 1);
  file.push_back(uint8_t(nm1)); file.push_back(uint8_t(nm1 >> 8)); file.push_back(uint8_t(nm1 >> 16));
  const uint8_t* m = static_cast<const uint8_t*>(chunk_meta);
  const uint8_t* p = static_cast<const uint8_t*>(page);
  file.insert(file.end(), m, m + meta_len);
  file.insert(file.end(), p, p + page_len);
  file.push_back(0);
  PcoB200Progress prog{0, 0};
  if (PcoB200Error e = pco_b200_decompress_ex(file.data(), file.size(), dtype, dst, dst_len, &prog, nullptr, 0, 0, nullptr)) return e;
  prog.finished = prog.n_processed >= page_n ? 1 : 0;
  if (progress) *progress = prog;
  if (bytes_read) *bytes_read = page_len;
  return PCO_B200_OK;
}

#ifdef PCOB_DEC_TIMING
// experiment builds only: read and reset the decode kernel's region timers
int pco_b200_debug_dec_timing(unsigned long long* out16) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out16, g_dec_timing, sizeof(unsigned long long) * 16);
  unsigned long long z[16] = {0};
  cudaMemcpyToSymbol(g_dec_timing, z, sizeof(z));
  return 0;
}
#endif

#ifdef PCOB_ENC_TIMING
int pco_b200_debug_enc_timing(unsigned long long* out32) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out32, g_enc_timing, sizeof(unsigned long long) * 32);
  unsigned long long z[32] = {0};
  cudaMemcpyToSymbol(g_enc_timing, z, sizeof(z));
  return 0;
}
#endif

// ModeSpec::Auto for one chunk in host memory (mode_search.hpp); no device involved
PcoB200Error pco_b200_choose_mode(const void* nums, size_t n, unsigned char dtype, PcoB200ModeChoice* out) {
  if (!out || (!nums && n)) return fail(PCO_B200_INVALID_ARGUMENT, "null argument");
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_ARGUMENT, "unknown number type byte");
  if (n > (size_t(1) << 24)) return fail(PCO_B200_INVALID_ARGUMENT, "count may not exceed 16777216 per chunk");
  std::memset(out, 0, sizeof(*out));
  mode_search::Choice c;
  const bool is_float = nt_is_float(dtype), is_signed = nt_is_signed(dtype);
  switch (nt_bits(dtype)) {
    case 64: c = is_float ? mode_search::choose_float<double>(static_cast<const uint64_t*>(nums), n) : mode_search::choose_int<uint64_t>(static_cast<const uint64_t*>(nums), n, is_signed); break;
    case 32: c = is_float ? mode_search::choose_float<float>(static_cast<const uint32_t*>(nums), n) : mode_search::choose_int<uint32_t>(static_cast<const uint32_t*>(nums), n, is_signed); break;
    case 16: c = is_float ? mode_search::choose_float<mode_search::Half>(static_cast<const uint16_t*>(nums), n) : mode_search::choose_int<uint16_t>(static_cast<const uint16_t*>(nums), n, is_signed); break;
    default: c = mode_search::choose_int<uint8_t>(static_cast<const uint8_t*>(nums), n, is_signed); break;
  }
  out->mode_spec = c.kind == 1 ? PCO_B200_MODE_TRY_INT_MULT : c.kind == 2 ? PCO_B200_MODE_TRY_FLOAT_MULT : c.kind == 3 ? PCO_B200_MODE_TRY_FLOAT_QUANT : PCO_B200_MODE_CLASSIC;
  out->float_quant_k = c.k;
  out->float_mult_base = c.base;
  out->float_mult_inv_base = c.inv_base;
  out->int_mult_base = c.int_base;
  out->bits_saved_per_num = c.bits_saved_per_num;
  return PCO_B200_OK;
}

void pco_b200_profile_enable(int on) { profiler_enabled().store(on != 0); }
// Test hook for the host logic of the speculative index-free walk (no device involved): follow_chunk_chain over caller-made tables.
// Returns the number of verified chunks; their candidate indices go to `verified` (room for m), the position behind the last one to *next_pos.
size_t pco_b200_debug_follow_chain(const uint64_t* cand, const uint32_t* statuses, const uint64_t* ends, uint32_t m, uint64_t pos, uint64_t n0, uint64_t out_off,
                                   uint64_t dst_len, uint64_t src_len, uint32_t* verified, uint64_t* next_pos) {
  uint64_t p = pos;
  const std::vector<uint32_t> chain = follow_chunk_chain(cand, statuses, ends, m, pos, n0, out_off, dst_len, src_len, &p);
  for (size_t i = 0; i < chain.size(); i++) verified[i] = chain[i];
  if (next_pos) *next_pos = p;
  return chain.size();
}
int pco_b200_zero_copy(int mask) { return mask < 0 ? zero_copy_mask().load() : zero_copy_mask().exchange(mask & 7); }
// Frees the calling thread's device scratch (a worker thread calls this before it exits; the buffers are otherwise kept for the
// thread's next call).
void pco_b200_thread_release(void) {
  Context& c = ctx();
  if (c.initialized && c.device_ok) release_buffers(c);
  readback_bounce().release();
}
// Which decode instantiation served the chunks of the last decode launch: counts[k] = chunks of class k
// (1, 2: decode_kernel<L, 1 / 2>; 3, 4: decode_narrow_kernel order 0 / 1).  Returns the number of chunks.
int pco_b200_profile_chunk_classes(unsigned* counts8) {
  Context& c = ctx();
  for (int i = 0; i < 8; i++) counts8[i] = 0;
  if (!c.device_ok || c.last_decode_chunks == 0 || !c.d_cls) return 0;
  std::vector<uint8_t> cls(c.last_decode_chunks);
  if (cudaMemcpy(cls.data(), c.d_cls, cls.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  for (uint8_t k : cls) counts8[(k & 0x7f) < 8 ? (k & 0x7f) : 0]++;
  return int(cls.size());
}
// Copies "name=ms;name=ms;..." of the last finished call into buf; returns the number of spans.
int pco_b200_profile_last(char* buf, size_t cap) {
  std::string s;
  for (auto& kv : profiler().last) s += kv.first + "=" + std::to_string(kv.second) + ";";
  if (cap) {
    size_t n = std::min(cap - 1, s.size());
    std::memcpy(buf, s.data(), n);
    buf[n] = 0;
  }
  return int(profiler().last.size());
}

size_t pco_b200_index_size_bound(size_t n, size_t n_chunks_hint) {
  size_t chunks = n_chunks_hint + 2;
  size_t batches = n / BATCH_N + 2 * chunks;
  return sizeof(IndexHeader) + chunks * sizeof(IndexChunk) + batches * MAX_VARS * sizeof(BatchEntry) + 16 * chunks + 64;
}

// Batched decompress of chunks whose byte offsets the caller knows (SURVEY.md 8b "decompress_chunks"): a container that
// keeps chunk / page offsets beside the bytes - pco's wrapped use case, a sharded writer's offset table - needs no side
// index.  The per-batch index is built on the device by one tANS walk per chunk, ALL CHUNKS IN PARALLEL (the standalone
// format's single serial cursor only exists because chunk lengths are not in the stream), then the ordinary decode runs.
PcoB200Error pco_b200_decompress_chunks(const void* compressed, size_t compressed_len, unsigned char dtype, const uint64_t* chunk_offsets,
                                        const uint32_t* chunk_ns, size_t n_chunks, void* dst, size_t dst_len, size_t* n_written, uint32_t flags,
                                        void* cuda_stream) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte: " + std::to_string(dtype));
  if (n_written) *n_written = 0;
  if (n_chunks == 0) return PCO_B200_OK;
  if (!chunk_offsets || !chunk_ns) return fail(PCO_B200_INVALID_ARGUMENT, "chunk_offsets and chunk_ns are required");
  if (n_chunks > 0x7fffffffull) return fail(PCO_B200_INVALID_ARGUMENT, "too many chunks");
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  const bool src_dev = flags & PCO_B200_SRC_ON_DEVICE, dst_dev = flags & PCO_B200_DST_ON_DEVICE;
  const size_t elem = nt_bits(dtype) / 8;
  // a standalone file (magic present) carries the format version and the uniform type; bare chunks are format 4.1
  uint32_t format_major = 4, uniform_type = 0;
  {
    uint8_t head[32] = {0};
    const size_t avail = std::min<size_t>(compressed_len, sizeof(head));
    if (avail) {
      if (src_dev) { PCOB_CUDA_TRY(cudaMemcpyAsync(head, compressed, avail, cudaMemcpyDeviceToHost, stream)); PCOB_CUDA_TRY(cudaStreamSynchronize(stream)); }
      else std::memcpy(head, compressed, avail);
    }
    static const uint8_t MAGIC[4] = {112, 99, 111, 33};
    if (avail >= 4 && std::memcmp(head, MAGIC, 4) == 0 && chunk_offsets[0] >= 4) {
      StandaloneHeader hdr;
      if (PcoB200Error e = parse_standalone_header(head, avail, compressed_len, &hdr)) return e;
      format_major = hdr.format_major;
      uniform_type = hdr.uniform_type;
    }
  }
  // index skeleton: chunk records from the caller's table, room for 2 vars of entries per chunk
  const uint64_t chunks_offset = sizeof(IndexHeader);
  std::vector<IndexChunk> recs(n_chunks);
  uint64_t off = (chunks_offset + uint64_t(n_chunks) * sizeof(IndexChunk) + 15) & ~uint64_t(15), out_off = 0;
  for (size_t i = 0; i < n_chunks; i++) {
    if (chunk_offsets[i] >= compressed_len) return fail(PCO_B200_INVALID_ARGUMENT, "chunk offset " + std::to_string(i) + " lies outside the buffer");
    if (chunk_ns[i] == 0 || chunk_ns[i] > (1u << 24)) return fail(PCO_B200_INVALID_ARGUMENT, "chunk " + std::to_string(i) + ": count must be 1..2^24");
    recs[i].chunk_offset = chunk_offsets[i];
    recs[i].n = chunk_ns[i];
    recs[i].n_vars = 0;
    recs[i].entries_offset = off;
    recs[i].out_offset = out_off;
    off += (uint64_t(MAX_VARS) * n_batches_of(chunk_ns[i]) * sizeof(BatchEntry) + 15) & ~uint64_t(15);
    out_off += chunk_ns[i];
  }
  const uint64_t n_total = out_off;
  if (n_total > dst_len) return fail(PCO_B200_INVALID_ARGUMENT, "dst holds " + std::to_string(dst_len) + " numbers, the chunks " + std::to_string(n_total));
  const uint8_t* d_src;
  if (src_dev) d_src = static_cast<const uint8_t*>(compressed);
  else {
    PCOB_CUDA_TRY(c.src.reserve(compressed_len + 16));
    PCOB_CUDA_TRY(copy_sliced(c.src.p, compressed, compressed_len, cudaMemcpyHostToDevice, stream));
    d_src = c.src.as<uint8_t>();
  }
  FileParams fp{d_src, compressed_len, dtype, uniform_type, format_major};
  PCOB_CUDA_TRY(c.index.reserve(off + 64));
  uint8_t* d_index = c.index.as<uint8_t>();
  PCOB_CUDA_TRY(cudaMemcpyAsync(d_index + chunks_offset, recs.data(), n_chunks * sizeof(IndexChunk), cudaMemcpyHostToDevice, stream));
  PCOB_CUDA_TRY(c.statuses.reserve((n_chunks + 1) * sizeof(uint32_t)));
  PCOB_CUDA_TRY(c.misc.reserve(sizeof(WalkResult)));
  PCOB_CUDA_TRY(cudaMemsetAsync(c.statuses.p, 0xff, n_chunks * sizeof(uint32_t), stream));
  profiler().begin("walk_kernel", stream);
  walk_kernel<SMALL_MAX_SIZE_LOG><<<uint32_t(n_chunks), WALK_THREADS, sizeof(WalkSmem<SMALL_MAX_SIZE_LOG>), stream>>>(
      fp, d_index, chunks_offset, uint32_t(n_chunks), 0, off, 0, 0, ~uint64_t(0), c.statuses.as<uint32_t>(), c.misc.as<WalkResult>(), 0);
  profiler().end(stream);
  PCOB_CUDA_TRY(cudaGetLastError());
  {
    std::vector<uint32_t> st(n_chunks);
    PCOB_CUDA_TRY(cudaMemcpyAsync(st.data(), c.statuses.p, n_chunks * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
    for (size_t i = 0; i < n_chunks; i++)
      if (st[i] != ST_OK) { profiler().resolve(); return status_to_error(st[i], ("chunk " + std::to_string(i)).c_str()); }
  }
  void* d_out = dst;
  if (!dst_dev) {
    PCOB_CUDA_TRY(c.out.reserve(n_total * elem + 64));
    d_out = c.out.p;
  }
  PcoB200Error e = launch_decode(c, fp, d_index, off, chunks_offset, uint32_t(n_chunks), d_out, dst_dev ? uint64_t(dst_len) : n_total, stream);
  profiler().resolve();
  if (e != PCO_B200_OK) return e;
  if (!dst_dev && n_total) {
    PCOB_CUDA_TRY(copy_sliced(dst, d_out, n_total * elem, cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
  }
  if (n_written) *n_written = size_t(n_total);
  return PCO_B200_OK;
}

PcoB200Error pco_b200_build_index(const void* compressed, size_t compressed_len, unsigned char dtype, void* index, size_t index_cap,
                                  size_t* index_len, uint32_t flags, void* cuda_stream) {
  if (!nt_valid(dtype)) return fail(PCO_B200_INVALID_TYPE, "unknown number type byte");
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  const bool src_dev = flags & PCO_B200_SRC_ON_DEVICE;
  uint8_t head[32] = {0};
  size_t avail = std::min<size_t>(compressed_len, sizeof(head));
  if (avail) {
    if (src_dev) { PCOB_CUDA_TRY(cudaMemcpyAsync(head, compressed, avail, cudaMemcpyDeviceToHost, stream)); PCOB_CUDA_TRY(cudaStreamSynchronize(stream)); }
    else std::memcpy(head, compressed, avail);
  }
  StandaloneHeader hdr;
  if (PcoB200Error e = parse_standalone_header(head, avail, compressed_len, &hdr)) return e;
  const uint8_t* d_src;
  if (src_dev) d_src = static_cast<const uint8_t*>(compressed);
  else {
    PCOB_CUDA_TRY(c.src.reserve(compressed_len + 16));
    PCOB_CUDA_TRY(copy_sliced(c.src.p, compressed, compressed_len, cudaMemcpyHostToDevice, stream));
    d_src = c.src.as<uint8_t>();
  }
  FileParams fp{d_src, compressed_len, dtype, hdr.uniform_type, hdr.format_major};
  if (index_cap < sizeof(IndexHeader) + sizeof(IndexChunk) + 64) return fail(PCO_B200_IO, "index buffer too small");
  // Split the caller's capacity: chunk records sized from a lower bound on chunk bytes, the rest for entries.
  uint64_t max_chunks = std::min<uint64_t>(uint64_t(compressed_len) / 5 + 2, (index_cap - sizeof(IndexHeader)) / (4 * sizeof(IndexChunk)));
  max_chunks = std::max<uint64_t>(1, std::min<uint64_t>(max_chunks, 0x7fffffffull));
  const uint64_t chunks_offset = sizeof(IndexHeader);
  uint64_t entries_begin = (chunks_offset + max_chunks * sizeof(IndexChunk) + 15) & ~uint64_t(15);
  if (entries_begin > index_cap) return fail(PCO_B200_IO, "index buffer too small");
  PCOB_CUDA_TRY(c.index.reserve(index_cap));
  PCOB_CUDA_TRY(c.misc.reserve(sizeof(WalkResult)));
  uint8_t* d_index = c.index.as<uint8_t>();
  walk_kernel<12><<<1, WALK_THREADS, sizeof(WalkSmem<12>), stream>>>(fp, d_index, chunks_offset, uint32_t(max_chunks), entries_begin, index_cap, hdr.first_chunk_byte,
                                                    0, ~uint64_t(0), nullptr, c.misc.as<WalkResult>(), 1);
  PCOB_CUDA_TRY(cudaGetLastError());
  WalkResult res;
  PCOB_CUDA_TRY(cudaMemcpyAsync(&res, c.misc.p, sizeof(res), cudaMemcpyDeviceToHost, stream));
  PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
  if (res.status == ST_INDEX_FULL) return fail(PCO_B200_IO, "index buffer too small");
  if (res.status != ST_TERMINATOR) return status_to_error(res.status, ("chunk " + std::to_string(res.n_chunks)).c_str());
  IndexHeader ih;
  std::memset(&ih, 0, sizeof(ih));
  ih.magic = INDEX_MAGIC;
  ih.version = 1;
  ih.n_chunks = res.n_chunks;
  ih.n_total = res.n_total;
  ih.file_len = compressed_len;
  ih.chunks_offset = chunks_offset;
  ih.end_byte = res.next_byte;
  size_t used = std::max<uint64_t>(res.entries_end, entries_begin);
  std::memcpy(index, &ih, sizeof(ih));
  if (used > sizeof(ih)) {
    PCOB_CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t*>(index) + sizeof(ih), d_index + sizeof(ih), used - sizeof(ih), cudaMemcpyDeviceToHost, stream));
    PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
  }
  if (index_len) *index_len = used;
  return PCO_B200_OK;
}

// ---------------------------------------------------------------------------
// Sharded writers (SURVEY.md 8e): device buffers other ranks can map, and the page gather (gather_kernels.cuh)
// ---------------------------------------------------------------------------
PcoB200Error pco_b200_ipc_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64) {
  if (!dev_ptr || !handle64) return fail(PCO_B200_INVALID_ARGUMENT, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the handle travels as 64 bytes");
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  void* p = nullptr;
  PCOB_CUDA_TRY(cudaMalloc(&p, bytes + 64));
  cudaIpcMemHandle_t h;
  cudaError_t ce = cudaIpcGetMemHandle(&h, p);
  if (ce != cudaSuccess) { cudaFree(p); return cuda_fail(ce, "cudaIpcGetMemHandle"); }
  std::memcpy(handle64, &h, 64);
  *dev_ptr = p;
  return PCO_B200_OK;
}
PcoB200Error pco_b200_ipc_open(const unsigned char* handle64, void** dev_ptr) {
  if (!dev_ptr || !handle64) return fail(PCO_B200_INVALID_ARGUMENT, "null argument");
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle64, 64);
  PCOB_CUDA_TRY(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return PCO_B200_OK;
}
PcoB200Error pco_b200_ipc_close(void* dev_ptr) {
  if (dev_ptr) PCOB_CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr));
  return PCO_B200_OK;
}
PcoB200Error pco_b200_ipc_free(void* dev_ptr) {
  if (dev_ptr) PCOB_CUDA_TRY(cudaFree(dev_ptr));
  return PCO_B200_OK;
}

PcoB200Error pco_b200_chunk_sizes(const void* index_dev, size_t index_len, uint64_t* sizes_dev, size_t n_chunks, void* cuda_stream) {
  if (n_chunks == 0) return PCO_B200_OK;
  if (!index_dev || !sizes_dev) return fail(PCO_B200_INVALID_ARGUMENT, "null argument");
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  PCOB_CUDA_TRY(c.misc.reserve(256));
  uint32_t* d_err = c.misc.as<uint32_t>() + 32;
  PCOB_CUDA_TRY(cudaMemsetAsync(d_err, 0, 4, stream));
  chunk_sizes_kernel<<<uint32_t(std::min<size_t>((n_chunks + 255) / 256, 1024)), 256, 0, stream>>>(static_cast<const uint8_t*>(index_dev), index_len, sizes_dev, uint32_t(n_chunks), d_err);
  PCOB_CUDA_TRY(cudaGetLastError());
  return PCO_B200_OK;  // asynchronous: a malformed index shows up as sizes the gather rejects (file length over capacity) or as d_err in pco_b200_gather_pages
}

PcoB200Error pco_b200_gather_pages(const void* chunks_dev, const uint64_t* all_sizes_dev, uint32_t world, uint32_t rank, size_t n_local, size_t n_total_numbers,
                                   unsigned char uniform_type, void* const* peer_files, size_t file_cap, uint64_t* file_len_dev, uint32_t max_ctas, void* cuda_stream) {
  if (world == 0 || world > uint32_t(GATHER_MAX_WORLD) || rank >= world) return fail(PCO_B200_INVALID_ARGUMENT, "world must be 1..16 and rank < world");
  if (!chunks_dev || !all_sizes_dev || !peer_files || !file_len_dev) return fail(PCO_B200_INVALID_ARGUMENT, "null argument");
  if (n_local > 0x7fffffffull) return fail(PCO_B200_INVALID_ARGUMENT, "too many chunks");
  Context& c = ctx();
  if (PcoB200Error e = ensure_device(c)) return e;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  GatherPeers peers;
  for (uint32_t r = 0; r < uint32_t(GATHER_MAX_WORLD); r++) peers.file[r] = r < world ? static_cast<uint8_t*>(peer_files[r]) : nullptr;
  for (uint32_t r = 0; r < world; r++)
    if (!peers.file[r]) return fail(PCO_B200_INVALID_ARGUMENT, "peer file buffer " + std::to_string(r) + " is null");
  const std::vector<uint8_t> header = make_standalone_header(n_total_numbers, uniform_type);
  // scratch: [src_off | dst_off] (2 x n_local u64), header bytes, error word; owned by the calling thread's context and reused
  const size_t off_bytes = 2 * n_local * sizeof(uint64_t);
  PCOB_CUDA_TRY(c.gather.reserve(off_bytes + 256));
  uint64_t* d_src_off = c.gather.as<uint64_t>();
  uint64_t* d_dst_off = d_src_off + n_local;
  uint8_t* d_header = c.gather.as<uint8_t>() + off_bytes;
  uint32_t* d_err = reinterpret_cast<uint32_t*>(d_header + 128);
  PCOB_CUDA_TRY(cudaMemcpyAsync(d_header, header.data(), header.size(), cudaMemcpyHostToDevice, stream));
  PCOB_CUDA_TRY(cudaMemsetAsync(d_err, 0, 4, stream));
  c.gather_err = d_err;
  gather_offsets_kernel<<<1, 1024, 0, stream>>>(all_sizes_dev, world, rank, uint32_t(n_local), header.size(), d_src_off, d_dst_off, file_len_dev);
  const uint32_t ctas = std::max(1u, max_ctas ? max_ctas : uint32_t(c.sm_count));
  // (no profiler span here: the gather is meant to run asynchronously beside the caller's next calls, whose span resolution would wait for it)
  push_pages_kernel<<<ctas, GATHER_THREADS, 0, stream>>>(static_cast<const uint8_t*>(chunks_dev), all_sizes_dev, d_src_off, d_dst_off, file_len_dev, peers, world, rank,
                                                        uint32_t(n_local), file_cap, d_header, uint32_t(header.size()), d_err);
  PCOB_CUDA_TRY(cudaGetLastError());
  return PCO_B200_OK;  // asynchronous on `stream`; pco_b200_gather_status reports a file buffer that was too small
}

// Blocks until the calling thread's last pco_b200_gather_pages has finished on `cuda_stream` and reports it: PCO_B200_IO when a
// file buffer was too small for the gathered file, PCO_B200_INVALID_ARGUMENT for a malformed side index.
PcoB200Error pco_b200_gather_status(void* cuda_stream) {
  Context& c = ctx();
  if (!c.gather_err) return PCO_B200_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  uint32_t st = 0;
  PCOB_CUDA_TRY(cudaMemcpyAsync(&st, c.gather_err, 4, cudaMemcpyDeviceToHost, stream));
  PCOB_CUDA_TRY(cudaStreamSynchronize(stream));
  if (st == ST_INSUFFICIENT_DATA) return fail(PCO_B200_IO, "failed to write whole buffer: a rank's file buffer is smaller than the gathered file");
  if (st != ST_OK) return status_to_error(st, "the page gather");
  return PCO_B200_OK;
}

}  // extern "C"
