/* pco_b200.h — extensions to the reference C ABI (cpcodec.h) that the three reference
 * functions cannot express: explicit mode/delta/paging specs, the non-uniform header
 * flavour, partial-destination decompression, the wrapped chunk/page API, device-resident
 * buffers on a caller stream, and the per-batch side index.
 *
 * Every entry point is plain C: pointers, sizes and POD structs; no torch / CUDA types in
 * signatures (a cudaStream_t travels as void*).  Each declaration cites the reference
 * interface it stands in for.  All functions are thread-safe; the library keeps only a
 * mutex-guarded cache of device scratch memory between calls.
 */
#ifndef PCO_B200_H
#define PCO_B200_H

#include <stddef.h>
#include <stdint.h>

#include "cpcodec.h"

#if defined(__cplusplus)
extern "C" {
#endif

/* pco::errors::ErrorKind (pco/src/errors.rs:8-24), plus two kinds the CPU reference cannot
 * produce: a missing/failed CUDA device, and a format feature the GPU path does not decode. */
typedef enum PcoB200Error {
  PCO_B200_OK = 0,
  PCO_B200_CORRUPTION = 1,
  PCO_B200_INSUFFICIENT_DATA = 2,
  PCO_B200_INVALID_ARGUMENT = 3,
  PCO_B200_IO = 4,          /* destination buffer too small (std::io::ErrorKind::WriteZero) */
  PCO_B200_INVALID_TYPE = 5,
  PCO_B200_CUDA = 6,        /* no device / launch failure: this library has no CPU fallback */
  PCO_B200_UNSUPPORTED = 7  /* valid pco, but outside the GPU hot path (see DESIGN.md) */
} PcoB200Error;

/* pco::ModeSpec (pco/src/chunk_config.rs:15-51) */
enum { PCO_B200_MODE_AUTO = 0, PCO_B200_MODE_CLASSIC = 1, PCO_B200_MODE_TRY_FLOAT_MULT = 2,
       PCO_B200_MODE_TRY_FLOAT_QUANT = 3, PCO_B200_MODE_TRY_INT_MULT = 4, PCO_B200_MODE_TRY_DICT = 5 };
/* pco::DeltaSpec (pco/src/chunk_config.rs:63-109) */
enum { PCO_B200_DELTA_AUTO = 0, PCO_B200_DELTA_NOOP = 1, PCO_B200_DELTA_TRY_CONSECUTIVE = 2,
       PCO_B200_DELTA_TRY_LOOKBACK = 3, PCO_B200_DELTA_TRY_CONV1 = 4 };
/* pco::PagingSpec (pco/src/chunk_config.rs:114-125) */
enum { PCO_B200_PAGING_EQUAL_PAGES_UP_TO = 0, PCO_B200_PAGING_EXACT = 1 };

/* pco::ChunkConfig (pco/src/chunk_config.rs:193-224) as a POD. */
typedef struct PcoB200ChunkConfig {
  uint32_t compression_level;   /* 0..12, default 8 */
  uint32_t mode_spec;           /* PCO_B200_MODE_* */
  double float_mult_base;       /* TryFloatMult(base) */
  uint64_t int_mult_base;       /* TryIntMult(base) */
  uint32_t float_quant_k;       /* TryFloatQuant(k) */
  uint32_t delta_spec;          /* PCO_B200_DELTA_* */
  uint32_t delta_order;         /* TryConsecutive(order) / TryConv1(order) */
  uint32_t paging_spec;         /* PCO_B200_PAGING_* */
  uint64_t max_page_n;          /* EqualPagesUpTo(n); 0 -> 2^18 */
  const uint64_t *exact_page_ns;/* Exact(vec) */
  uint64_t n_exact_pages;
  uint32_t enable_8_bit;
  uint32_t reserved;
} PcoB200ChunkConfig;

/* pco::Progress (pco/src/progress.rs:3-11) */
typedef struct PcoB200Progress {
  size_t n_processed;
  int finished;
} PcoB200Progress;

/* Buffer-location flags for the *_ex entry points. */
enum { PCO_B200_SRC_ON_DEVICE = 1u, PCO_B200_DST_ON_DEVICE = 2u, PCO_B200_INDEX_ON_DEVICE = 4u,
       /* compress only: emit the chunks (type byte, n, meta, page) back to back with no standalone header and no
        * terminator -- the unit a rank contributes when chunks are sharded across GPUs (SURVEY.md §8e) */
       PCO_B200_CHUNKS_ONLY = 8u };

/* Message of the last error raised on the calling thread (pco::errors::PcoError::message). */
const char *pco_b200_last_error_message(void);
/* 1 if a usable sm_100 device is present. */
int pco_b200_device_available(void);

/* pco::standalone::simple_decompress_into (pco/src/standalone/simple.rs:100-143): never errors on a
 * short or long dst; decodes whole 256-batches then one scratch batch into a short dst. */
PcoB200Error pco_b200_simple_decompress_into(const void *compressed, size_t compressed_len, unsigned char dtype,
                                             void *dst, size_t dst_len, PcoB200Progress *progress);

/* As above, with buffers optionally resident in HBM (flags), work enqueued on `cuda_stream`
 * (NULL = default stream; the call returns after the stream work completes), and an optional
 * side index (`index`, `index_len` bytes; NULL = walk the tANS stream on the device first).
 * The side index is metadata *beside* the bit-exact .pco bytes (docs/format.md:34-38). */
PcoB200Error pco_b200_decompress_ex(const void *compressed, size_t compressed_len, unsigned char dtype, void *dst,
                                    size_t dst_len, PcoB200Progress *progress, const void *index, size_t index_len,
                                    uint32_t flags, void *cuda_stream);

/* Stream-ordered decompress of a file whose bytes, side index and destination all live in device memory (no reference
 * counterpart).  The call only enqueues work on `cuda_stream`: no device-to-host copy, no synchronisation, no allocation, so a
 * caller can keep issuing work on the same thread and can capture the call in a CUDA graph.  The caller declares n_chunks and
 * n_total (what the compress that wrote the index reported) and passes a workspace of at least
 * pco_b200_decompress_async_workspace_size(n_total, n_chunks, dtype) bytes that no other call uses while this one runs.
 * The return value only reports the arguments: PCO_B200_INVALID_TYPE for an unknown dtype, PCO_B200_INVALID_ARGUMENT for a null
 * pointer, n_chunks == 0, dst_len < n_total, an index shorter than its chunk table or not 8-byte aligned, or a workspace that is
 * too small; PCO_B200_CUDA without a device or for a launch failure.  What the device finds lands in *d_result (device memory)
 * when the stream reaches it: `status` is the PcoB200Error pco_b200_decompress_ex returns for the same bytes, `first_bad_chunk`
 * the lowest failing chunk (0xffffffff when the file header or the side index failed, or nothing did).  Files the fast kernels
 * decline (Dict, Lookback, Conv1, tANS tables over 2^10 states) report PCO_B200_UNSUPPORTED: this path has no cold fallback.
 * The first call on a thread (and on a device) does one-time set-up that cannot be captured; call
 * pco_b200_decompress_async_prepare(dtype) before capturing. */
typedef struct PcoB200AsyncResult {
  uint32_t status;          /* PcoB200Error */
  uint32_t first_bad_chunk;
  uint64_t n_total;         /* numbers the file holds (= numbers written when status is PCO_B200_OK) */
  uint32_t finished;        /* 1: the whole file was decoded (pco::Progress::finished) */
  uint32_t reserved;
} PcoB200AsyncResult;
size_t pco_b200_decompress_async_workspace_size(size_t n_total, size_t n_chunks, unsigned char dtype);
PcoB200Error pco_b200_decompress_async_prepare(unsigned char dtype);
PcoB200Error pco_b200_decompress_async(const void *d_src, size_t src_len, unsigned char dtype, const void *d_index, size_t index_len,
                                       size_t n_chunks, size_t n_total, void *d_dst, size_t dst_len, void *d_workspace,
                                       size_t workspace_len, PcoB200AsyncResult *d_result, void *cuda_stream);

/* pco::standalone::simple_compress (pco/src/standalone/simple.rs:58-91): header carries uniform type 0.
 * config may be NULL (pco::ChunkConfig::default()).  Fails with PCO_B200_IO if dst is too small. */
PcoB200Error pco_b200_simple_compress(const void *nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig *config,
                                      void *dst, size_t dst_cap, size_t *n_written);
/* pco::standalone::simple_compress_into (pco/src/standalone/simple.rs:22-48): header carries the number type. */
PcoB200Error pco_b200_simple_compress_into(const void *nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig *config,
                                           void *dst, size_t dst_cap, size_t *n_written);
/* Full-control compress: header flavour (uniform_type_header), optional side index output
 * (index_cap >= pco_b200_index_size_bound(n, n_chunks)), device-resident buffers and stream. */
PcoB200Error pco_b200_compress_ex(const void *nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig *config,
                                  int uniform_type_header, void *dst, size_t dst_cap, size_t *n_written, void *index,
                                  size_t index_cap, size_t *index_len, uint32_t flags, void *cuda_stream);

/* Batched decompress without a side index, for callers that know where their chunks are (SURVEY.md 8b; no reference counterpart:
 * the reference decodes chunk after chunk, pco/src/standalone/decompressor.rs:270-273).  `compressed` holds n_chunks standalone
 * chunks (type byte, 24-bit n - 1, chunk meta, page) at byte offsets chunk_offsets[i] - a standalone file, or the bare chunks
 * that PCO_B200_CHUNKS_ONLY emits; chunk_ns[i] = numbers in chunk i.  The numbers land back to back in dst (dst_len >= sum of
 * chunk_ns).  The per-batch index is built on the device, one tANS walk per chunk, all chunks in parallel.  A count that does not
 * match the chunk's own header is PCO_B200_INVALID_ARGUMENT. */
PcoB200Error pco_b200_decompress_chunks(const void *compressed, size_t compressed_len, unsigned char dtype,
                                        const uint64_t *chunk_offsets, const uint32_t *chunk_ns, size_t n_chunks, void *dst,
                                        size_t dst_len, size_t *n_written, uint32_t flags, void *cuda_stream);

/* Build the side index of a standalone file (one serial tANS walk per chunk on the device).
 * index_cap >= pco_b200_index_size_bound(n_total, 2). */
size_t pco_b200_index_size_bound(size_t n, size_t n_chunks_hint);
PcoB200Error pco_b200_build_index(const void *compressed, size_t compressed_len, unsigned char dtype, void *index,
                                  size_t index_cap, size_t *index_len, uint32_t flags, void *cuda_stream);

/* ModeSpec::Auto as the reference resolves it for ONE chunk of numbers in HOST memory (pco/src/data_types/unsigned.rs:28-35,
 * pco/src/data_types/float.rs:70-98: int_mult::choose_base for integers; Classic vs FloatMult vs FloatQuant bids for f32 / f64 on the
 * sample of pco/src/sampling.rs:62-103).  Host-only planner logic: needs no device, reads ~n/40 numbers.  out->mode_spec is a
 * PCO_B200_MODE_* value with its parameter in the matching field, ready to be pasted into a PcoB200ChunkConfig; FloatMult also
 * reports the inverse the reference's splitter would multiply by (snapping to 1/100 etc. makes it differ from 1/base in the last bit,
 * which only changes the secondary latents' values, never validity).  f16 is searched in the half crate's arithmetic like the
 * reference does; a FloatMult answer for f16 is the reference's choice, but the GPU path has no f16 FloatMult kernel (PCO_B200_UNSUPPORTED). */
typedef struct PcoB200ModeChoice {
  uint32_t mode_spec;
  uint32_t float_quant_k;
  double float_mult_base;
  double float_mult_inv_base;
  uint64_t int_mult_base;
  double bits_saved_per_num; /* the winning bid's estimate (0 for Classic and IntMult) */
} PcoB200ModeChoice;
PcoB200Error pco_b200_choose_mode(const void *nums, size_t n, unsigned char dtype, PcoB200ModeChoice *out);

/* Measurement hooks (no reference counterpart): when enabled, every kernel launched by the next call is bracketed by
 * CUDA events on the launching stream; pco_b200_profile_last returns "kernel=milliseconds;..." for the last call. */
void pco_b200_profile_enable(int on);
int pco_b200_profile_last(char *buf, size_t cap);
/* Threading: the library keeps one scratch context per calling host thread (device buffers grown on demand and reused by that
 * thread's next call), so calls from different threads - each with its own cudaStream_t - run concurrently, e.g. compress of
 * chunk group g + 1 on one thread while group g decompresses on another (both PCIe directions busy).  A worker thread that is
 * about to exit returns its device scratch with pco_b200_thread_release(). */
void pco_b200_thread_release(void);
/* Page-locked host buffers in place ("zero copy"): with bit 0 set, pco_b200_compress_ex (explicit Classic configs) reads a HOST `nums`
 * that is page-locked (cudaHostAlloc / cudaHostRegister, e.g. torch pin_memory) straight over PCIe in its one pass over the input; with
 * bit 1 set, pco_b200_decompress_ex (side-index path) has the decode kernels store into a page-locked HOST `dst` directly; with bit 2
 * set, pco_b200_compress_ex has the bit-pack kernel store the file into a page-locked HOST `dst` directly.  No staging
 * buffer in HBM and no copy-engine transfer for those streams; pageable buffers take the staged path whatever the mask says.  The mask is
 * process-wide; the call returns the previous one (a negative argument only reads it).  Environment: PCOB200_ZEROCOPY. */
int pco_b200_zero_copy(int mask);
/* Host logic of the index-free decompressor, exposed for tests (needs no device): among `m` sorted candidate chunk starts with the
 * status and end position a speculative walk gave each, follow the chain of real chunks from `pos` (a chunk is real when a verified
 * chunk ends on it).  Returns how many were verified; their candidate indices in `verified[0..]`, the position behind the last in *next_pos. */
size_t pco_b200_debug_follow_chain(const uint64_t *cand, const uint32_t *statuses, const uint64_t *ends, uint32_t m, uint64_t pos, uint64_t n0,
                                   uint64_t out_off, uint64_t dst_len, uint64_t src_len, uint32_t *verified, uint64_t *next_pos);
/* counts8[k] = chunks of the last decode launch served by decode class k (1, 2: general kernel with 1 / 2 latent vars;
 * 3, 4: narrow kernel, delta order 0 / 1); returns the number of chunks. */
int pco_b200_profile_chunk_classes(unsigned *counts8);

/* ---- sharded writers (no reference counterpart; SURVEY.md 8e): chunk c of the logical standalone file is compressed on rank
 * c mod G (PCO_B200_CHUNKS_ONLY); the page gather then leaves the WHOLE file - header | chunk_0 | chunk_1 | ... | 0x00, byte-identical
 * to a single-GPU / reference file of the same numbers (pco/src/standalone/simple.rs:62-91, compressor.rs:157) - in every rank's file
 * buffer.  The ranks' GPUs do the exchange themselves: a device-side scan of all ranks' chunk sizes gives every chunk's file offset
 * and each rank stores its chunks into every rank's buffer over NVLink (peer memory mapped through cudaIpc handles; no host copy,
 * no size on the host).  One process per GPU; handles are exchanged once by whatever the host uses for rendezvous. */
/* a device buffer other processes can map, and its 64-byte handle */
PcoB200Error pco_b200_ipc_alloc(size_t bytes, void **dev_ptr, unsigned char *handle64);
PcoB200Error pco_b200_ipc_open(const unsigned char *handle64, void **dev_ptr); /* map another rank's buffer (peer access is enabled on demand) */
PcoB200Error pco_b200_ipc_close(void *dev_ptr);
PcoB200Error pco_b200_ipc_free(void *dev_ptr);
/* sizes_dev[i] = bytes of chunk i of a CHUNKS_ONLY compress, from its side index (both on the device; asynchronous on cuda_stream) */
PcoB200Error pco_b200_chunk_sizes(const void *index_dev, size_t index_len, uint64_t *sizes_dev, size_t n_chunks, void *cuda_stream);
/* chunks_dev: this rank's chunk bytes back to back (+ 16 readable bytes of slack); all_sizes_dev[r * n_local + i]: bytes of rank r's
 * i-th chunk = chunk i * world + r of the file (0 where a rank has fewer chunks), e.g. one all-gather of the pco_b200_chunk_sizes
 * outputs; peer_files[r]: rank r's file buffer as mapped in this process (file_cap bytes each; peer_files[rank] is this rank's own);
 * file_len_dev: receives the file length; max_ctas bounds the copy kernel's grid (0 = one CTA per SM) so that it can run beside
 * other work.  Asynchronous on cuda_stream; pco_b200_gather_status waits for it and reports a buffer that was too small. */
PcoB200Error pco_b200_gather_pages(const void *chunks_dev, const uint64_t *all_sizes_dev, uint32_t world, uint32_t rank, size_t n_local, size_t n_total_numbers,
                                   unsigned char uniform_type, void *const *peer_files, size_t file_cap, uint64_t *file_len_dev, uint32_t max_ctas,
                                   void *cuda_stream);
PcoB200Error pco_b200_gather_status(void *cuda_stream);

/* ---- wrapped format (pco/src/wrapped/: FileCompressor / ChunkCompressor / FileDecompressor / ChunkDecompressor /
 * PageDecompressor), for callers that keep chunk metadata and pages in their own container.  A chunk's PagingSpec may
 * yield several pages; they share the chunk's bins (pco/src/wrapped/chunk_compressor.rs:129-140).  Classic mode with any
 * number of pages; the two-var modes (IntMult / FloatMult / FloatQuant) with ONE page per chunk, several are
 * PCO_B200_UNSUPPORTED for now.
 * A wrapped chunk with one page is the same bytes as a standalone chunk without its 4-byte preamble: chunk meta, then the page. */
typedef struct PcoB200ChunkCompressor PcoB200ChunkCompressor;
/* FileCompressor::write_header (pco/src/wrapped/file_compressor.rs; format version bytes, metadata/format_version.rs:87-91) */
PcoB200Error pco_b200_file_compressor_write_header(void *dst, size_t dst_cap, size_t *n_written);
/* FileDecompressor::new (pco/src/wrapped/file_decompressor.rs): checks the header bytes, returns how many were read */
PcoB200Error pco_b200_file_decompressor_read_header(const void *src, size_t src_len, size_t *n_read);
/* FileCompressor::chunk_compressor + ChunkCompressor::new (pco/src/wrapped/chunk_compressor.rs:442-500): does the compression */
PcoB200Error pco_b200_chunk_compressor_new(const void *nums, size_t n, unsigned char dtype, const PcoB200ChunkConfig *config,
                                           PcoB200ChunkCompressor **out);
void pco_b200_chunk_compressor_free(PcoB200ChunkCompressor *cc);
size_t pco_b200_chunk_compressor_n_pages(const PcoB200ChunkCompressor *cc);                  /* n_per_page().len() (:544-547) */
size_t pco_b200_chunk_compressor_page_n(const PcoB200ChunkCompressor *cc, size_t page_idx);  /* n_per_page()[i] */
size_t pco_b200_chunk_compressor_meta_size(const PcoB200ChunkCompressor *cc); /* exact; the reference's meta_size_hint is a bound (:557-562) */
PcoB200Error pco_b200_chunk_compressor_write_meta(const PcoB200ChunkCompressor *cc, void *dst, size_t dst_cap, size_t *n_written); /* :564-568 */
size_t pco_b200_chunk_compressor_page_size(const PcoB200ChunkCompressor *cc, size_t page_idx); /* exact; page_size_hint (:599-601) */
/* write_page (:659-705): page_idx out of range -> PCO_B200_INVALID_ARGUMENT (:661-666) */
PcoB200Error pco_b200_chunk_compressor_write_page(const PcoB200ChunkCompressor *cc, size_t page_idx, void *dst, size_t dst_cap,
                                                  size_t *n_written);
/* FileDecompressor::chunk_decompressor (metadata/chunk.rs:127-174): byte size of the chunk meta at the head of src */
PcoB200Error pco_b200_chunk_meta_size(const void *src, size_t src_len, unsigned char dtype, size_t *meta_len);
/* ChunkDecompressor::page_decompressor + PageDecompressor::read (pco/src/wrapped/page_decompressor.rs:193-252): decodes a page of
 * page_n numbers into dst (dst_len elements); bytes_read = bytes of `page` consumed (page_len must cover the page) */
PcoB200Error pco_b200_page_decompress(const void *chunk_meta, size_t meta_len, const void *page, size_t page_len, size_t page_n,
                                      unsigned char dtype, void *dst, size_t dst_len, PcoB200Progress *progress, size_t *bytes_read);

#if defined(__cplusplus)
}
#endif
#endif /* PCO_B200_H */
