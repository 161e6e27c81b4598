// Decode-side kernels for the pco hot path on sm_100a:
//   walk_kernel    — K6: serial tANS walk that produces the per-batch side index (cold path)
//   decode_kernel  — K7+K8+K9 fused: tANS symbols -> offsets unpack -> un-delta -> join -> store
//
// Reference behaviour restated here (paths relative to /root/reference):
//   tANS decode step        pco/src/page_latent_decompressor.rs:89-177, pco/src/ans/decoding.rs:27-48
//   table spread            pco/src/ans/spec.rs:24-59
//   offsets                 pco/src/page_latent_decompressor.rs:15-44
//   consecutive un-delta    pco/src/delta/consecutive.rs:35-50, pco/src/delta/mod.rs:29-33
//   joins                   pco/src/mode/{classic.rs:14-24,float_mult.rs:17-36,int_mult.rs:38-54,float_quant.rs:13-39}
//   per-batch driver        pco/src/wrapped/page_decompressor.rs:115-221
#pragma once
#include "codec_common.cuh"

namespace pcob200 {

#ifndef PCOB_DEC_NV1_BLOCKS
#define PCOB_DEC_NV1_BLOCKS 2
#endif
#ifndef PCOB_DEC_MIN_BLOCKS
#define PCOB_DEC_MIN_BLOCKS 2
#endif
#ifndef PCOB_DEC_TILE_ROWS
#define PCOB_DEC_TILE_ROWS 256
#endif
constexpr int DEC_THREADS = 256;
constexpr int DEC_TILE_ROWS = PCOB_DEC_TILE_ROWS;  // (var, batch) rows of the symbol tile; <= DEC_THREADS
constexpr int DEC_WARPS = DEC_THREADS / 32;
constexpr int SMALL_MAX_SIZE_LOG = 10;
constexpr int SMALL_MAX_BINS = 256;
constexpr int SYM_ROW_WORDS = 65;  // 256 one-byte symbols + 4 bytes pad: odd word stride -> conflict-free rows
constexpr int CHAIN_RING = 32;
constexpr int WIN_WORDS = 128;                  // 512-byte window of compressed bytes per (warp, var)
constexpr uint32_t WIN_USABLE_BITS = WIN_WORDS * 32 - 64;

// Optional region timers (build with -DPCOB_DEC_TIMING): per-warp clock64() deltas accumulated into global counters.
#ifdef PCOB_DEC_TIMING
__device__ unsigned long long g_dec_timing[16];
#define PCOB_TICK(idx)                              \
  do {                                              \
    long long _now = clock64();                     \
    _tacc[idx] += (unsigned long long)(_now - _tprev); \
    _tprev = _now;                                  \
  } while (0)
#else
#define PCOB_TICK(idx) do { } while (0)
#endif

// node word: next_state_idx_base (bits 0-15) | field (bits 16-23) | bits_to_read (bits 24-31): byte-aligned so that
// four symbols pack with byte permutes
//   decode tables: field = bin index;  walker tables: field = bin offset_bits
__device__ __forceinline__ uint32_t node_base(uint32_t n) { return n & 0xffffu; }
__device__ __forceinline__ uint32_t node_field(uint32_t n) { return (n >> 16) & 0xffu; }
__device__ __forceinline__ uint32_t node_btr(uint32_t n) { return n >> 24; }
// the fields of four nodes as four bytes
__device__ __forceinline__ uint32_t node_fields4(uint32_t n0, uint32_t n1, uint32_t n2, uint32_t n3) {
  return __byte_perm(__byte_perm(n0, n1, 0x0062), __byte_perm(n2, n3, 0x0062), 0x5410);
}

// Shared-memory accesses by explicit 32-bit shared address: the compiler otherwise re-derives the CTA's shared window
// (S2UR SR_CgaCtaId + ULEA) in front of every access made through a generic pointer, on the address path of the lookups.
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// ---------------------------------------------------------------------------
// Shared memory layout of one decode CTA (SMALL variant: size_log <= 10, n_bins <= 256)
// ---------------------------------------------------------------------------
struct BinEntry {            // what phase B needs about a bin, in one 16-byte shared-memory load
  uint64_t lower;            // (+ MID when the var is delta'd: folds toggle_center into the add)
  uint32_t ob;               // offset bits
  uint32_t mask;             // (1 << ob) - 1 for ob <= 32
};

struct BuildScratch {        // only live while the tables are built; shares storage with the symbol tile
  uint64_t bin_lower[MAX_VARS][SMALL_MAX_BINS];
  uint8_t bin_ob[MAX_VARS][SMALL_MAX_BINS];
  uint16_t bin_weight[MAX_VARS][SMALL_MAX_BINS];
  uint32_t bin_cum[MAX_VARS][SMALL_MAX_BINS + 1];
  uint16_t sym_of_state[MAX_VARS][1 << SMALL_MAX_SIZE_LOG];
  uint32_t rank_counter[MAX_VARS][SMALL_MAX_BINS];
};

struct DecodeSmem {
  ChunkHdr hdr;
  alignas(16) BinEntry bin[MAX_VARS][SMALL_MAX_BINS];
  uint32_t bin32[MAX_VARS][SMALL_MAX_BINS];  // compact: (lower - bin_base) | offset_bits << 25, valid when bin_compact[v]
  uint64_t bin_base[MAX_VARS];
  uint32_t bin_compact[MAX_VARS];
  // delta carry chain: mvec[b % CHAIN_RING] = true moments at the start of batch b once m_flag[...] == b + 1
  uint64_t mvec[CHAIN_RING][MAX_ORDER];
  volatile uint32_t m_flag[CHAIN_RING];
  uint64_t binom_full[MAX_ORDER];          // C(256, t): keeps the chain link free of global loads
  uint64_t binom_lane8[32][MAX_ORDER];     // C(8 * lane, t)
  uint32_t err;
  union {
    alignas(16) uint32_t win[DEC_WARPS][MAX_VARS][WIN_WORDS + 4];  // per-warp staged copy of a batch's offset bits
    BuildScratch build;                                             // only live while the bins are loaded
  };
};

// ---------------------------------------------------------------------------
// Scratch produced by symwalk_kernel and consumed by decode_kernel (HBM, sized from the destination):
//   symbols : one byte per stored latent, rows of 256; chunk task t owns rows from sym_row0(t) on, row (v, b) = v * nb_out + b
//   offsets : per (v, b) the chunk-relative bit position of the batch's offsets section (= end of its tANS section)
// nb_out = batches the destination can take from the chunk, so both arrays are bounded by the destination length
// whatever an (untrusted) index claims.
// ---------------------------------------------------------------------------
__host__ __device__ inline uint64_t scratch_row0(uint64_t out_offset, uint32_t task_idx) { return uint64_t(MAX_VARS) * (out_offset / BATCH_N + task_idx); }
__host__ __device__ inline uint64_t scratch_rows_total(uint64_t out_len, uint32_t n_tasks) { return uint64_t(MAX_VARS) * (out_len / BATCH_N + n_tasks + 1); }

// ---------------------------------------------------------------------------
// Chunk classes: symwalk_kernel parses and validates every chunk header anyway, so it also decides which decode
// instantiation owns the chunk (d_cls, one byte per chunk): 1 / 2 = decode_kernel<L, 1 / 2> (any refusal is reported
// by decode_kernel<L, 1>), 3 / 4 = decode_narrow_kernel (decode_narrow.cuh) with delta order 0 / 1.
// ---------------------------------------------------------------------------
constexpr uint32_t CLS_NARROW0 = 3, CLS_NARROW1 = 4, CLS_NARROWK = 5;  // narrow class with delta order 0 / 1 / 2..7
constexpr uint32_t CLS_DONE = 0x80;  // fused_narrow_kernel (decode_fused.cuh) has finished the chunk: the two-kernel path skips it
constexpr uint32_t NARROW_MAX_OB = 15, NARROW_LOW_BITS = 16;

struct NarrowInfo {   // one per chunk, in HBM scratch; only written for chunks of a narrow class
  uint64_t base;      // lower of bin 0 (+ MID when the var is delta'd: folds toggle_center into the add)
  uint64_t moment0;   // the page's delta moment (order 1)
  uint32_t n;
  uint32_t pad[3];
  uint32_t q[SMALL_MAX_BINS];  // offset_bits | (lower - lower_0) << 7
};
static_assert(sizeof(NarrowInfo) % 16 == 0, "NarrowInfo rows are loaded with vector accesses");

// ---------------------------------------------------------------------------
// Cooperative table build for one latent var (all threads of the CTA call this).
// WALKER = true stores offset_bits in the node field; false stores the bin index.
// ---------------------------------------------------------------------------
template <bool WALKER>
__device__ void build_var_tables(const BitSrc& src, ChunkHdr& hdr, int v, uint32_t* node, uint64_t* bin_lower, uint8_t* bin_ob,
                                 uint16_t* bin_weight, uint32_t* bin_cum, uint16_t* sym_of_state, uint32_t* rank_counter, uint32_t* err,
                                 bool add_mid_to_lower, bool build_nodes = true) {
  const VarHdr vh = hdr.var[v];
  const uint32_t n_bins = vh.n_bins;
  const uint32_t size_log = vh.ans_size_log;
  const uint32_t size = 1u << size_log;
  const int tid = threadIdx.x, nt = blockDim.x;
  const uint64_t mid = uint64_t(1) << (vh.latent_bits - 1);
  const uint64_t lmask = vh.latent_bits == 64 ? ~uint64_t(0) : ((uint64_t(1) << vh.latent_bits) - 1);
  const uint32_t obb = offset_bits_bits(vh.latent_bits);
  // 1. bins (metadata/chunk_latent_var.rs:22-53)
  uint32_t my_max_ob = 0;
  for (uint32_t i = tid; i < n_bins; i += nt) {
    uint64_t p = vh.bins_bit + uint64_t(i) * vh.bin_stride;
    uint32_t weight = uint32_t(read_bits_safe(src, p, size_log)) + 1;
    uint64_t lower = read_bits_safe(src, p + size_log, vh.latent_bits);
    uint32_t ob = uint32_t(read_bits_safe(src, p + size_log + vh.latent_bits, obb));
    if (ob > vh.latent_bits) atomicMax(err, (uint32_t)ST_CORRUPTION);
    bin_weight[i] = uint16_t(weight);
    if (!WALKER) bin_lower[i] = add_mid_to_lower ? ((lower + mid) & lmask) : lower;
    bin_ob[i] = uint8_t(ob);
    rank_counter[i] = 0;
    my_max_ob = max(my_max_ob, ob);
  }
  if (n_bins == 0 && tid == 0) {
    // zero bins: one implicit symbol with weight 1 (ans/spec.rs:61-66); size_log must be 0
    bin_weight[0] = 1;
    if (!WALKER) bin_lower[0] = add_mid_to_lower ? mid : 0;
    bin_ob[0] = 0;
    rank_counter[0] = 0;
  }
  if (my_max_ob) atomicMax(&hdr.var[v].max_offset_bits, my_max_ob);
  __syncthreads();
  const uint32_t nb = n_bins == 0 ? 1 : n_bins;
  // 2. cumulative weights (serial: <= 256 adds by one thread; a few hundred cycles)
  if (tid == 0) {
    uint32_t c = 0;
    for (uint32_t i = 0; i < nb; i++) { bin_cum[i] = c; c += bin_weight[i]; }
    bin_cum[nb] = c;
    if (c != size) atomicMax(err, (uint32_t)ST_CORRUPTION);  // ans/spec.rs:38-44
  }
  __syncthreads();
  if (*err || !build_nodes) return;
  // 3. spread (ans/spec.rs:24-59): step t -> state (stride * t) & (size - 1)
  uint32_t stride = (3 * size) / 5;
  if ((stride & 1) == 0) stride += 1;
  for (uint32_t t = tid; t < size; t += nt) {
    // largest i with bin_cum[i] <= t
    uint32_t lo = 0, hi = nb;  // invariant: cum[lo] <= t < cum[hi]
    while (hi - lo > 1) {
      uint32_t m = (lo + hi) >> 1;
      if (bin_cum[m] <= t) lo = m; else hi = m;
    }
    sym_of_state[(stride * t) & (size - 1)] = uint16_t(lo);
  }
  __syncthreads();
  // 4. decoder nodes in state order (ans/decoding.rs:27-48): x_s = weight + (#earlier states of the symbol)
  if (tid < 32) {
    const uint32_t lane = tid;
    for (uint32_t base = 0; base < size; base += 32) {
      uint32_t s = base + lane;
      bool active = s < size;
      uint32_t sym = active ? sym_of_state[s] : 0xffffffffu;
      uint32_t m = __match_any_sync(0xffffffffu, sym);
      uint32_t in_group = __popc(m & ((1u << lane) - 1));
      uint32_t prev = active ? rank_counter[sym] : 0;
      __syncwarp();
      if (active && in_group == 0) rank_counter[sym] = prev + __popc(m);
      __syncwarp();
      if (active) {
        uint32_t x_s = uint32_t(bin_weight[sym]) + prev + in_group;
        uint32_t btr = __clz(x_s) - __clz(size);
        uint32_t nbase = (x_s << btr) - size;
        uint32_t field = WALKER ? uint32_t(bin_ob[sym]) : sym;
        node[s] = nbase | (field << 16) | (btr << 24);
      }
    }
  }
  __syncthreads();
}

struct FileParams {
  const void* src;
  uint64_t src_len;
  uint32_t dtype;
  uint32_t uniform_type;
  uint32_t format_major;
};

// Stream-ordered decompress (pco_b200_decompress_async, decode_async.cuh) parses the standalone header and checks the side index on
// the device: async_validate_kernel leaves an AsyncGate in the caller's workspace, and the decode kernels read it in their prologue
// as `const uint32_t* gate`.  A closed gate makes every CTA return at once; an open one carries the header fields the host would
// otherwise have put into FileParams.  gate == nullptr on every other entry point (the host parsed the header).
struct AsyncGate {
  uint32_t open;          // 1: header and index passed; 0: async_validate_kernel has written the result already
  uint32_t uniform_type;  // from the standalone header
  uint32_t format_major;
  uint32_t finished;      // the index saw the file's terminator
  uint64_t n_total;
  uint64_t reserved;
};
__device__ __forceinline__ bool gate_closed(const uint32_t* gate, FileParams& fp) {
  if (gate == nullptr) return false;
  const AsyncGate* g = reinterpret_cast<const AsyncGate*>(gate);
  if (g->open == 0) return true;
  fp.uniform_type = g->uniform_type;
  fp.format_major = g->format_major;
  return false;
}

// ---------------------------------------------------------------------------
// walk_kernel (K6): builds the side index of a standalone file in place.
//   serial_file_mode = 1: a single CTA walks the file chunk after chunk from `first_chunk_byte`
//       (chunk boundaries are not in the stream: a chunk's length is only known once its tANS
//       sections have been walked), appending IndexChunk records and BatchEntry arrays.
//   serial_file_mode = 0: one CTA per pre-filled IndexChunk (offsets, n and entries_offset known).
// Layout written: index_base + chunks_offset : IndexChunk[]; entries at index_base + entries_offset.
// ---------------------------------------------------------------------------
constexpr int WR_BLOCKS = 128;  // ring: 128 blocks of 16 bytes
constexpr int WR_AHEAD = 64;    // blocks kept requested ahead of the cursor
constexpr int WR_STEP = 8;      // blocks per cp.async group
template <int CAP_LOG>   // 12: any table the format allows on this path; 10: what the decode kernels take (4x less shared memory)
struct WalkSmem {
  ChunkHdr hdr;
  uint32_t node[MAX_VARS][1 << CAP_LOG];
  // build scratch of ONE var (the vars' tables are built one after the other): 23 KB per CTA at CAP_LOG 10, so that 9 CTAs share an
  // SM and 1024 chunks are walked in a single wave (with per-var scratch: 36 KB, 6 CTAs, two waves - twice the time)
  uint8_t bin_ob[1 << CAP_LOG];
  uint16_t bin_weight[1 << CAP_LOG];
  uint32_t bin_cum[(1 << CAP_LOG) + 1];
  uint16_t sym_of_state[1 << CAP_LOG];
  uint32_t rank_counter[1 << CAP_LOG];
  uint32_t err;
  uint64_t next_chunk_byte;
  uint32_t status;
  alignas(16) uint32_t ring[WR_BLOCKS * 4];  // the walking thread's window on the stream (WalkRing)
};

struct WalkResult {     // written by the serial walker
  uint32_t n_chunks;    // chunks fully indexed in this launch
  uint32_t status;      // ST_TERMINATOR (clean end), ST_INDEX_FULL (resume later), or an error kind
  uint64_t next_byte;   // where the next chunk (or the byte after the terminator) starts
  uint64_t entries_end; // first free byte (from index_base) after the entries written
  uint64_t n_total;     // numbers in the indexed chunks
};

__host__ __device__ inline uint32_t n_batches_of(uint32_t n) { return (n + BATCH_N - 1) / BATCH_N; }

// Walk one chunk whose header is already parsed and tables built (WALKER nodes: the field byte is the bin's offset_bits), by ONE
// thread: the chunk's bit cursor is a single serial chain (batch boundaries are not in the stream: a batch's offsets section is as long
// as the sum of the offset bits of the symbols just walked, page_latent_decompressor.rs:106-134).  What the chain costs per group of 4
// symbols is its latency, so the loop is kept to the chain: the four node lookups go out together (32-bit shared addresses, states held
// as byte offsets), the stream is read from a shared-memory ring that cp.async fills ~1 KB ahead of the cursor (no global load and no
// 64-bit address arithmetic inside the chain), the four offset_bits bytes are summed with one dot product, and nothing lives in local
// memory (the states of the two latent vars are separate registers).  Splitting the 4 interleaved chains over 4 lanes (one lookup + a
// two-shuffle prefix of the bit counts per step) was measured SLOWER than one thread - the shuffles sit on the cursor dependency.

struct WalkRing {
  uint32_t ring_sa;                 // shared address of the ring
  const ulonglong2* blocks;         // the file as 16-byte blocks
  uint64_t max_blk;                 // last readable block
  uint64_t base_blk;                // block the relative bit positions count from
  uint64_t fetched;                 // blocks [.., fetched) have been requested (absolute block index, multiple of WR_STEP)
  __device__ __forceinline__ void request_upto(uint64_t upto) {
    while (fetched < upto) {
#pragma unroll
      for (int q = 0; q < WR_STEP; q++) {
        const uint64_t bi = fetched + q;
        const void* gp = blocks + (bi <= max_blk ? bi : max_blk);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(ring_sa + uint32_t(bi % WR_BLOCKS) * 16u), "l"(gp));
      }
      asm volatile("cp.async.commit_group;");
      fetched += WR_STEP;
    }
  }
  // the cursor is at relative bit `rbit`: keep WR_AHEAD blocks requested ahead of it and make the blocks it can touch next readable
  __device__ __forceinline__ void advance(uint32_t rbit) {
    const uint64_t cur = base_blk + (rbit >> 7);
    if (cur + 8 > fetched || fetched == 0) {  // first use, or a jump past what was requested (a long offsets section): start over at the cursor
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      fetched = cur & ~uint64_t(WR_STEP - 1);
      request_upto(fetched + WR_AHEAD + WR_STEP);
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      return;
    }
    request_upto(((cur + WR_AHEAD) & ~uint64_t(WR_STEP - 1)) + WR_STEP);
    // fetched >= cur + WR_AHEAD + 1; all but the 6 newest groups (48 blocks) are complete: blocks < cur + 17 are in the ring
    asm volatile("cp.async.wait_group 6;" ::: "memory");
  }
  __device__ __forceinline__ uint32_t word(uint32_t rel_word) const {  // 32-bit word `rel_word` counted from base_blk
    return lds_u32(ring_sa + (((uint32_t(base_blk & (WR_BLOCKS - 1)) << 2) + rel_word) & (WR_BLOCKS * 4 - 1)) * 4u);
  }
};

template <int CAP_LOG>
__device__ inline uint32_t walk_chunk_serial(const BitSrc& src, const ChunkHdr& hdr, const uint32_t (*node)[1 << CAP_LOG], uint64_t chunk_bit0,
                                             BatchEntry* entries, uint64_t* end_bit_out, uint32_t ring_sa) {
  const uint32_t nb = n_batches_of(hdr.n);
  WalkRing ring;
  ring.ring_sa = ring_sa;
  ring.blocks = reinterpret_cast<const ulonglong2*>(src.words);
  ring.max_blk = (src.n_bits == 0 ? 0 : (src.n_bits - 1) >> 6) >> 1;
  ring.base_blk = chunk_bit0 >> 7;
  ring.fetched = 0;
  const uint64_t base_bit = ring.base_blk << 7;
  // relative positions fit 32 bits: a chunk holds <= 2^24 numbers of <= 14 + 64 bits
  if (hdr.body_bit - base_bit > 0xffffffffull) return ST_CORRUPTION;
  uint32_t rbit = uint32_t(hdr.body_bit - base_bit);
  const uint64_t limit64 = src.n_bits - base_bit;
  const uint32_t limit = limit64 > 0xffffffffull ? 0xffffffffu : uint32_t(limit64);
  const uint32_t nv = hdr.n_vars;
  // states as byte offsets into the var's node table
  uint32_t a0 = hdr.init_state[0][0] << 2, a1 = hdr.init_state[0][1] << 2, a2 = hdr.init_state[0][2] << 2, a3 = hdr.init_state[0][3] << 2;
  uint32_t b0 = 0, b1 = 0, b2 = 0, b3 = 0;
  if (nv > 1) { b0 = hdr.init_state[1][0] << 2; b1 = hdr.init_state[1][1] << 2; b2 = hdr.init_state[1][2] << 2; b3 = hdr.init_state[1][3] << 2; }
  const uint32_t node_sa0 = smem_addr(node[0]), node_sa1 = smem_addr(node[nv > 1 ? 1 : 0]);
  const uint32_t stored0 = var_stored_n(hdr.n, hdr.var[0].delta_order), stored1 = nv > 1 ? var_stored_n(hdr.n, hdr.var[1].delta_order) : 0;
  const uint32_t nbins0 = hdr.var[0].n_bins, nbins1 = nv > 1 ? hdr.var[1].n_bins : 0;
  const uint32_t chunk_rel = uint32_t(chunk_bit0 - base_bit);  // entries count bits from the chunk's type byte
  ring.advance(rbit);
  for (uint32_t b = 0; b < nb; b++) {
#pragma unroll
    for (uint32_t v = 0; v < 2; v++) {
      if (v >= nv) break;
      const uint32_t cnt = batch_count(v == 0 ? stored0 : stored1, b);
      uint32_t s0 = v == 0 ? a0 : b0, s1 = v == 0 ? a1 : b1, s2 = v == 0 ? a2 : b2, s3 = v == 0 ? a3 : b3;
      BatchEntry e;
      e.bit_pos = rbit - chunk_rel;
      e.st[0] = uint16_t(s0 >> 2); e.st[1] = uint16_t(s1 >> 2); e.st[2] = uint16_t(s2 >> 2); e.st[3] = uint16_t(s3 >> 2);
      entries[size_t(v) * nb + b] = e;
      if (cnt == 0) continue;
      const uint32_t node_sa = v == 0 ? node_sa0 : node_sa1;
      uint32_t obs = 0;
      if ((v == 0 ? nbins0 : nbins1) > 1) {
        // bit reader: `acc` holds the next `avail` (> 32) bits of the stream, `nxt` the word after them - loaded ahead, so the refill that
        // follows every pair of symbols is a shift and an OR, and no shared-memory address on the chain depends on the cursor
        uint32_t wp = rbit >> 5;
        uint64_t acc = ((uint64_t(ring.word(wp + 1)) << 32) | ring.word(wp)) >> (rbit & 31);
        uint32_t avail = 64 - (rbit & 31);
        wp += 2;
        uint32_t nxt = ring.word(wp);
        auto refill = [&]() {
          if (avail <= 32) {
            acc |= uint64_t(nxt) << avail;
            avail += 32;
            wp += 1;
            if ((wp & 31) == 0) ring.advance(wp << 5);  // entering a new 1024-bit region: top the ring up
            nxt = ring.word(wp);
          }
        };
        uint32_t i = 0;
        for (; i + 4 <= cnt; i += 4) {
          const uint32_t n0 = lds_u32(node_sa + s0), n1 = lds_u32(node_sa + s1), n2 = lds_u32(node_sa + s2), n3 = lds_u32(node_sa + s3);
          const uint32_t c0 = node_btr(n0), c1 = node_btr(n1), c2 = node_btr(n2), c3 = node_btr(n3);
          obs = __dp4a(node_fields4(n0, n1, n2, n3), 0x01010101u, obs);
          {
            const uint32_t g = uint32_t(acc);  // c0 + c1 <= 28 bits
            s0 = (node_base(n0) + (g & ((1u << c0) - 1))) << 2;
            s1 = (node_base(n1) + ((g >> c0) & ((1u << c1) - 1))) << 2;
            acc >>= (c0 + c1);
            avail -= c0 + c1;
            refill();
          }
          {
            const uint32_t g = uint32_t(acc);
            s2 = (node_base(n2) + (g & ((1u << c2) - 1))) << 2;
            s3 = (node_base(n3) + ((g >> c2) & ((1u << c3) - 1))) << 2;
            acc >>= (c2 + c3);
            avail -= c2 + c3;
            refill();
          }
          rbit += c0 + c1 + c2 + c3;
        }
        // ragged tail of the page's last batch (page_latent_decompressor.rs:144-177)
        auto tail_step = [&](uint32_t& sj) {
          const uint32_t nn = lds_u32(node_sa + sj);
          const uint32_t cb = node_btr(nn);
          obs += node_field(nn);
          sj = (node_base(nn) + (uint32_t(acc) & ((1u << cb) - 1))) << 2;
          acc >>= cb;
          avail -= cb;
          rbit += cb;
          refill();
        };
        if (i < cnt) tail_step(s0);
        if (i + 1 < cnt) tail_step(s1);
        if (i + 2 < cnt) tail_step(s2);
      } else {
        obs = cnt * node_field(lds_u32(node_sa));
      }
      if (v == 0) { a0 = s0; a1 = s1; a2 = s2; a3 = s3; } else { b0 = s0; b1 = s1; b2 = s2; b3 = s3; }
      // the offsets section: obs bits (<= 256 x 64)
      if (obs > limit - min(rbit, limit)) return ST_INSUFFICIENT_DATA;
      rbit += obs;
      if (rbit > limit) return ST_INSUFFICIENT_DATA;
      if (rbit > 0xfff00000u) return ST_CORRUPTION;  // cannot happen for a chunk of <= 2^24 numbers
      ring.advance(rbit);
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  uint64_t bit = base_bit + rbit;
  // trailing bits of the page must be zero (wrapped/page_decompressor.rs:184-188)
  uint32_t pad = uint32_t((8 - (bit & 7)) & 7);
  if (pad && read_bits_safe(src, bit, pad) != 0) return ST_CORRUPTION;
  bit += pad;
  *end_bit_out = bit;
  return ST_OK;
}

// One warp builds the tables, its first lane walks.  Measured for 1024 chunks (profiles/r02_k_walk_variants.txt): 128 threads x 8 CTAs/SM
// (64 registers) 10.6 ms, 64 x 8 (128 registers) 13.6 ms, 64 x 16 15.3 ms, 32 x 8 8.5 ms
#ifndef PCOB_WALK_THREADS
#define PCOB_WALK_THREADS 32
#endif
#ifndef PCOB_WALK_MIN_BLOCKS
#define PCOB_WALK_MIN_BLOCKS 8
#endif
constexpr int WALK_THREADS = PCOB_WALK_THREADS;
template <int CAP_LOG>
__global__ void __launch_bounds__(WALK_THREADS, PCOB_WALK_MIN_BLOCKS) walk_kernel(FileParams fp, uint8_t* index_base, uint64_t chunks_offset, uint32_t max_chunks,
                                                   uint64_t entries_begin, uint64_t entries_cap_end, uint64_t first_chunk_byte,
                                                   uint64_t first_out_offset, uint64_t stop_after_total, uint32_t* statuses, WalkResult* result,
                                                   int serial_file_mode, uint64_t* chunk_ends = nullptr) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  WalkSmem<CAP_LOG>& sm = *reinterpret_cast<WalkSmem<CAP_LOG>*>(smem_raw);
  const BitSrc src = make_bitsrc(fp.src, fp.src_len);
  const int tid = threadIdx.x;
  IndexChunk* chunks = reinterpret_cast<IndexChunk*>(index_base + chunks_offset);
  uint32_t c = serial_file_mode ? 0 : blockIdx.x;
  uint64_t chunk_byte = serial_file_mode ? first_chunk_byte : chunks[c].chunk_offset;
  uint64_t entries_off = entries_begin, out_off = first_out_offset;
  uint32_t final_status = ST_OK;
  for (;;) {
    if (serial_file_mode && c >= max_chunks) { final_status = ST_INDEX_FULL; break; }
    const uint64_t chunk_bit0 = src.mis_bits + chunk_byte * 8;
    if (tid == 0) {
      sm.err = 0;
      parse_chunk_header(src, chunk_bit0, fp.dtype, fp.uniform_type, fp.format_major, true, sm.hdr);
      if (sm.hdr.status == ST_OK) {
        for (uint32_t v = 0; v < sm.hdr.n_vars; v++) {
          const VarHdr& vh = sm.hdr.var[v];
          if (vh.ans_size_log > uint32_t(CAP_LOG) || vh.n_bins > (1u << CAP_LOG)) sm.hdr.status = ST_UNSUPPORTED;
          if (vh.n_bins == 0 && var_stored_n(sm.hdr.n, vh.delta_order) > 0) sm.hdr.status = ST_CORRUPTION;  // page_decompressor.rs:52-57
        }
        // per-chunk mode: the caller sized this chunk's entries from the count it gave
        if (!serial_file_mode && sm.hdr.status == ST_OK && chunks[c].n != sm.hdr.n) sm.hdr.status = ST_INVALID_ARGUMENT;
      }
    }
    __syncthreads();
    uint32_t st = sm.hdr.status;
    if (st == ST_OK) {
      for (uint32_t v = 0; v < sm.hdr.n_vars; v++)
        build_var_tables<true>(src, sm.hdr, v, sm.node[v], nullptr, sm.bin_ob, sm.bin_weight, sm.bin_cum, sm.sym_of_state, sm.rank_counter, &sm.err, false);
      __syncthreads();
      if (sm.err) st = sm.err;
    }
    if (tid == 0) {
      uint64_t end_bit = chunk_bit0;
      if (st == ST_OK) {
        uint32_t nb = n_batches_of(sm.hdr.n);
        uint64_t need = uint64_t(sm.hdr.n_vars) * nb * sizeof(BatchEntry);
        uint64_t eo = serial_file_mode ? entries_off : chunks[c].entries_offset;
        if (eo + need > entries_cap_end) {
          st = ST_INDEX_FULL;
        } else {
          st = walk_chunk_serial<CAP_LOG>(src, sm.hdr, sm.node, chunk_bit0, reinterpret_cast<BatchEntry*>(index_base + eo), &end_bit, smem_addr(sm.ring));
          if (st == ST_OK) {
            IndexChunk ic;
            ic.chunk_offset = chunk_byte;
            ic.n = sm.hdr.n;
            ic.n_vars = sm.hdr.n_vars;
            ic.entries_offset = eo;
            ic.out_offset = serial_file_mode ? out_off : chunks[c].out_offset;
            chunks[c] = ic;
            entries_off = eo + ((need + 15) & ~uint64_t(15));
            out_off += sm.hdr.n;
          }
        }
      }
      if (statuses) statuses[c] = st;
      sm.status = st;
      sm.next_chunk_byte = (end_bit - src.mis_bits) >> 3;
      if (chunk_ends && !serial_file_mode) chunk_ends[c] = sm.next_chunk_byte;  // where this chunk ends: the next chunk's first byte
    }
    __syncthreads();
    if (!serial_file_mode) return;
    if (sm.status != ST_OK) { final_status = sm.status; break; }
    chunk_byte = sm.next_chunk_byte;
    c += 1;
    // pco::standalone::simple_decompress_into stops reading once dst is exhausted mid-chunk (simple.rs:116-139)
    if (tid == 0) sm.status = (out_off > stop_after_total) ? ST_DST_FULL : ST_OK;
    __syncthreads();
    if (sm.status == ST_DST_FULL) { final_status = ST_DST_FULL; break; }
    __syncthreads();
  }
  if (tid == 0 && serial_file_mode) {
    result->n_chunks = c;
    result->status = final_status;
    result->next_byte = chunk_byte + (final_status == ST_TERMINATOR ? 1 : 0);
    result->entries_end = entries_off;
    result->n_total = out_off - first_out_offset;
  }
}

// ---------------------------------------------------------------------------
// find_chunk_starts_kernel: every byte position in [begin, end) whose 4 bytes equal `pattern` (a chunk's type byte and its 24-bit
// count - 1, docs/format.md:186-192), appended to `out` in no particular order.  Chunk lengths are not in a standalone file, so the
// index-free decompressor cannot know where chunk k + 1 starts before it has walked chunk k - but chunks of one file almost always
// share their first 4 bytes (same type, same count), so every position that LOOKS like such a chunk start is walked speculatively,
// all in parallel, and the host then follows the chain of (start, end) pairs from the first chunk: a candidate is a real chunk
// start exactly when a verified chunk ends on it (host_api.cu, decompress_fast 3b).  A thread takes 8 positions.
// ---------------------------------------------------------------------------
constexpr int FIND_THREADS = 256;
constexpr int FIND_PER_THREAD = 8;
__global__ void __launch_bounds__(FIND_THREADS) find_chunk_starts_kernel(const uint8_t* __restrict__ src, uint64_t begin, uint64_t end, uint32_t pattern,
                                                                        uint64_t* __restrict__ out, uint32_t cap, uint32_t* __restrict__ count) {
  const uint64_t p0 = begin + (uint64_t(blockIdx.x) * FIND_THREADS + threadIdx.x) * FIND_PER_THREAD;
  if (p0 >= end) return;
  // positions p0 .. p0 + 7 need bytes p0 .. p0 + 10; `end` already leaves room for the 4 bytes of the last position
  uint32_t b[FIND_PER_THREAD + 3];
#pragma unroll
  for (int i = 0; i < FIND_PER_THREAD + 3; i++) b[i] = (p0 + i < end + 3) ? uint32_t(src[p0 + i]) : 0x100u;  // 0x100 never matches
#pragma unroll
  for (int i = 0; i < FIND_PER_THREAD; i++) {
    const uint32_t w = b[i] | (b[i + 1] << 8) | (b[i + 2] << 16) | (b[i + 3] << 24);
    if (w == pattern && (b[i] | b[i + 1] | b[i + 2] | b[i + 3]) < 0x100u && p0 + i < end) {
      const uint32_t k = atomicAdd(count, 1u);
      if (k < cap) out[k] = p0 + i;
    }
  }
}

// ---------------------------------------------------------------------------
// Latent-type helpers
// ---------------------------------------------------------------------------
template <typename L> struct LT;
template <> struct LT<uint8_t> { static constexpr int BITS = 8; };
template <> struct LT<uint16_t> { static constexpr int BITS = 16; };
template <> struct LT<uint32_t> { static constexpr int BITS = 32; };
template <> struct LT<uint64_t> { static constexpr int BITS = 64; };

// from_latent_ordered on bit patterns (data_types/unsigned.rs:155-161, signed.rs:46-52, float.rs:392-400)
template <typename L>
__device__ __forceinline__ L from_latent_ordered(L l, bool is_float, bool is_signed) {
  constexpr L MID = L(L(1) << (LT<L>::BITS - 1));
  if (is_float) return (l & MID) ? L(l ^ MID) : L(~l);
  if (is_signed) return L(l + MID);
  return l;
}
template <typename L>
__device__ __forceinline__ L to_latent_ordered(L bits, bool is_float, bool is_signed) {
  constexpr L MID = L(L(1) << (LT<L>::BITS - 1));
  if (is_float) return (bits & MID) ? L(~bits) : L(bits ^ MID);
  if (is_signed) return L(bits - MID);
  return bits;
}

// int_float_from_latent (data_types/float.rs:208-226) then `* base` without FMA contraction, returned as bits
__device__ __forceinline__ uint64_t float_mult_unadjusted(uint64_t l, uint64_t base_bits) {
  const uint64_t MID = uint64_t(1) << 63;
  const bool neg = l < MID;
  const uint64_t abs_int = neg ? (MID - 1 - l) : (l - MID);
  const uint64_t gpi = uint64_t(1) << 53;
  // The sign goes on as a bit, never as a floating-point negation: the value may be a NaN, the sign of a NaN is not a value the
  // compiler has to keep through `-f`, and it did not always (negative NaNs came back positive in some builds).
  uint64_t fb = abs_int < gpi ? (uint64_t)__double_as_longlong(__ull2double_rn(abs_int)) : 0x4340000000000000ull + (abs_int - gpi);
  if (neg) fb ^= MID;
  const double f = __longlong_as_double((long long)fb);
  // x86/ARM propagate the operand NaN (quieted, sign and payload kept); NVIDIA GPUs return the canonical NaN.
  // The reference runs on the CPU, so reproduce its bits (base is validated finite, so only f can be NaN).
  if (f != f) return fb | 0x0008000000000000ull;
  return (uint64_t)__double_as_longlong(__dmul_rn(f, __longlong_as_double((long long)base_bits)));
}
__device__ __forceinline__ uint32_t float_mult_unadjusted(uint32_t l, uint32_t base_bits) {
  const uint32_t MID = 1u << 31;
  const bool neg = l < MID;
  const uint32_t abs_int = neg ? (MID - 1 - l) : (l - MID);
  const uint32_t gpi = 1u << 24;
  uint32_t fb = abs_int < gpi ? __float_as_uint(__uint2float_rn(abs_int)) : 0x4b800000u + (abs_int - gpi);
  if (neg) fb ^= MID;  // see the f64 overload
  const float f = __uint_as_float(fb);
  if (f != f) return fb | 0x00400000u;  // CPU NaN propagation
  return __float_as_uint(__fmul_rn(f, __uint_as_float(base_bits)));
}
__device__ __forceinline__ uint16_t float_mult_unadjusted(uint16_t, uint16_t) { return 0; }  // f16 float_mult: not on the GPU path
__device__ __forceinline__ uint8_t float_mult_unadjusted(uint8_t, uint8_t) { return 0; }

// C(n, j) mod 2^64 for j < MAX_ORDER, by Pascal additions (exact in wrapping arithmetic)
struct Binoms {
  uint64_t lane8[32][MAX_ORDER];  // C(8 * lane, j)
  uint64_t full[MAX_ORDER];       // C(256, j)
};

// read `nbits` (<= LT<L>::BITS) at absolute bit position `pos` from global words
template <typename L>
__device__ __forceinline__ L read_offset(const uint64_t* __restrict__ cw, uint64_t max_word, uint64_t pos, uint32_t nbits) {
  if (LT<L>::BITS <= 32) {
    // 32-bit words: up to 32 bits at bit offset r < 32 span two words
    const uint32_t* c32 = reinterpret_cast<const uint32_t*>(cw);
    uint64_t wi = pos >> 5;
    uint64_t max32 = max_word * 2 + 1;
    uint32_t lo = __ldg(c32 + (wi <= max32 ? wi : max32));
    uint32_t hi = __ldg(c32 + (wi + 1 <= max32 ? wi + 1 : max32));
    uint32_t v = __funnelshift_r(lo, hi, uint32_t(pos & 31));
    return L(nbits >= 32 ? v : (v & ((1u << nbits) - 1)));
  } else {
    uint64_t wi = pos >> 6;
    uint32_t r = uint32_t(pos & 63);
    uint64_t lo = __ldg(cw + (wi <= max_word ? wi : max_word));
    uint64_t hi = __ldg(cw + (wi + 1 <= max_word ? wi + 1 : max_word));
    uint64_t v = r ? ((lo >> r) | (hi << (64 - r))) : lo;
    return L(nbits >= 64 ? v : (v & ((uint64_t(1) << nbits) - 1)));
  }
}

template <typename L>
__device__ __forceinline__ L shfl_up_L(L v, int d) {
  if (sizeof(L) == 8) {
    uint32_t lo = __shfl_up_sync(0xffffffffu, uint32_t(uint64_t(v)), d);
    uint32_t hi = __shfl_up_sync(0xffffffffu, uint32_t(uint64_t(v) >> 32), d);
    return L((uint64_t(hi) << 32) | lo);
  }
  return L(__shfl_up_sync(0xffffffffu, uint32_t(v), d));
}
template <typename L>
__device__ __forceinline__ L shfl_idx_L(L v, int src) {
  if (sizeof(L) == 8) {
    uint32_t lo = __shfl_sync(0xffffffffu, uint32_t(uint64_t(v)), src);
    uint32_t hi = __shfl_sync(0xffffffffu, uint32_t(uint64_t(v) >> 32), src);
    return L((uint64_t(hi) << 32) | lo);
  }
  return L(__shfl_sync(0xffffffffu, uint32_t(v), src));
}

// One zero-seeded exclusive scan level over the warp's 256 values (8 consecutive per lane), wrapping.
// Returns the batch total through `total` (valid in all lanes).
template <typename L>
__device__ __forceinline__ void warp_excl_scan8(L (&x)[8], L& total, int lane) {
  L run = 0;
#pragma unroll
  for (int e = 0; e < 8; e++) {
    L t = x[e];
    x[e] = run;
    run = L(run + t);
  }
  L inc = run;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    L o = shfl_up_L<L>(inc, d);
    if (lane >= d) inc = L(inc + o);
  }
  L excl = L(inc - run);
#pragma unroll
  for (int e = 0; e < 8; e++) x[e] = L(x[e] + excl);
  total = shfl_idx_L<L>(inc, 31);
}

// Field of up to 32 (WIDE: 64) bits at bit position p of a shared-memory window of 32-bit words.
template <typename L, bool WIDE>
__device__ __forceinline__ L win_extract(const uint32_t* __restrict__ win, uint32_t p, uint32_t nbits, uint32_t mask) {
  const uint32_t w = p >> 5, r = p & 31;
  const uint32_t lo = win[w], mid = win[w + 1];
  const uint32_t v0 = __funnelshift_r(lo, mid, r);
  if (!WIDE) return L(v0 & mask);
  if (nbits <= 32) return L(v0 & mask);
  const uint32_t hi = win[w + 2];
  const uint32_t v1 = __funnelshift_r(mid, hi, r);
  const uint32_t m1 = nbits >= 64 ? 0xffffffffu : ((1u << (nbits - 32)) - 1);
  return L((uint64_t(v1 & m1) << 32) | v0);
}

// from_latent_ordered with the number kind hoisted: 0 unsigned, 1 signed, 2 float
template <typename L>
__device__ __forceinline__ L from_latent_kind(L l, int kind) {
  constexpr L MID = L(L(1) << (LT<L>::BITS - 1));
  if (kind == 0) return l;
  if (kind == 1) return L(l ^ MID);
  const L s = L(l >> (LT<L>::BITS - 1));
  return L(l ^ L(L(s - 1) | MID));
}

// ---------------------------------------------------------------------------
// Consecutive un-delta (delta/consecutive.rs:35-50) of a batch held 8-per-lane in registers, split in two:
//   undelta_local : K nested exclusive scans with ZERO seeds (needs nothing from earlier batches); c_j = batch sum of x^(j+1)
//   apply_moments : adds (A^i m)_0 to element i, where m are the true moments at the batch start (linearity of the recurrence
//                   m' = A m + e d,  A = I + superdiagonal, so (A^n)_{j,j+t} = C(n,t) mod 2^w)
// The moments travel along a chain m_{b+1} = A^256 m_b + c_b; each warp runs the link of its own batch.
// ---------------------------------------------------------------------------
template <typename L, int K>
__device__ __forceinline__ void undelta_local(L (&x)[8], L (&c)[K], int lane) {
#pragma unroll
  for (int lvl = 0; lvl < K; lvl++) {
    L total;
    warp_excl_scan8<L>(x, total, lane);
    c[K - 1 - lvl] = total;
  }
}

// One batch's un-delta, everything in registers: zero-seeded scans, then this warp's link of the moment chain
// (wait for m_b, publish m_{b+1} = A^256 m_b + c_b), then fold m_b into the 8 values of each lane.  The link reads only
// shared memory: with most of L1 carved out for shared memory, a global or local load here is an L2 round trip on
// the one serial dependency of the chunk (measured: 52 % of warp time was chain wait before this).
template <typename L, int K>
__device__ __forceinline__ void undelta_chain(L (&x)[8], DecodeSmem& sm, uint32_t b, int lane) {
  L c[K];
  undelta_local<L, K>(x, c, lane);
  const uint32_t slot = b % CHAIN_RING, nslot = (b + 1) % CHAIN_RING;
  L bl8[K];
#pragma unroll
  for (int t = 0; t < K; t++) bl8[t] = L(sm.binom_lane8[lane][t]);
  while (sm.m_flag[slot] != b + 1) {
  }
  __threadfence_block();
  L m[K];
#pragma unroll
  for (int k = 0; k < K; k++) m[k] = L(sm.mvec[slot][k]);
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < K; j++) {
      L acc = c[j];
#pragma unroll
      for (int t = 0; j + t < K; t++) acc = L(acc + L(L(sm.binom_full[t]) * m[j + t]));
      sm.mvec[nslot][j] = uint64_t(acc);
    }
    __threadfence_block();
    sm.m_flag[nslot] = b + 2;
  }
  L s[K];
#pragma unroll
  for (int j = 0; j < K; j++) {
    L acc = 0;
#pragma unroll
    for (int t = 0; j + t < K; t++) acc = L(acc + L(bl8[t] * m[j + t]));
    s[j] = acc;
  }
#pragma unroll
  for (int e = 0; e < 8; e++) {
    x[e] = L(x[e] + s[0]);
#pragma unroll
    for (int j = 0; j + 1 < K; j++) s[j] = L(s[j] + s[j + 1]);
  }
}

// 8 consecutive numbers per lane <-> global memory, 16-byte accesses
template <typename L, int K>
__device__ __noinline__ void undelta_chain_out_of_line(L* x, DecodeSmem& sm, uint32_t b, int lane) {
  L r[8];
#pragma unroll
  for (int e = 0; e < 8; e++) r[e] = x[e];
  undelta_chain<L, K>(r, sm, b, lane);
#pragma unroll
  for (int e = 0; e < 8; e++) x[e] = r[e];
}
// only the copy handed to the out-of-line function lives in local memory; the caller's registers stay registers
template <typename L, int K>
__device__ __forceinline__ void undelta_chain_cold(L (&x)[8], DecodeSmem& sm, uint32_t b, int lane) {
  L tmp[8];
#pragma unroll
  for (int e = 0; e < 8; e++) tmp[e] = x[e];
  undelta_chain_out_of_line<L, K>(tmp, sm, b, lane);
#pragma unroll
  for (int e = 0; e < 8; e++) x[e] = tmp[e];
}

// 8 consecutive numbers of a lane -> global memory.  32-byte stores (STG.E.ENL2.256, sm_100) when the destination allows:
// with 16-byte stores every instruction of the warp fills half of 32 sectors, and the L1 was the busiest unit of the decode
// kernels (81 % of peak in decode_narrow_kernel; 0.78 -> 0.58 ms with whole-sector stores).
template <typename L>
__device__ __forceinline__ void store8(L* __restrict__ dst, const L (&r)[8]) {
  if (sizeof(L) == 8) {
    if ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) {
#pragma unroll
      for (int q = 0; q < 2; q++)
        asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * q), "l"(uint64_t(r[4 * q])), "l"(uint64_t(r[4 * q + 1])),
                     "l"(uint64_t(r[4 * q + 2])), "l"(uint64_t(r[4 * q + 3])) : "memory");
    } else {
#pragma unroll
      for (int q = 0; q < 4; q++)
        asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(dst + 2 * q), "l"(uint64_t(r[2 * q])), "l"(uint64_t(r[2 * q + 1])) : "memory");
    }
  } else if (sizeof(L) == 4) {
    if ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) {
      asm volatile("st.global.v8.u32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(uint32_t(r[0])), "r"(uint32_t(r[1])), "r"(uint32_t(r[2])),
                   "r"(uint32_t(r[3])), "r"(uint32_t(r[4])), "r"(uint32_t(r[5])), "r"(uint32_t(r[6])), "r"(uint32_t(r[7])) : "memory");
    } else {
#pragma unroll
      for (int q = 0; q < 2; q++)
        asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * q), "r"(uint32_t(r[4 * q])), "r"(uint32_t(r[4 * q + 1])),
                     "r"(uint32_t(r[4 * q + 2])), "r"(uint32_t(r[4 * q + 3])) : "memory");
    }
  } else if (sizeof(L) == 2) {  // 8 numbers = 16 bytes: one store when aligned
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
      asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(uint32_t(r[0]) | (uint32_t(r[1]) << 16)), "r"(uint32_t(r[2]) | (uint32_t(r[3]) << 16)),
                   "r"(uint32_t(r[4]) | (uint32_t(r[5]) << 16)), "r"(uint32_t(r[6]) | (uint32_t(r[7]) << 16)) : "memory");
    } else {
#pragma unroll
      for (int e = 0; e < 8; e++) dst[e] = r[e];
    }
  } else {  // 8 numbers = 8 bytes
    if ((reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
      asm volatile("st.global.v2.u32 [%0], {%1, %2};" ::"l"(dst), "r"(uint32_t(r[0]) | (uint32_t(r[1]) << 8) | (uint32_t(r[2]) << 16) | (uint32_t(r[3]) << 24)),
                   "r"(uint32_t(r[4]) | (uint32_t(r[5]) << 8) | (uint32_t(r[6]) << 16) | (uint32_t(r[7]) << 24)) : "memory");
    } else {
#pragma unroll
      for (int e = 0; e < 8; e++) dst[e] = r[e];
    }
  }
}
template <typename L>
__device__ __forceinline__ void load8(const L* __restrict__ src, L (&r)[8]) {
  if (sizeof(L) == 8) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const uint4 v = s4[q];
      r[2 * q] = L((uint64_t(v.y) << 32) | v.x);
      r[2 * q + 1] = L((uint64_t(v.w) << 32) | v.z);
    }
  } else if (sizeof(L) == 4) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    const uint4 a = s4[0], bq = s4[1];
    r[0] = L(a.x); r[1] = L(a.y); r[2] = L(a.z); r[3] = L(a.w);
    r[4] = L(bq.x); r[5] = L(bq.y); r[6] = L(bq.z); r[7] = L(bq.w);
  } else {
#pragma unroll
    for (int e = 0; e < 8; e++) r[e] = src[e];
  }
}

// ---------------------------------------------------------------------------
// symwalk_kernel (K7a): the serial part of decoding a batch - its 256-symbol tANS walk - for every batch of a chunk.
// One CTA of 4 warps per chunk; a warp takes 32 consecutive batches of one var at a time, a lane per batch
// (page_latent_decompressor.rs:89-177):
//   1. every lane stages the bytes its next 64 symbols can read into its private shared-memory row with 16-byte
//      cp.async from its exact position (rows, not the span of the 32 batches: the offsets sections that lie between
//      the tANS sections are never staged) - per-thread scattered global reads inside the walk were what stalled the
//      first design;
//   2. per 4 symbols: one register window over the row, 4 node lookups, 4 extractions; the bin indices go to a padded
//      shared tile;
//   3. every 64 symbols the tile leaves as 64-byte pieces of the 256-byte symbol rows, and at the end each batch's
//      end position = start of its offsets section.
// The walk is a 256-step dependent chain per lane: latency-bound, so it wants warps - 32 KB of shared memory per CTA
// puts 7 CTAs (28 warps) on an SM and the whole 1024-chunk workload in a single wave.
// ---------------------------------------------------------------------------
constexpr int SW_THREADS = 128;
constexpr int SW_WARPS = SW_THREADS / 32;
#ifndef PCOB_SW_ROWS
#define PCOB_SW_ROWS 64
#endif
// Row staging: every lane keeps a private row with the bytes its next SW_ROW_SYMS symbols can read (<= 10 bits each,
// + 16 bytes of start alignment + the window's over-read), refilled with 16-byte cp.async from its exact position.
// Only tANS bits are staged (the offsets sections between them are not), so a CTA needs 32 KB and 7 fit on an SM.
// Measured on C2 (1024 chunks): one 13 KiB stage per warp holding the whole span of its 32 batches, 3 CTAs per SM:
// 0.305 ms; rows of 128 symbols, 5 CTAs: 0.305 ms; rows of 64 symbols, 7 CTAs: 0.266 ms.  More node replicas at the
// price of CTAs per SM (16 / 32 copies, 5 / 4 CTAs) were slower: 0.300 / 0.312 ms.
constexpr int SW_ROW_SYMS = PCOB_SW_ROWS;
constexpr int SW_ROW_BLOCKS = ((SW_ROW_SYMS * SMALL_MAX_SIZE_LOG / 8 + 15) / 16 + 2) | 1;  // odd: rows start in different banks
constexpr int SW_STAGE_BYTES = 32 * SW_ROW_BLOCKS * 16;
constexpr int SW_STAGE_WORDS = SW_STAGE_BYTES / 4;
#ifndef PCOB_SW_NODE_WORDS
#define PCOB_SW_NODE_WORDS 2048
#endif
#ifndef PCOB_SW_SLAB
#define PCOB_SW_SLAB 64
#endif
constexpr int SW_NODE_WORDS = PCOB_SW_NODE_WORDS;   // decoder nodes per CTA, replicated when the tables are small (see below)
constexpr int SW_SLAB = PCOB_SW_SLAB; // symbols per tile flush
constexpr int SW_TILE_ROW = SW_SLAB / 4 + 1;  // words per tile row (odd: conflict-free rows)
static_assert(SW_ROW_SYMS % SW_SLAB == 0 && BATCH_N % SW_ROW_SYMS == 0, "a row refill covers whole slabs");

// 32 lanes look up 32 unrelated states per step.  A var's node table is stored R times when it is small, copy r
// interleaved at word (state * R + r), lane l reading copy l mod R: lanes with different copies never share a bank.
struct SymWalkSmem {
  ChunkHdr hdr;
  uint32_t node[SW_NODE_WORDS];
  uint32_t err;
  uint32_t not_narrow;
  union {
    struct {
      BuildScratch build;
      uint32_t node_plain[MAX_VARS][1 << SMALL_MAX_SIZE_LOG];
    } b;
    struct {
      alignas(16) uint32_t stage[SW_WARPS][SW_STAGE_WORDS + 16];
      alignas(16) uint32_t tile[SW_WARPS][32 * SW_TILE_ROW + 3];
    } w;
  };
};

__global__ void __launch_bounds__(SW_THREADS) symwalk_kernel(FileParams fp, const IndexChunk* __restrict__ chunks, const uint8_t* __restrict__ index_base,
                                                              uint64_t index_len, uint64_t out_len, uint8_t* __restrict__ d_syms, uint32_t* __restrict__ d_offs,
                                                              uint8_t* __restrict__ d_nvars, NarrowInfo* __restrict__ d_narrow, int classes_preset,
                                                              const uint32_t* __restrict__ gate) {
  if (gate_closed(gate, fp)) return;
  if (classes_preset && (d_nvars[blockIdx.x] & CLS_DONE)) return;  // fused_narrow_kernel has decoded (or refused) this chunk
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SymWalkSmem& sm = *reinterpret_cast<SymWalkSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const IndexChunk task = chunks[blockIdx.x];
  const BitSrc src = make_bitsrc(fp.src, fp.src_len);
  const uint64_t max_word = src.n_bits == 0 ? 0 : (src.n_bits - 1) >> 6;
  const uint64_t max_blk = max_word >> 1;
  const uint64_t chunk_bit0 = src.mis_bits + task.chunk_offset * 8;
  // every refusal below is reported by decode_kernel, which parses the same header
  if (tid == 0) {
    sm.err = 0;
    sm.not_narrow = 0;
    parse_chunk_header(src, chunk_bit0, fp.dtype, fp.uniform_type, fp.format_major, true, sm.hdr);
    if (sm.hdr.status == ST_OK) {
      for (uint32_t v = 0; v < sm.hdr.n_vars; v++) {
        const VarHdr& vh = sm.hdr.var[v];
        if (vh.ans_size_log > SMALL_MAX_SIZE_LOG || vh.n_bins > SMALL_MAX_BINS) sm.hdr.status = ST_UNSUPPORTED;
        if (vh.n_bins == 0 && var_stored_n(sm.hdr.n, vh.delta_order) > 0) sm.hdr.status = ST_CORRUPTION;
      }
      if (task.n != 0 && task.n != sm.hdr.n) sm.hdr.status = ST_CORRUPTION;
    }
  }
  __syncthreads();
  // which decode_kernel instantiation owns the chunk (a refused header goes to the one-var kernel, which reports it)
  if (tid == 0) d_nvars[blockIdx.x] = uint8_t(sm.hdr.status == ST_OK && sm.hdr.n_vars == 2 ? 2 : 1);
  if (sm.hdr.status != ST_OK) return;
  const uint32_t n_vars = sm.hdr.n_vars;
  const bool need_index = (sm.hdr.var[0].n_bins > 1) || (n_vars > 1 && sm.hdr.var[1].n_bins > 1);
  if (!need_index || task.entries_offset == 0 || !index_base) return;  // trivial vars: section starts are closed-form
  // a stale or foreign index must not send the walk outside the index buffer (decode_kernel reports it)
  if (task.entries_offset > index_len || uint64_t(n_vars) * n_batches_of(sm.hdr.n) * sizeof(BatchEntry) > index_len - task.entries_offset) return;
  for (uint32_t v = 0; v < n_vars; v++)
    build_var_tables<false>(src, sm.hdr, v, sm.b.node_plain[v], sm.b.build.bin_lower[v], sm.b.build.bin_ob[v], sm.b.build.bin_weight[v],
                            sm.b.build.bin_cum[v], sm.b.build.sym_of_state[v], sm.b.build.rank_counter[v], &sm.err, false);
  __syncthreads();
  if (sm.err) return;
#ifndef PCOB_NO_NARROW
  // narrow class (decode_narrow.cuh): the header and bins are parsed and validated at this point
  if (d_narrow && n_vars == 1 && sm.hdr.mode == MODE_CLASSIC && sm.hdr.var[0].delta_order <= 1 && sm.hdr.var[0].latent_bits >= 32 &&
      sm.hdr.var[0].n_bins >= 2 && sm.hdr.var[0].max_offset_bits <= NARROW_MAX_OB) {
    const VarHdr& vh = sm.hdr.var[0];
    const uint64_t lmask = vh.latent_bits == 64 ? ~uint64_t(0) : ((uint64_t(1) << vh.latent_bits) - 1);
    const uint64_t lower0 = sm.b.build.bin_lower[0][0];
    NarrowInfo* ni = d_narrow + blockIdx.x;
    for (uint32_t i = tid; i < vh.n_bins; i += SW_THREADS) {
      const uint64_t d = (sm.b.build.bin_lower[0][i] - lower0) & lmask;
      if (d >> NARROW_LOW_BITS) sm.not_narrow = 1;
      ni->q[i] = uint32_t(sm.b.build.bin_ob[0][i]) | (uint32_t(d) << 7);
    }
    __syncthreads();
    if (tid == 0 && !sm.not_narrow) {
      const uint64_t mid = uint64_t(1) << (vh.latent_bits - 1);
      ni->base = vh.delta_order ? ((lower0 + mid) & lmask) : lower0;
      ni->moment0 = sm.hdr.moments[0][0];
      ni->n = sm.hdr.n;
      d_nvars[blockIdx.x] = uint8_t(vh.delta_order ? CLS_NARROW1 : CLS_NARROW0);
    }
  }
#endif
  // replicate: var v owns SW_NODE_WORDS / n_vars words (>= its 2^size_log); rep_log = log2 of its copy count
  const uint32_t region = SW_NODE_WORDS / n_vars;
  const uint32_t rep_log0 = min(5u, uint32_t(31 - __clz(region >> sm.hdr.var[0].ans_size_log)));
  const uint32_t rep_log1 = n_vars > 1 ? min(5u, uint32_t(31 - __clz(region >> sm.hdr.var[1].ans_size_log))) : 0u;
  for (uint32_t v = 0; v < n_vars; v++) {
    const uint32_t rl = v == 0 ? rep_log0 : rep_log1;
    const uint32_t cells = (1u << sm.hdr.var[v].ans_size_log) << rl;
    for (uint32_t i = tid; i < cells; i += SW_THREADS) sm.node[v * region + i] = sm.b.node_plain[v][i >> rl];
  }
  __syncthreads();  // the build scratch and plain tables (aliased by stage and tile) are dead
  const uint32_t n = sm.hdr.n;
  const uint32_t n_out = task.out_offset >= out_len ? 0u : uint32_t(min(uint64_t(n), out_len - task.out_offset));
  const uint32_t nb_total = n_batches_of(n), nb_out = n_batches_of(n_out);
  const BatchEntry* entries = reinterpret_cast<const BatchEntry*>(index_base + task.entries_offset);
  const uint64_t row0 = scratch_row0(task.out_offset, blockIdx.x);
  const uint32_t groups = (nb_out + 31) / 32;
  uint32_t* stg = sm.w.stage[warp];
  uint32_t* tile = sm.w.tile[warp];
  const uint32_t stg_sa = uint32_t(__cvta_generic_to_shared(stg));
  for (uint32_t item = warp; item < n_vars * groups; item += SW_WARPS) {
    const uint32_t v = item / groups, b0 = (item % groups) * 32;
    const VarHdr& vh = sm.hdr.var[v];
    const uint32_t stored = var_stored_n(n, vh.delta_order);
    const uint32_t nbg = min(32u, nb_out - b0);  // batches of this group
    uint32_t* offs = d_offs + row0 + size_t(v) * nb_out;
    // lane k: entry of batch b0 + k
    BatchEntry e;
    e.bit_pos = 0; e.st[0] = e.st[1] = e.st[2] = e.st[3] = 0;
    if (uint32_t(lane) < nbg) e = entries[size_t(v) * nb_total + b0 + lane];
    if (vh.n_bins <= 1) {  // no tANS bits: the offsets section starts where the batch starts
      if (uint32_t(lane) < nbg) offs[b0 + lane] = e.bit_pos;
      continue;
    }
    const uint32_t size_log = vh.ans_size_log;
    const uint32_t rl = v == 0 ? rep_log0 : rep_log1;
    const uint32_t* node = sm.node + v * region + (uint32_t(lane) & ((1u << rl) - 1));  // this lane's copy
    const uint32_t node_sa = smem_addr(node);
    const uint32_t sl = rl + 2;  // states are kept as byte offsets into the lane's copy
    {
      // ---- row staging: all batches of the group are walked at once
      const bool mine = uint32_t(lane) < nbg;
      const uint32_t b = b0 + lane;
      const int cnt = mine ? int(batch_count(stored, b)) : 0;
      const uint32_t smask = (1u << size_log) - 1;
      uint32_t s0 = min(uint32_t(e.st[0]), smask) << sl, s1 = min(uint32_t(e.st[1]), smask) << sl;
      uint32_t s2 = min(uint32_t(e.st[2]), smask) << sl, s3 = min(uint32_t(e.st[3]), smask) << sl;
      uint32_t* row = tile + lane * SW_TILE_ROW;
      const uint32_t row_sa = smem_addr(row);
      const uint32_t* rowp = stg + lane * (SW_ROW_BLOCKS * 4);
      const uint32_t row_g = stg_sa + uint32_t(lane) * (SW_ROW_BLOCKS * 16);
      uint8_t* sym_rows = d_syms + (row0 + size_t(v) * nb_out + b0) * BATCH_N;
      uint64_t bit = min(chunk_bit0 + e.bit_pos, src.n_bits);
      for (int part = 0; part < BATCH_N / SW_ROW_SYMS; part++) {
        const uint64_t blk = bit >> 7;
        if (cnt > part * SW_ROW_SYMS) {
#pragma unroll
          for (uint32_t q = 0; q < uint32_t(SW_ROW_BLOCKS); q++) {
            const void* gp = reinterpret_cast<const ulonglong2*>(src.words) + min(blk + q, max_blk);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(row_g + q * 16), "l"(gp));
          }
        }
        asm volatile("cp.async.commit_group;");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        uint32_t wpos = uint32_t(bit & 127);
        uint32_t w = wpos >> 5;
        uint32_t x0 = lds_u32(row_g + 4 * w), x1 = lds_u32(row_g + 4 * w + 4), x2 = lds_u32(row_g + 4 * w + 8);  // register window over the stream
        for (int slab = part * (SW_ROW_SYMS / SW_SLAB); slab < (part + 1) * (SW_ROW_SYMS / SW_SLAB); slab++) {
          const int i0 = slab * SW_SLAB;
          if (size_log <= 8) {
            // four symbols read <= 32 bits: one 32-bit window per group, fields by bit-field extract
  #pragma unroll 4
            for (int i = i0; i < i0 + SW_SLAB; i += 4) {
              if (i + 4 <= cnt) {
                const uint32_t n0 = lds_u32(node_sa + s0), n1 = lds_u32(node_sa + s1), n2 = lds_u32(node_sa + s2), n3 = lds_u32(node_sa + s3);
                const uint32_t g = __funnelshift_r(x0, x1, wpos & 31);
                const uint32_t c0 = node_btr(n0), c1 = node_btr(n1), c2 = node_btr(n2), c3 = node_btr(n3);
                const uint32_t sh2 = c0 + c1, sh3 = sh2 + c2;
                s0 = (node_base(n0) + (g & ((1u << c0) - 1))) << sl;
                s1 = (node_base(n1) + ((g >> c0) & ((1u << c1) - 1))) << sl;
                s2 = (node_base(n2) + ((g >> sh2) & ((1u << c2) - 1))) << sl;
                s3 = (node_base(n3) + ((g >> sh3) & ((1u << c3) - 1))) << sl;
                sts_u32(row_sa + (i - i0), node_fields4(n0, n1, n2, n3));
                wpos += sh3 + c3;
                if ((wpos >> 5) != w) { w = wpos >> 5; x0 = lds_u32(row_g + 4 * w); x1 = lds_u32(row_g + 4 * w + 4); }
              }
            }
          } else {
  #pragma unroll 2
            for (int i = i0; i < i0 + SW_SLAB; i += 4) {
              if (i + 4 <= cnt) {
                const uint32_t n0 = lds_u32(node_sa + s0), n1 = lds_u32(node_sa + s1), n2 = lds_u32(node_sa + s2), n3 = lds_u32(node_sa + s3);
                const uint32_t r = wpos & 31;
                const uint64_t g = (uint64_t(__funnelshift_r(x1, x2, r)) << 32) | __funnelshift_r(x0, x1, r);
                const uint32_t c0 = node_btr(n0), c1 = node_btr(n1), c2 = node_btr(n2), c3 = node_btr(n3);
                const uint32_t sh2 = c0 + c1, sh3 = sh2 + c2;
                s0 = (node_base(n0) + (uint32_t(g) & ((1u << c0) - 1))) << sl;
                s1 = (node_base(n1) + (uint32_t(g >> c0) & ((1u << c1) - 1))) << sl;
                s2 = (node_base(n2) + (uint32_t(g >> sh2) & ((1u << c2) - 1))) << sl;
                s3 = (node_base(n3) + (uint32_t(g >> sh3) & ((1u << c3) - 1))) << sl;
                sts_u32(row_sa + (i - i0), node_fields4(n0, n1, n2, n3));
                wpos += sh3 + c3;
                if ((wpos >> 5) != w) { w = wpos >> 5; x0 = lds_u32(row_g + 4 * w); x1 = lds_u32(row_g + 4 * w + 4); x2 = lds_u32(row_g + 4 * w + 8); }
              }
            }
          }
          if (cnt > i0 && cnt < i0 + SW_SLAB && (cnt & 3)) {  // ragged tail of the page's last batch (page_latent_decompressor.rs:144-177)
            const int i = cnt & ~3;
            uint32_t packed = 0;
            uint32_t sarr[4] = {s0, s1, s2, s3};
            for (int j = 0; i + j < cnt; j++) {
              const uint32_t nn = lds_u32(node_sa + sarr[j]);
              const uint32_t ww = wpos >> 5, r = wpos & 31;
              const uint32_t val = __funnelshift_r(rowp[ww], rowp[ww + 1], r) & ((1u << node_btr(nn)) - 1);
              packed |= node_field(nn) << (8 * j);
              sarr[j] = (node_base(nn) + val) << sl;
              wpos += node_btr(nn);
            }
            sts_u32(row_sa + (i - i0), packed);
          }
          __syncwarp();
          // the slab of rows k0..k1 -> SW_SLAB-byte pieces of the 256-byte symbol rows (16 bytes per lane)
          if (__any_sync(0xffffffffu, cnt > i0)) {
            constexpr uint32_t SEGS = SW_SLAB / 16;  // 16-byte pieces per row and slab
            for (uint32_t idx = lane; idx < nbg * SEGS; idx += 32) {
              const uint32_t rr = idx / SEGS, seg = idx % SEGS;
              const uint32_t* tp = tile + rr * SW_TILE_ROW + seg * 4;
              *reinterpret_cast<uint4*>(sym_rows + size_t(rr) * BATCH_N + i0 + seg * 16) = make_uint4(tp[0], tp[1], tp[2], tp[3]);
            }
          }
          __syncwarp();
        }
        bit = (blk << 7) + wpos;
      }
      if (mine) offs[b] = uint32_t(min(bit, src.n_bits) - chunk_bit0);
    }
  }
}

// ---------------------------------------------------------------------------
// decode_kernel: one CTA per chunk, one warp per batch; symbols and section starts come from symwalk_kernel.
// ---------------------------------------------------------------------------
// NV = latent vars of the chunks this instantiation serves (1: classic, 2: int_mult / float_mult / float_quant); the
// host launches both and a CTA leaves at once when its chunk belongs to the other (symwalk_kernel recorded each
// chunk's var count) - one-var chunks then run with the registers of one var and a third CTA per SM.
template <typename L, int NV>
__global__ void __launch_bounds__(DEC_THREADS, NV == 1 ? PCOB_DEC_NV1_BLOCKS : 2)
decode_kernel(FileParams fp, const IndexChunk* __restrict__ chunks, uint32_t* __restrict__ statuses, const uint8_t* __restrict__ index_base, uint64_t index_len,
              L* __restrict__ out, uint64_t out_len, const Binoms* __restrict__ binoms, const uint8_t* __restrict__ d_syms,
              const uint32_t* __restrict__ d_offs, const uint8_t* __restrict__ d_nvars, const uint32_t* __restrict__ gate) {
  if (gate_closed(gate, fp)) return;
  if (d_nvars[blockIdx.x] != NV) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  DecodeSmem& sm = *reinterpret_cast<DecodeSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const IndexChunk task = chunks[blockIdx.x];
  const BitSrc src = make_bitsrc(fp.src, fp.src_len);
  const uint64_t max_word = src.n_bits == 0 ? 0 : (src.n_bits - 1) >> 6;
  const uint64_t chunk_bit0 = src.mis_bits + task.chunk_offset * 8;
  const bool is_float = nt_is_float(fp.dtype), is_signed = nt_is_signed(fp.dtype);
#ifdef PCOB_DEC_TIMING
  long long _tprev = clock64();
  unsigned long long _tacc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#endif

  if (tid == 0) {
    sm.err = 0;
    parse_chunk_header(src, chunk_bit0, fp.dtype, fp.uniform_type, fp.format_major, true, sm.hdr);
    if (sm.hdr.status == ST_OK) {
      for (uint32_t v = 0; v < sm.hdr.n_vars; v++) {
        const VarHdr& vh = sm.hdr.var[v];
        if (vh.ans_size_log > SMALL_MAX_SIZE_LOG || vh.n_bins > SMALL_MAX_BINS) sm.hdr.status = ST_UNSUPPORTED;
        if (v > 0 && vh.delta_order > 0) sm.hdr.status = ST_UNSUPPORTED;  // secondary_uses_delta: never written by pco
        if (vh.n_bins == 0 && var_stored_n(sm.hdr.n, vh.delta_order) > 0) sm.hdr.status = ST_CORRUPTION;
      }
      if (sm.hdr.mode == MODE_FLOAT_MULT && LT<L>::BITS < 32) sm.hdr.status = ST_UNSUPPORTED;
      if (task.n != 0 && task.n != sm.hdr.n) sm.hdr.status = ST_CORRUPTION;
      if (sm.hdr.n_vars != NV) sm.hdr.status = ST_CORRUPTION;  // cannot happen: symwalk_kernel parsed the same bytes
    }
  }
  for (int i = tid; i < CHAIN_RING; i += DEC_THREADS) sm.m_flag[i] = 0;
  for (int i = tid; i < 32 * MAX_ORDER; i += DEC_THREADS) sm.binom_lane8[i / MAX_ORDER][i % MAX_ORDER] = binoms->lane8[i / MAX_ORDER][i % MAX_ORDER];
  if (tid < MAX_ORDER) sm.binom_full[tid] = binoms->full[tid];
  __syncthreads();
  if (sm.hdr.status != ST_OK) {
    if (tid == 0) statuses[blockIdx.x] = sm.hdr.status;
    return;
  }
  constexpr uint32_t n_vars = NV;
  for (uint32_t v = 0; v < n_vars; v++)
    build_var_tables<false>(src, sm.hdr, v, nullptr, sm.build.bin_lower[v], sm.build.bin_ob[v], sm.build.bin_weight[v], sm.build.bin_cum[v],
                            sm.build.sym_of_state[v], sm.build.rank_counter[v], &sm.err, /*add_mid_to_lower=*/sm.hdr.var[v].delta_order > 0,
                            /*build_nodes=*/false);
  __syncthreads();
  if (sm.err) {
    if (tid == 0) statuses[blockIdx.x] = sm.err;
    return;
  }
  for (uint32_t v = 0; v < n_vars; v++) {
    const uint32_t nbv = max(sm.hdr.var[v].n_bins, 1u);
    for (uint32_t i = tid; i < nbv; i += DEC_THREADS) {
      BinEntry be;
      be.lower = sm.build.bin_lower[v][i];
      be.ob = sm.build.bin_ob[v][i];
      be.mask = be.ob >= 32 ? 0xffffffffu : ((1u << be.ob) - 1);
      sm.bin[v][i] = be;
    }
  }
  __syncthreads();
  if (tid < int(n_vars)) {
    // bins whose lowers span < 2^25 (deltas around a centre, small alphabets, ...) get a 4-byte table entry: one
    // shared-memory wavefront per lookup instead of four
    const uint32_t v = tid, nbv = max(sm.hdr.var[v].n_bins, 1u);
    const uint64_t lmask = LT<L>::BITS == 64 ? ~uint64_t(0) : ((uint64_t(1) << LT<L>::BITS) - 1);
    uint64_t base = sm.bin[v][0].lower;
    bool ok = true;
    // lowers ascend in symbol order for every stream pco writes; measure the span relative to the first bin
    for (uint32_t i = 0; i < nbv; i++) {
      const uint64_t d = (sm.bin[v][i].lower - base) & lmask;
      if (d >= (1u << 25)) ok = false;
    }
    sm.bin_base[v] = base;
    sm.bin_compact[v] = ok ? 1u : 0u;
    if (ok)
      for (uint32_t i = 0; i < nbv; i++) sm.bin32[v][i] = uint32_t((sm.bin[v][i].lower - base) & lmask) | (sm.bin[v][i].ob << 25);
  }

  const uint32_t n = sm.hdr.n;
  // pco::standalone::simple_decompress_into semantics: emit only what fits in the destination
  const uint32_t n_out = task.out_offset >= out_len ? 0u : uint32_t(min(uint64_t(n), out_len - task.out_offset));
  const uint32_t nb_total = n_batches_of(n);
  const uint32_t nb_out = n_batches_of(n_out);
  const uint32_t order = sm.hdr.var[0].delta_order;
  const bool need_index = (sm.hdr.var[0].n_bins > 1) || (n_vars > 1 && sm.hdr.var[1].n_bins > 1);
  const BatchEntry* entries = (task.entries_offset != 0 && index_base)
                                  ? reinterpret_cast<const BatchEntry*>(index_base + task.entries_offset) : nullptr;
  if (need_index && (!entries || task.entries_offset > index_len ||
                     uint64_t(n_vars) * nb_total * sizeof(BatchEntry) > index_len - task.entries_offset)) {
    if (tid == 0) statuses[blockIdx.x] = ST_INVALID_ARGUMENT;  // no index, or one that does not cover this chunk (stale / foreign)
    return;
  }
  // closed-form section sizes when every var is trivial (n_bins <= 1)
  const uint32_t ob0 = sm.hdr.var[0].n_bins >= 1 ? sm.build.bin_ob[0][0] : 0;
  const uint32_t ob1 = (n_vars > 1 && sm.hdr.var[1].n_bins >= 1) ? sm.build.bin_ob[1][0] : 0;
  const uint32_t stored0 = var_stored_n(n, sm.hdr.var[0].delta_order);
  const uint32_t stored1 = n_vars > 1 ? var_stored_n(n, sm.hdr.var[1].delta_order) : 0;

  if (tid == 0 && order > 0) {
    for (uint32_t k = 0; k < order; k++) sm.mvec[0][k] = sm.hdr.moments[0][k];
    __threadfence_block();
    sm.m_flag[0] = 1;
  }
  __syncthreads();  // tables, bin entries and the chain seed are in place; the build scratch (aliased by the tile) is dead

  PCOB_TICK(0);  // prologue
  const int kind = is_float ? 2 : (is_signed ? 1 : 0);
  const uint32_t mode = sm.hdr.mode;
  uint32_t end_err = 0;
  const uint64_t row0 = scratch_row0(task.out_offset, blockIdx.x);
  // chunk-relative bit position of batch b's offsets section for var v
  auto off_of = [&](uint32_t v, uint32_t b) -> uint32_t {
    if (need_index) return d_offs[row0 + size_t(v) * nb_out + b];
    // all vars trivial: batches before b contribute count0*ob0 + count1*ob1 bits
    const uint64_t c0 = min(uint64_t(b) * BATCH_N, uint64_t(stored0));
    const uint64_t c1 = min(uint64_t(b) * BATCH_N, uint64_t(stored1));
    uint64_t before = c0 * ob0 + c1 * ob1;
    if (v == 1) before += uint64_t(batch_count(stored0, b)) * ob0;
    return uint32_t(min(sm.hdr.body_bit + before, src.n_bits) - chunk_bit0);
  };
  // ---------------- one warp per batch ----------------
  // A batch's offset bits are one contiguous run of the stream.  Each warp copies a 512-byte window of it with two
  // coalesced 8-byte loads per lane -- issued one batch ahead so the DRAM/L2 latency hides behind the previous
  // batch -- parks it in shared memory and extracts the variable-width fields from there.  The section starts and the
  // symbols (8 per lane) were produced by symwalk_kernel.
  {
    uint64_t pf[NV][2];
    uint32_t off_cur[NV] = {}, off_nxt[NV] = {};
    uint2 sy_nxt[NV];
    auto issue_window_loads = [&](const uint32_t (&off)[NV]) {
#pragma unroll
      for (uint32_t v = 0; v < NV; v++) {
        if (v < n_vars && sm.hdr.var[v].max_offset_bits > 0) {
          const uint64_t wb = (chunk_bit0 + off[v]) >> 6;
          const uint64_t i0 = wb + lane, i1 = wb + 32 + lane;
          pf[v][0] = __ldg(src.words + (i0 <= max_word ? i0 : max_word));
          pf[v][1] = __ldg(src.words + (i1 <= max_word ? i1 : max_word));
        }
      }
    };
    auto load_syms = [&](uint32_t b) {
#pragma unroll
      for (uint32_t v = 0; v < NV; v++) {
        sy_nxt[v] = make_uint2(0u, 0u);
        if (v < n_vars && sm.hdr.var[v].n_bins > 1)
          sy_nxt[v] = __ldg(reinterpret_cast<const uint2*>(d_syms + (row0 + size_t(v) * nb_out + b) * BATCH_N) + lane);
      }
    };
    if (uint32_t(warp) < nb_out) {
#pragma unroll
      for (uint32_t v = 0; v < NV; v++) if (v < n_vars) off_cur[v] = off_of(v, warp);
      issue_window_loads(off_cur);
      load_syms(warp);
      if (uint32_t(warp) + DEC_WARPS < nb_out) {
#pragma unroll
        for (uint32_t v = 0; v < NV; v++) if (v < n_vars) off_nxt[v] = off_of(v, warp + DEC_WARPS);
      }
    }
    for (uint32_t b = warp; b < nb_out; b += DEC_WARPS) {
      const uint32_t out_cnt = min(uint32_t(BATCH_N), n_out - b * BATCH_N);  // numbers this batch emits
      __syncwarp();
#pragma unroll
      for (uint32_t v = 0; v < NV; v++) {
        if (v < n_vars && sm.hdr.var[v].max_offset_bits > 0) {
          uint2* w2 = reinterpret_cast<uint2*>(sm.win[warp][v]);
          w2[lane] = make_uint2(uint32_t(pf[v][0]), uint32_t(pf[v][0] >> 32));
          w2[32 + lane] = make_uint2(uint32_t(pf[v][1]), uint32_t(pf[v][1] >> 32));
        }
      }
      __syncwarp();
      uint2 sy_cur[NV];
#pragma unroll
      for (uint32_t v = 0; v < NV; v++) sy_cur[v] = sy_nxt[v];
      uint32_t off_n2[NV] = {};
      if (b + DEC_WARPS < nb_out) {
        issue_window_loads(off_nxt);
        load_syms(b + DEC_WARPS);
        if (b + 2 * DEC_WARPS < nb_out) {
#pragma unroll
          for (uint32_t v = 0; v < NV; v++) if (v < n_vars) off_n2[v] = off_of(v, b + 2 * DEC_WARPS);
        }
      }
      PCOB_TICK(3);  // window staging
      L lat[NV][8];
      uint64_t last_end = 0;
#pragma unroll
      for (uint32_t v = 0; v < NV; v++) {
        if (v >= n_vars) break;
        const VarHdr& vh = sm.hdr.var[v];
        const uint32_t cnt = batch_count(v == 0 ? stored0 : stored1, b);
        const bool full = cnt == BATCH_N;
        uint32_t sy[8];
        {
          const uint32_t p0 = sy_cur[v].x, p1 = sy_cur[v].y;  // zero when the var has one bin
#pragma unroll
          for (int e = 0; e < 8; e++) sy[e] = ((e < 4 ? p0 : p1) >> (8 * (e & 3))) & 0xffu;
        }
        const bool compact = sm.bin_compact[v] != 0;
        if (compact && vh.max_offset_bits <= 32) {
          // ---- fast path: 4-byte bin entries (lower - base | offset_bits << 25) and fields of <= 32 bits.  The lane keeps
          // the 8 packed entries, finds its bit span by the warp scan, pulls the 4 words that cover a span of <= 96 bits
          // once, and peels the fields off the low end of that register window.
          const uint32_t bin_sa = smem_addr(&sm.bin32[v][0]);
          uint32_t q[8];
          uint32_t lane_bits = 0;
#pragma unroll
          for (int e = 0; e < 8; e++) {
            q[e] = lds_u32(bin_sa + 4 * sy[e]);
            if (!full && uint32_t(lane * 8 + e) >= cnt) q[e] &= 0x1ffffffu;
            lane_bits += q[e] >> 25;
          }
          uint32_t inc = lane_bits;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += o;
          }
          const uint32_t total_bits = __shfl_sync(0xffffffffu, inc, 31);
          const uint64_t sec_bit = chunk_bit0 + off_cur[v];
          if (total_bits <= WIN_USABLE_BITS && !__any_sync(0xffffffffu, lane_bits > 96)) {
            last_end = sec_bit + total_bits;
            const L base = L(sm.bin_base[v]);
            const uint32_t p = uint32_t(sec_bit & 63) + (inc - lane_bits);
            const uint32_t wa = smem_addr(sm.win[warp][v]) + 4 * (p >> 5), r = p & 31;
            uint32_t x0 = lds_u32(wa), x1 = lds_u32(wa + 4), x2 = lds_u32(wa + 8);
            const uint32_t x3 = lds_u32(wa + 12);
            x0 = __funnelshift_r(x0, x1, r); x1 = __funnelshift_r(x1, x2, r); x2 = __funnelshift_r(x2, x3, r);
#pragma unroll
            for (int e = 0; e < 8; e++) {
              const uint32_t ob = q[e] >> 25;
              uint32_t f;
              asm("bfe.u32 %0, %1, 0, %2;" : "=r"(f) : "r"(x0), "r"(ob));
              lat[v][e] = L(L(base + L(q[e] & 0x1ffffffu)) + L(f));
              x0 = __funnelshift_rc(x0, x1, ob); x1 = __funnelshift_rc(x1, x2, ob); x2 = __funnelshift_rc(x2, 0u, ob);
            }
            continue;
          }
        }
        // ---- bins: offset bits and lower bound of every latent
        uint32_t obv[8];
        L lowv[8];
        uint32_t lane_bits = 0;
        if (compact) {
          const L base = L(sm.bin_base[v]);
#pragma unroll
          for (int e = 0; e < 8; e++) {
            const uint32_t q = sm.bin32[v][sy[e]];
            obv[e] = q >> 25;
            lowv[e] = L(base + L(q & 0x1ffffffu));
          }
        } else {
#pragma unroll
          for (int e = 0; e < 8; e++) {
            const uint4 q = *reinterpret_cast<const uint4*>(&sm.bin[v][sy[e]]);
            lowv[e] = L((uint64_t(q.y) << 32) | q.x);
            obv[e] = q.z;
          }
        }
#pragma unroll
        for (int e = 0; e < 8; e++) {
          if (!full && uint32_t(lane * 8 + e) >= cnt) obv[e] = 0;
          lane_bits += obv[e];
        }
        uint32_t inc = lane_bits;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
          if (lane >= d) inc += o;
        }
        const uint32_t total_bits = __shfl_sync(0xffffffffu, inc, 31);
        const uint64_t sec_bit = chunk_bit0 + off_cur[v];
        last_end = sec_bit + total_bits;
        if (vh.max_offset_bits == 0) {
#pragma unroll
          for (int e = 0; e < 8; e++) lat[v][e] = lowv[e];
        } else if (total_bits <= WIN_USABLE_BITS) {
          const uint32_t* win = sm.win[warp][v];
          uint32_t p = uint32_t(sec_bit & 63) + (inc - lane_bits);
          const bool narrow = LT<L>::BITS <= 32 || vh.max_offset_bits <= 32;
          if (narrow && !__any_sync(0xffffffffu, lane_bits > 64)) {
            // the lane's 8 fields are contiguous and span <= 64 bits: fetch its 3 words once, extract from registers
            const uint32_t w = p >> 5;
            const uint32_t x0 = win[w], x1 = win[w + 1], x2 = win[w + 2];
            uint32_t pos = p & 31;
#pragma unroll
            for (int e = 0; e < 8; e++) {
              const uint32_t wd = pos >> 5, rr = pos & 31;
              const uint32_t lo = wd == 0 ? x0 : (wd == 1 ? x1 : x2);
              const uint32_t hi = wd == 0 ? x1 : (wd == 1 ? x2 : 0u);
              const uint32_t f = __funnelshift_r(lo, hi, rr) & uint32_t(~(~uint64_t(0) << obv[e]));
              lat[v][e] = L(lowv[e] + L(f));
              pos += obv[e];
            }
          } else if (narrow) {
#pragma unroll
            for (int e = 0; e < 8; e++) {
              lat[v][e] = L(lowv[e] + win_extract<L, false>(win, p, obv[e], uint32_t(~(~uint64_t(0) << obv[e]))));
              p += obv[e];
            }
          } else {
#pragma unroll
            for (int e = 0; e < 8; e++) {
              lat[v][e] = L(lowv[e] + win_extract<L, true>(win, p, obv[e], uint32_t(~(~uint64_t(0) << min(obv[e], 32u)))));
              p += obv[e];
            }
          }
        } else {
          // section longer than the staged window (mean offset > ~15.7 bits): read the stream directly
          uint64_t pos = sec_bit + (inc - lane_bits);
#pragma unroll
          for (int e = 0; e < 8; e++) {
            L off = 0;
            if (obv[e] != 0) off = read_offset<L>(src.words, max_word, min(pos, src.n_bits), obv[e]);
            pos += obv[e];
            lat[v][e] = L(lowv[e] + off);
          }
        }
        // positions past the stored latents of a delta'd var hold deltas that cannot influence any emitted
        // number (page_latent_decompressor.rs:244-248); any value works there
      }
      PCOB_TICK(4);  // symbols, bins, scan, extraction
      L* dst = out + task.out_offset + size_t(b) * BATCH_N + lane * 8;
      if (order > 0) {
        // ---- un-delta of the primary (delta/consecutive.rs:35-50)
        PCOB_TICK(5);
        switch (order) {
          case 1: undelta_chain<L, 1>(lat[0], sm, b, lane); break;
          case 2: undelta_chain<L, 2>(lat[0], sm, b, lane); break;
          // orders >= 3 are rare: out of line, so that their moment vectors do not set the kernel's register budget
          case 3: undelta_chain_cold<L, 3>(lat[0], sm, b, lane); break;
          case 4: undelta_chain_cold<L, 4>(lat[0], sm, b, lane); break;
          case 5: undelta_chain_cold<L, 5>(lat[0], sm, b, lane); break;
          case 6: undelta_chain_cold<L, 6>(lat[0], sm, b, lane); break;
          default: undelta_chain_cold<L, 7>(lat[0], sm, b, lane); break;
        }
        PCOB_TICK(6);  // scans + chain wait + link + fold
      }
      {
        // ---- join (mode/*.rs)
        L res[8];
        if (mode == MODE_CLASSIC) {
#pragma unroll
          for (int e = 0; e < 8; e++) res[e] = from_latent_kind<L>(lat[0][e], kind);
        } else if (NV > 1 && mode == MODE_INT_MULT) {
          const L base = L(sm.hdr.mode_base);
#pragma unroll
          for (int e = 0; e < 8; e++) res[e] = from_latent_kind<L>(L(L(lat[0][e] * base) + lat[NV - 1][e]), kind);
        } else if (NV > 1 && mode == MODE_FLOAT_MULT) {
          constexpr L MID = L(L(1) << (LT<L>::BITS - 1));
          const L base_bits = from_latent_ordered<L>(L(sm.hdr.mode_base), true, false);
#pragma unroll
          for (int e = 0; e < 8; e++) {
            const L un = float_mult_unadjusted(lat[0][e], base_bits);
            const L u = to_latent_ordered<L>(un, true, false);
            res[e] = from_latent_kind<L>(L(L(u + lat[NV - 1][e]) + MID), 2);
          }
        } else if (NV > 1) {  // MODE_FLOAT_QUANT
          const uint32_t k = sm.hdr.mode_k;
          constexpr L MID = L(L(1) << (LT<L>::BITS - 1));
          const L sign_cutoff = L(MID >> k);
          const L kmax = L(L(L(1) << k) - 1);
#pragma unroll
          for (int e = 0; e < 8; e++) {
            const L pq = lat[0][e];
            const L lowest = pq >= sign_cutoff ? lat[NV - 1][e] : L(kmax - lat[NV - 1][e]);
            res[e] = from_latent_kind<L>(L(L(pq << k) + lowest), 2);
          }
        }
        if (out_cnt == BATCH_N && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
          store8<L>(dst, res);  // 16-byte stores; a chunk that starts at an odd element offset takes the element-wise path
        } else {
#pragma unroll
          for (int e = 0; e < 8; e++)
            if (uint32_t(lane * 8 + e) < out_cnt) dst[e] = res[e];
        }
      }
      PCOB_TICK(7);  // chain link, moments, join, store
      // ---- end-of-page checks by the warp that owns the last batch (page_decompressor.rs:184-188)
      if (b == nb_total - 1 && lane == 0) {
        const uint64_t bit = last_end;
        if (bit > src.n_bits) end_err = ST_INSUFFICIENT_DATA;
        else {
          const uint32_t pad = uint32_t((8 - (bit & 7)) & 7);
          if (pad && read_bits_safe(src, bit, pad) != 0) end_err = ST_CORRUPTION;
        }
      }
#pragma unroll
      for (uint32_t v = 0; v < NV; v++) { off_cur[v] = off_nxt[v]; off_nxt[v] = off_n2[v]; }
    }
  }
  PCOB_TICK(8);  // loop tail
#ifdef PCOB_DEC_TIMING
  if (lane == 0)
    for (int i = 0; i < 10; i++) atomicAdd(&g_dec_timing[i], _tacc[i]);
#endif
  if (end_err) atomicMax(&sm.err, end_err);
  __syncthreads();
  if (tid == 0) statuses[blockIdx.x] = sm.err;
}

}  // namespace pcob200
