// fused_narrow_kernel: K7a + K7b + K8 + K9 in ONE kernel for the chunks that delta coding usually produces (the narrow
// class of decode_narrow.cuh: classic mode, consecutive order 0 / 1, 2..256 bins whose lowers lie within 2^16 of the first
// and whose offsets take <= 15 bits, 32- and 64-bit number types).
//
// One CTA of 8 warps per chunk:
//   * prologue: the chunk's first 4 KiB (header, bins, page meta) arrive in shared memory by ONE bulk copy
//     (cp.async.bulk + mbarrier transaction count - the TMA engine, no register staging); thread 0 parses the header out of
//     shared memory, the CTA builds the decoder nodes and the packed bin table and classifies the chunk.  A chunk that is
//     not of the narrow class only gets its class byte; the host then runs symwalk_kernel + decode_kernel for those.
//   * FZ_WALKERS walker warps (page_latent_decompressor.rs:89-177): a lane per batch, 32 consecutive batches at a time; a walker stages the
//     tANS bytes of its lanes with cp.async rows, walks 4 interleaved chains per lane and writes the bin indices into a
//     shared-memory ring (FZ_NBUF buffers of 32 symbol rows), together with the bit position where each batch's offsets
//     section starts.  full/empty mbarriers carry the hand-over.
//   * the other (FZ_DECODERS) warps decode, a warp per batch in batch order (page_latent_decompressor.rs:15-44, delta/consecutive.rs:35-50,
//     mode/classic.rs:14-24): symbols from the ring, the offsets window by cp.async one batch ahead, fields peeled off
//     register windows, the order-1 un-delta as one 32-bit scan + the fence-free carry record, 32-byte stores.
// Compared with symwalk_kernel + decode_narrow_kernel the symbol bytes never leave the SM (no 0.27 GB scratch written and
// read back), the section starts are not stored, the header is parsed once, and the compressed bytes are read by one kernel.
#pragma once
#include "decode_narrow.cuh"

namespace pcob200 {

#ifndef PCOB_FZ_NBUF
#define PCOB_FZ_NBUF 3
#endif
#ifndef PCOB_FZ_WALKERS
#define PCOB_FZ_WALKERS 2
#endif
// measured on C2 (1024 chunks x 2^18 u64, profiles/r02_c_fused_variants.txt), kernel / decompress call in ms:
//   1 walker, 2 buffers, rows of 64: 1.010 / 1.068    2 walkers, 3 buffers, rows of 64: 0.676 / 0.753    rows of 128: 0.658 / 0.727
//   3 walkers (5 decoders): 0.706 / 0.823             2 walkers, 2 buffers: 0.734 / 0.812              rows of 256 (3 CTAs/SM): 0.708 / 0.786
//   round-1 pair symwalk_kernel + decode_narrow_kernel: 0.751 / 0.823
#ifndef PCOB_FZ_ROW_SYMS
#define PCOB_FZ_ROW_SYMS 128
#endif
#ifndef PCOB_FZ_NODE_WORDS
#define PCOB_FZ_NODE_WORDS 2048
#endif
#ifndef PCOB_FZ_MIN_BLOCKS
#define PCOB_FZ_MIN_BLOCKS 4
#endif
#ifndef PCOB_FZ_THREADS
#define PCOB_FZ_THREADS 256
#endif
constexpr int FZ_THREADS = PCOB_FZ_THREADS;
constexpr int FZ_WARPS = FZ_THREADS / 32;
static_assert(FZ_WARPS == 8 || FZ_WARPS == 4, "the role rotation below masks with FZ_WARPS - 1");
constexpr int FZ_WALKERS = PCOB_FZ_WALKERS;          // walker warps: walker w takes the groups g = w (mod FZ_WALKERS)
constexpr int FZ_DECODERS = FZ_WARPS - FZ_WALKERS;
constexpr int FZ_NBUF = PCOB_FZ_NBUF;               // ring buffers of 32 symbol rows: group g lives in buffer g mod FZ_NBUF
// a walker lane's stage row: the bytes its next FZ_ROW_SYMS symbols can read (<= 10 bits each + 16 bytes of start alignment + the
// window's over-read), refilled with 16-byte cp.async from its exact position
constexpr int FZ_ROW_SYMS = PCOB_FZ_ROW_SYMS;
constexpr int FZ_ROW_BLOCKS = ((FZ_ROW_SYMS * SMALL_MAX_SIZE_LOG / 8 + 15) / 16 + 2) | 1;  // odd: rows start in different banks
constexpr int FZ_STAGE_WORDS = 32 * FZ_ROW_BLOCKS * 4;
static_assert(BATCH_N % FZ_ROW_SYMS == 0, "a batch is a whole number of stage rows");
static_assert(FZ_NBUF >= 2 && FZ_NBUF >= FZ_WALKERS, "every walker needs a buffer to work on");
constexpr int FZ_ROW_WORDS = 65;                     // 256 symbol bytes + 1 word: odd stride, a lane per row writes conflict-free
constexpr int FZ_BUF_WORDS = 32 * FZ_ROW_WORDS;
constexpr int FZ_NODE_WORDS = PCOB_FZ_NODE_WORDS;    // decoder nodes, replicated when the table is small
constexpr int FZ_HEAD_BYTES = 4096;                  // bulk-staged head of the chunk: header + <= 256 bins + page meta of one var
constexpr int FZ_RING = 32;                          // carry-chain slots (> batches in flight)
constexpr int FZ_MRING = 16;                         // moment-chain slots for delta orders >= 2

// ---- mbarrier / bulk-copy primitives (shared::cta addresses as 32-bit values) ----
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 t;\n\tmbarrier.arrive.shared::cta.b64 t, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 t;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 t, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
#ifndef PCOB_FZ_WAIT_NS
#define PCOB_FZ_WAIT_NS 0
#endif
// A waiting warp must not eat the issue slots of the warps it waits for: between two failed tries it sleeps (PCOB_FZ_WAIT_NS > 0).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
#if PCOB_FZ_WAIT_NS > 0
  while (!mbar_test(bar, parity)) __nanosleep(PCOB_FZ_WAIT_NS);
#elif defined(PCOB_FZ_TRYWAIT_HINT_NS)
  // try_wait with a suspend-time hint: the warp may sleep in hardware up to that long and is woken by the phase completion
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}" ::"r"(bar), "r"(parity), "r"(uint32_t(PCOB_FZ_TRYWAIT_HINT_NS)) : "memory");
#else
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
#endif
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

struct FusedSmem {
  ChunkHdr hdr;
  uint32_t q[SMALL_MAX_BINS];                       // offset_bits | (lower - lower_0) << 7
  uint32_t node[FZ_NODE_WORDS];
  union {
    alignas(16) uint64_t link[FZ_RING][2];          // order 1 carry chain: {first number of batch b, b + 1}
    struct {                                        // orders >= 2: mvec[b % FZ_MRING] = true moments at the start of batch b once m_flag[...] == b + 1
      uint64_t mvec[FZ_MRING][MAX_ORDER];
      volatile uint32_t m_flag[FZ_MRING];
    } mo;
  };
  alignas(8) uint64_t full_bar[FZ_NBUF], empty_bar[FZ_NBUF], head_bar;
  uint32_t ring_off[FZ_NBUF][32];                   // chunk-relative bit position of each batch's offsets section
  uint32_t err, not_narrow;
  uint64_t base, moment0;
  union {
    struct {                                        // prologue only
      alignas(16) uint8_t head[FZ_HEAD_BYTES + 16];
      BuildScratch build;
      uint32_t node_plain[1 << SMALL_MAX_SIZE_LOG];
    } pro;
    struct {
      uint32_t ring[FZ_NBUF][FZ_BUF_WORDS];
      alignas(16) uint32_t stage[FZ_WALKERS][FZ_STAGE_WORDS + 16];
      alignas(16) uint32_t win[FZ_DECODERS][2][NW_WIN_WORDS];
    } run;
  };
};

// The walker warp: lane k walks batch 32 g + k of group g.
__device__ __forceinline__ void fused_walker(FusedSmem& sm, const BitSrc& src, uint64_t chunk_bit0, const BatchEntry* __restrict__ entries, uint32_t nb_out,
                                             uint32_t stored, uint32_t size_log, uint32_t rep_log, int walker, int lane) {
  const uint64_t max_blk = (src.n_bits == 0 ? 0 : (src.n_bits - 1) >> 6) >> 1;
  const uint32_t node_sa = smem_addr(sm.node + (uint32_t(lane) & ((1u << rep_log) - 1)));  // this lane's copy
  const uint32_t sl = rep_log + 2;                                                           // states are byte offsets into the lane's copy
  const uint32_t smask = (1u << size_log) - 1;
  const uint32_t stg_sa = smem_addr(sm.run.stage[walker]);
  const uint32_t row_g = stg_sa + uint32_t(lane) * (FZ_ROW_BLOCKS * 16);
  const uint32_t* rowp = sm.run.stage[walker] + lane * (FZ_ROW_BLOCKS * 4);
  const uint32_t groups = (nb_out + 31) / 32;
  BatchEntry e_nxt;
  e_nxt.bit_pos = 0; e_nxt.st[0] = e_nxt.st[1] = e_nxt.st[2] = e_nxt.st[3] = 0;
  if (uint32_t(walker) * 32 + lane < nb_out) e_nxt = entries[uint32_t(walker) * 32 + lane];
  for (uint32_t g = walker; g < groups; g += FZ_WALKERS) {
    const uint32_t rb = g % FZ_NBUF, ph = g / FZ_NBUF;
    const BatchEntry e = e_nxt;
    const uint32_t b = g * 32 + lane;
    const bool mine = b < nb_out;
    if (b + 32 * FZ_WALKERS < nb_out) e_nxt = entries[b + 32 * FZ_WALKERS];  // the walker's next entry is in flight while this group is walked
    if (ph > 0) mbar_wait(smem_addr(&sm.empty_bar[rb]), (ph - 1) & 1u);  // the decoders have taken group g - FZ_NBUF out of the buffer
    const int cnt = mine ? int(batch_count(stored, b)) : 0;
    uint32_t s0 = min(uint32_t(e.st[0]), smask) << sl, s1 = min(uint32_t(e.st[1]), smask) << sl;
    uint32_t s2 = min(uint32_t(e.st[2]), smask) << sl, s3 = min(uint32_t(e.st[3]), smask) << sl;
    const uint32_t row_sa = smem_addr(sm.run.ring[rb] + lane * FZ_ROW_WORDS);
    uint64_t bit = min(chunk_bit0 + e.bit_pos, src.n_bits);
    // word w of a row holds symbols 4w..4w+3; decoder lane l wants words 2l and 2l+1: even words go to slot l, odd ones to 32 + l
    auto slot = [](int i) -> uint32_t { return uint32_t(((i >> 3) + ((i & 4) << 3)) << 2); };  // byte offset of symbol group i (multiple of 4)
    for (int part = 0; part < BATCH_N / FZ_ROW_SYMS; part++) {
      const uint64_t blk = bit >> 7;
      if (cnt > part * FZ_ROW_SYMS) {
#pragma unroll
        for (uint32_t qd = 0; qd < uint32_t(FZ_ROW_BLOCKS); qd++) {
          const void* gp = reinterpret_cast<const ulonglong2*>(src.words) + min(blk + qd, max_blk);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(row_g + qd * 16), "l"(gp));
        }
      }
      asm volatile("cp.async.commit_group;");
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      uint32_t wpos = uint32_t(bit & 127);
      uint32_t w = wpos >> 5;
      uint32_t x0 = lds_u32(row_g + 4 * w), x1 = lds_u32(row_g + 4 * w + 4), x2 = lds_u32(row_g + 4 * w + 8);
      const int i0 = part * FZ_ROW_SYMS;
      if (size_log <= 8) {
#pragma unroll 4
        for (int i = i0; i < i0 + FZ_ROW_SYMS; i += 4) {
          if (i + 4 <= cnt) {
            const uint32_t n0 = lds_u32(node_sa + s0), n1 = lds_u32(node_sa + s1), n2 = lds_u32(node_sa + s2), n3 = lds_u32(node_sa + s3);
            const uint32_t gw = __funnelshift_r(x0, x1, wpos & 31);
            const uint32_t c0 = node_btr(n0), c1 = node_btr(n1), c2 = node_btr(n2), c3 = node_btr(n3);
            const uint32_t sh2 = c0 + c1, sh3 = sh2 + c2;
            s0 = (node_base(n0) + (gw & ((1u << c0) - 1))) << sl;
            s1 = (node_base(n1) + ((gw >> c0) & ((1u << c1) - 1))) << sl;
            s2 = (node_base(n2) + ((gw >> sh2) & ((1u << c2) - 1))) << sl;
            s3 = (node_base(n3) + ((gw >> sh3) & ((1u << c3) - 1))) << sl;
            sts_u32(row_sa + slot(i), node_fields4(n0, n1, n2, n3));
            wpos += sh3 + c3;
            if ((wpos >> 5) != w) { w = wpos >> 5; x0 = lds_u32(row_g + 4 * w); x1 = lds_u32(row_g + 4 * w + 4); }
          }
        }
      } else {
#pragma unroll 2
        for (int i = i0; i < i0 + FZ_ROW_SYMS; i += 4) {
          if (i + 4 <= cnt) {
            const uint32_t n0 = lds_u32(node_sa + s0), n1 = lds_u32(node_sa + s1), n2 = lds_u32(node_sa + s2), n3 = lds_u32(node_sa + s3);
            const uint32_t r = wpos & 31;
            const uint64_t gw = (uint64_t(__funnelshift_r(x1, x2, r)) << 32) | __funnelshift_r(x0, x1, r);
            const uint32_t c0 = node_btr(n0), c1 = node_btr(n1), c2 = node_btr(n2), c3 = node_btr(n3);
            const uint32_t sh2 = c0 + c1, sh3 = sh2 + c2;
            s0 = (node_base(n0) + (uint32_t(gw) & ((1u << c0) - 1))) << sl;
            s1 = (node_base(n1) + (uint32_t(gw >> c0) & ((1u << c1) - 1))) << sl;
            s2 = (node_base(n2) + (uint32_t(gw >> sh2) & ((1u << c2) - 1))) << sl;
            s3 = (node_base(n3) + (uint32_t(gw >> sh3) & ((1u << c3) - 1))) << sl;
            sts_u32(row_sa + slot(i), node_fields4(n0, n1, n2, n3));
            wpos += sh3 + c3;
            if ((wpos >> 5) != w) { w = wpos >> 5; x0 = lds_u32(row_g + 4 * w); x1 = lds_u32(row_g + 4 * w + 4); x2 = lds_u32(row_g + 4 * w + 8); }
          }
        }
      }
      if (cnt > i0 && cnt < i0 + FZ_ROW_SYMS && (cnt & 3)) {  // ragged tail of the page's last batch (page_latent_decompressor.rs:144-177)
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
        sts_u32(row_sa + slot(i), packed);
      }
      __syncwarp();  // every lane is done with its stage row before the next part's copies land
      bit = (blk << 7) + wpos;
    }
    if (mine) sm.ring_off[rb][lane] = uint32_t(min(bit, src.n_bits) - chunk_bit0);
    mbar_arrive(smem_addr(&sm.full_bar[rb]));  // 32 arrivals (release) complete the group's phase
  }
}

// Consecutive un-delta of order K >= 2 (delta/consecutive.rs:35-50) for a batch held 8 per lane: K nested zero-seeded warp scans, this
// warp's link of the moment chain m_{b+1} = A^256 m_b + c_b (A = I + superdiagonal, (A^n)_{j,j+t} = C(n, t)), then m_b folded into the
// lane's values by linearity - the general kernel's scheme (decode_kernels.cuh undelta_chain) with the binomials C(8 lane, t) and
// C(256, t) computed in registers (exact: < 2^40) instead of read from a table.
template <typename L, int K>
__device__ __forceinline__ void fused_undelta(L (&x)[8], FusedSmem& sm, uint32_t b, int lane) {
  L c[K];
  undelta_local<L, K>(x, c, lane);
  uint64_t bl[K], bf[K];
  bl[0] = 1;
  bf[0] = 1;
  const uint64_t n8 = uint64_t(lane) * 8;
#pragma unroll
  for (int t = 1; t < K; t++) {
    bl[t] = n8 + 1 >= uint64_t(t) + 1 && n8 >= uint64_t(t - 1) ? bl[t - 1] * (n8 - uint64_t(t - 1)) / uint64_t(t) : 0;  // C(n, t) = C(n, t-1) (n - t + 1) / t
    bf[t] = bf[t - 1] * uint64_t(256 - (t - 1)) / uint64_t(t);
  }
  const uint32_t slot = b % FZ_MRING, nslot = (b + 1) % FZ_MRING;
  while (sm.mo.m_flag[slot] != b + 1) {
  }
  __threadfence_block();
  L m[K];
#pragma unroll
  for (int k = 0; k < K; k++) m[k] = L(sm.mo.mvec[slot][k]);
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < K; j++) {
      L acc = c[j];
#pragma unroll
      for (int t = 0; j + t < K; t++) acc = L(acc + L(bf[t] * uint64_t(m[j + t])));
      sm.mo.mvec[nslot][j] = uint64_t(acc);
    }
    __threadfence_block();
    sm.mo.m_flag[nslot] = b + 2;
  }
  L sft[K];
#pragma unroll
  for (int j = 0; j < K; j++) {
    L acc = 0;
#pragma unroll
    for (int t = 0; j + t < K; t++) acc = L(acc + L(bl[t] * uint64_t(m[j + t])));
    sft[j] = acc;
  }
#pragma unroll
  for (int e = 0; e < 8; e++) {
    x[e] = L(x[e] + sft[0]);
#pragma unroll
    for (int j = 0; j + 1 < K; j++) sft[j] = L(sft[j] + sft[j + 1]);
  }
}

// A decoder warp: batches d, d + FZ_DECODERS, ... of the chunk (K = consecutive delta order, 0 or 1).
template <typename L, int K>
__device__ __forceinline__ void fused_decoder(FusedSmem& sm, const FileParams& fp, const BitSrc& src, const IndexChunk& task, uint64_t chunk_bit0, L* __restrict__ out,
                                              uint32_t n, uint32_t n_out, int d, int lane) {
  const uint64_t max_blk = (src.n_bits == 0 ? 0 : (src.n_bits - 1) >> 6) >> 1;
  const uint64_t cblk0 = chunk_bit0 >> 7;
  const uint32_t cbr = uint32_t(chunk_bit0 & 127);
  const uint32_t max_rel = max_blk > cblk0 ? uint32_t(min(max_blk - cblk0, uint64_t(0xffffffffu))) : 0u;
  const ulonglong2* __restrict__ chunk_blk = reinterpret_cast<const ulonglong2*>(src.words) + min(cblk0, max_blk);
  const uint32_t nb_total = n_batches_of(n), nb_out = n_batches_of(n_out);
  const uint32_t stored = var_stored_n(n, K);
  const L base = L(sm.base);
  const int kind = nt_is_float(fp.dtype) ? 2 : (nt_is_signed(fp.dtype) ? 1 : 0);
  const uint32_t q_sa = smem_addr(sm.q);
  const uint32_t win_sa = smem_addr(sm.run.win[d][0]);
  const uint32_t link_sa = smem_addr(&sm.link[0][0]);
  uint32_t end_err = 0;
  L* __restrict__ dst = out + task.out_offset + size_t(d) * BATCH_N + lane * 8;

  auto issue_window = [&](uint32_t off, uint32_t bufi) {
    const uint32_t rel = min(((cbr + off) >> 7) + uint32_t(lane), max_rel);
    const void* gp = chunk_blk + rel;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(win_sa + bufi * uint32_t(NW_WIN_WORDS * 4) + uint32_t(lane) * 16u), "l"(gp));
    asm volatile("cp.async.commit_group;");
  };
  // symbols (8 per lane) and section start of batch bb out of the ring; non-blocking variant for the look-ahead
  auto fetch = [&](uint32_t bb, uint32_t& off, uint2& sy, bool blocking) -> bool {
    const uint32_t g = bb >> 5, rb = g % FZ_NBUF, parity = (g / FZ_NBUF) & 1u;
    const uint32_t bar = smem_addr(&sm.full_bar[rb]);
    if (blocking) mbar_wait(bar, parity);
    else if (!__all_sync(0xffffffffu, mbar_test(bar, parity) ? 1 : 0)) return false;  // every lane acquires the phase itself
    const uint32_t row_sa = smem_addr(sm.run.ring[rb] + (bb & 31u) * FZ_ROW_WORDS);
    sy.x = lds_u32(row_sa + 4u * uint32_t(lane));
    sy.y = lds_u32(row_sa + 4u * (32u + uint32_t(lane)));
    off = sm.ring_off[rb][bb & 31u];
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_addr(&sm.empty_bar[rb]));
    return true;
  };

  uint32_t off_cur = 0, off_nxt = 0;
  uint2 sy_cur = make_uint2(0u, 0u), sy_nxt = make_uint2(0u, 0u);
  bool have = false;
  uint32_t buf = 0;
  for (uint32_t b = d; b < nb_out; b += FZ_DECODERS) {
    if (!have) {
      fetch(b, off_cur, sy_cur, true);
      issue_window(off_cur, buf);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();  // this batch's window is visible to the warp; every lane is done with the other buffer
    const uint2 sy = sy_cur;
    have = false;
    if (b + FZ_DECODERS < nb_out && fetch(b + FZ_DECODERS, off_nxt, sy_nxt, false)) {
      issue_window(off_nxt, buf ^ 1u);
      have = true;
    }
    const uint32_t cnt = batch_count(stored, b);
    // ---- bins of the lane's 8 latents
    uint32_t q[8];
    q[0] = lds_u32(q_sa + ((sy.x << 2) & 0x3fcu));
    q[1] = lds_u32(q_sa + ((sy.x >> 6) & 0x3fcu));
    q[2] = lds_u32(q_sa + ((sy.x >> 14) & 0x3fcu));
    q[3] = lds_u32(q_sa + ((sy.x >> 22) & 0x3fcu));
    q[4] = lds_u32(q_sa + ((sy.y << 2) & 0x3fcu));
    q[5] = lds_u32(q_sa + ((sy.y >> 6) & 0x3fcu));
    q[6] = lds_u32(q_sa + ((sy.y >> 14) & 0x3fcu));
    q[7] = lds_u32(q_sa + ((sy.y >> 22) & 0x3fcu));
    if (cnt != uint32_t(BATCH_N)) {  // the page's last batch: latents past the stored ones read no bits and add nothing
#pragma unroll
      for (int e = 0; e < 8; e++)
        if (uint32_t(lane * 8 + e) >= cnt) q[e] = 0;
    }
    uint32_t P[8];
    P[0] = q[0];
#pragma unroll
    for (int e = 1; e < 8; e++) P[e] = P[e - 1] + q[e];
    const uint32_t lane_bits = P[7] & 127u;
    uint32_t inc = lane_bits;
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) inc = scan_step_up(inc, dd);
    const uint32_t sec_rel = cbr + off_cur;  // bit position of the section, from the chunk's first 16-byte block
    uint32_t f[8];
    {
      const uint32_t wbase = win_sa + buf * uint32_t(NW_WIN_WORDS * 4);
      const uint32_t pa = (sec_rel & 127u) + (inc - lane_bits);
      const uint32_t pb = pa + (P[3] & 127u);
      const uint32_t wa = wbase + ((pa >> 5) << 2), wb = wbase + ((pb >> 5) << 2);
      const uint32_t a0 = lds_u32(wa), a1 = lds_u32(wa + 4), a2 = lds_u32(wa + 8);
      const uint32_t b0 = lds_u32(wb), b1 = lds_u32(wb + 4), b2 = lds_u32(wb + 8);
      uint32_t lo = shr_wrap(a0, a1, pa), hi = shr_wrap(a1, a2, pa);
#pragma unroll
      for (int e = 0; e < 4; e++) {
        f[e] = lo & ~ones_shl_wrap(q[e]);
        if (e < 3) {
          lo = shr_wrap(lo, hi, q[e]);
          hi = shr_wrap(hi, 0u, q[e]);
        }
      }
      lo = shr_wrap(b0, b1, pb);
      hi = shr_wrap(b1, b2, pb);
#pragma unroll
      for (int e = 4; e < 8; e++) {
        f[e] = lo & ~ones_shl_wrap(q[e]);
        if (e < 7) {
          lo = shr_wrap(lo, hi, q[e]);
          hi = shr_wrap(hi, 0u, q[e]);
        }
      }
    }
    L res[8];
    if (K == 0) {
#pragma unroll
      for (int e = 0; e < 8; e++) res[e] = L(base + L((q[e] >> 7) + f[e]));
    } else if (K >= 2) {
      // stored deltas (lower + offset, MID folded into base); positions past the page's stored latents hold values that cannot reach
      // an emitted number (page_latent_decompressor.rs:244-248)
#pragma unroll
      for (int e = 0; e < 8; e++) res[e] = L(base + L((q[e] >> 7) + f[e]));
      fused_undelta<L, (K >= 2 ? K : 2)>(res, sm, b, lane);
    } else {
      uint32_t F[8];
      F[0] = f[0];
#pragma unroll
      for (int e = 1; e < 8; e++) F[e] = F[e - 1] + f[e];
      const uint32_t T = (P[7] >> 7) + F[7];
      uint32_t incT = T;
#pragma unroll
      for (int dd = 1; dd < 32; dd <<= 1) incT = scan_step_up(incT, dd);
      const uint32_t totT = __shfl_sync(0xffffffffu, incT, 31);
      const uint32_t slot = b % FZ_RING, nslot = (b + 1) % FZ_RING;
      uint64_t m64, fl;
      for (;;) {
        asm volatile("ld.volatile.shared.v2.u64 {%0, %1}, [%2];" : "=l"(m64), "=l"(fl) : "r"(link_sa + 16 * slot) : "memory");
        if (fl == b + 1) break;
#ifdef PCOB_FZ_LINK_SLEEP_NS
        __nanosleep(PCOB_FZ_LINK_SLEEP_NS);
#endif
      }
      const L m = L(m64);
      if (lane == 0)
        asm volatile("st.volatile.shared.v2.u64 [%0], {%1, %2};" ::"r"(link_sa + 16 * nslot), "l"(uint64_t(L(L(m + L(uint64_t(base) << 8)) + L(totT)))),
                     "l"(uint64_t(b + 2)) : "memory");
      L D = L(L(m + L(uint64_t(base) * uint64_t(lane * 8))) + L(incT - T));
      res[0] = D;
#pragma unroll
      for (int e = 1; e < 8; e++) {
        D = L(D + base);
        res[e] = L(D + L((P[e - 1] >> 7) + F[e - 1]));
      }
    }
    if (kind != 0) {
#pragma unroll
      for (int e = 0; e < 8; e++) res[e] = from_latent_kind<L>(res[e], kind);
    }
    const uint32_t out_cnt = min(uint32_t(BATCH_N), n_out - b * BATCH_N);
    if (out_cnt == uint32_t(BATCH_N) && (reinterpret_cast<uintptr_t>(dst) & (sizeof(L) >= 4 ? 15 : sizeof(L) * 8 - 1)) == 0) {
      store8<L>(dst, res);
    } else {
#pragma unroll
      for (int e = 0; e < 8; e++)
        if (uint32_t(lane * 8 + e) < out_cnt) dst[e] = res[e];
    }
    dst += FZ_DECODERS * BATCH_N;
    if (b == nb_total - 1) {  // end-of-page checks by the warp that owns the last batch (page_decompressor.rs:184-188)
      const uint32_t total_bits = __shfl_sync(0xffffffffu, inc, 31);
      const uint64_t bit = (cblk0 << 7) + sec_rel + total_bits;
      if (lane == 0) {
        if (bit > src.n_bits) end_err = ST_INSUFFICIENT_DATA;
        else {
          const uint32_t pad = uint32_t((8 - (bit & 7)) & 7);
          if (pad && read_bits_safe(src, bit, pad) != 0) end_err = ST_CORRUPTION;
        }
      }
    }
    off_cur = off_nxt;
    sy_cur = sy_nxt;
    buf ^= 1u;
  }
  if (end_err) atomicMax(&sm.err, end_err);
}

// d_cls[c] on return: CLS_DONE | class = the chunk is done (decoded here as narrow order 0 / 1, or refused with its status
// written), 1 / 2 = it belongs to decode_kernel<L, 1 / 2> (symwalk_kernel + decode_kernel run for those).
template <typename L>
__global__ void __launch_bounds__(FZ_THREADS, PCOB_FZ_MIN_BLOCKS)
fused_narrow_kernel(FileParams fp, const IndexChunk* __restrict__ chunks, const uint8_t* __restrict__ index_base, uint64_t index_len,
                    uint32_t* __restrict__ statuses, uint8_t* __restrict__ d_cls, L* __restrict__ out, uint64_t out_len,
                    const uint32_t* __restrict__ gate) {
  if (gate_closed(gate, fp)) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FusedSmem& sm = *reinterpret_cast<FusedSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const IndexChunk task = chunks[blockIdx.x];
  const BitSrc src = make_bitsrc(fp.src, fp.src_len);
  const uint64_t chunk_bit0 = src.mis_bits + task.chunk_offset * 8;
  // ---- head of the chunk -> shared memory by one bulk copy
  const uint64_t max_blk = (src.n_bits == 0 ? 0 : (src.n_bits - 1) >> 6) >> 1;
  const uint64_t a0_blk = chunk_bit0 >> 7;
  const bool in_file = task.chunk_offset < fp.src_len;
  uint32_t head_bytes = 0;
  if (in_file) head_bytes = uint32_t(min(uint64_t(FZ_HEAD_BYTES), (max_blk - a0_blk + 1) * 16));
  if (tid == 0) {
    sm.err = 0;
    sm.not_narrow = 0;
    for (int i = 0; i < FZ_NBUF; i++) {
      mbar_init(smem_addr(&sm.full_bar[i]), 32);
      mbar_init(smem_addr(&sm.empty_bar[i]), 32);
    }
    mbar_init(smem_addr(&sm.head_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (head_bytes) {
      mbar_expect_tx(smem_addr(&sm.head_bar), head_bytes);
      bulk_g2s(smem_addr(sm.pro.head), reinterpret_cast<const ulonglong2*>(src.words) + a0_blk, head_bytes, smem_addr(&sm.head_bar));
    }
  }
  __syncthreads();
  if (head_bytes) mbar_wait(smem_addr(&sm.head_bar), 0);
  // the staged bytes as a bit source of their own; positions below are relative to it until `rebase`
  BitSrc hs;
  hs.words = reinterpret_cast<const uint64_t*>(sm.pro.head);
  hs.mis_bits = 0;
  hs.n_bits = in_file ? min(uint64_t(head_bytes) * 8, src.n_bits - (a0_blk << 7)) : 0;
  const uint64_t a0 = a0_blk << 7;
  const bool head_capped = uint64_t(head_bytes) * 8 < src.n_bits - min(src.n_bits, a0);  // the file goes on behind the staged bytes
  __shared__ uint32_t use_global;
  if (tid == 0) {
    use_global = 0;
    if (!in_file) {
      sm.hdr.status = ST_INVALID_ARGUMENT;  // the index points outside the file
    } else {
      parse_chunk_header(hs, chunk_bit0 - a0, fp.dtype, fp.uniform_type, fp.format_major, true, sm.hdr);
      if (sm.hdr.status == ST_INSUFFICIENT_DATA && head_capped) {  // header longer than the staged head: parse the file itself
        use_global = 1;
        parse_chunk_header(src, chunk_bit0, fp.dtype, fp.uniform_type, fp.format_major, true, sm.hdr);
      }
    }
    if (sm.hdr.status == ST_OK) {
      for (uint32_t v = 0; v < sm.hdr.n_vars; v++) {
        const VarHdr& vh = sm.hdr.var[v];
        if (vh.ans_size_log > SMALL_MAX_SIZE_LOG || vh.n_bins > SMALL_MAX_BINS) sm.hdr.status = ST_UNSUPPORTED;
        if (v > 0 && vh.delta_order > 0) sm.hdr.status = ST_UNSUPPORTED;  // secondary_uses_delta: never written by pco
        if (vh.n_bins == 0 && var_stored_n(sm.hdr.n, vh.delta_order) > 0) sm.hdr.status = ST_CORRUPTION;
      }
      if (sm.hdr.mode == MODE_FLOAT_MULT && LT<L>::BITS < 32) sm.hdr.status = ST_UNSUPPORTED;
      if (task.n != 0 && task.n != sm.hdr.n) sm.hdr.status = ST_CORRUPTION;
    }
  }
  __syncthreads();
  if (sm.hdr.status != ST_OK) {
    if (tid == 0) { statuses[blockIdx.x] = sm.hdr.status; d_cls[blockIdx.x] = CLS_DONE; }
    return;
  }
  const uint32_t n_vars = sm.hdr.n_vars;
  const VarHdr vh0 = sm.hdr.var[0];
  // everything the general kernels serve is handed over untouched
  const bool candidate = n_vars == 1 && sm.hdr.mode == MODE_CLASSIC && vh0.n_bins >= 2 &&
                         task.entries_offset != 0 && index_base != nullptr;
  if (!candidate) {
    if (tid == 0) { statuses[blockIdx.x] = 0xffffffffu; d_cls[blockIdx.x] = uint8_t(n_vars == 2 ? 2 : 1); }  // status: not decoded yet
    return;
  }
  {
    const BitSrc& bs = use_global ? src : hs;
    build_var_tables<false>(bs, sm.hdr, 0, sm.pro.node_plain, sm.pro.build.bin_lower[0], sm.pro.build.bin_ob[0], sm.pro.build.bin_weight[0], sm.pro.build.bin_cum[0],
                            sm.pro.build.sym_of_state[0], sm.pro.build.rank_counter[0], &sm.err, false);
  }
  __syncthreads();
  if (sm.err) {
    if (tid == 0) { statuses[blockIdx.x] = sm.err; d_cls[blockIdx.x] = CLS_DONE; }
    return;
  }
  if (sm.hdr.var[0].max_offset_bits > NARROW_MAX_OB) {
    if (tid == 0) { statuses[blockIdx.x] = 0xffffffffu; d_cls[blockIdx.x] = 1; }
    return;
  }
  {
    const uint64_t lmask = vh0.latent_bits == 64 ? ~uint64_t(0) : ((uint64_t(1) << vh0.latent_bits) - 1);
    const uint64_t lower0 = sm.pro.build.bin_lower[0][0];
    for (uint32_t i = tid; i < uint32_t(SMALL_MAX_BINS); i += FZ_THREADS) {
      uint32_t qv = 0;
      if (i < vh0.n_bins) {
        const uint64_t dlt = (sm.pro.build.bin_lower[0][i] - lower0) & lmask;
        if (dlt >> NARROW_LOW_BITS) sm.not_narrow = 1;
        qv = uint32_t(sm.pro.build.bin_ob[0][i]) | (uint32_t(dlt) << 7);
      }
      sm.q[i] = qv;
    }
    if (tid == 0) {
      const uint64_t mid = uint64_t(1) << (vh0.latent_bits - 1);
      sm.base = vh0.delta_order ? ((lower0 + mid) & lmask) : lower0;
      sm.moment0 = sm.hdr.moments[0][0];
    }
    // replicate the decoder nodes: copy r of state s at word s * R + r, lane l reads copy l mod R
    const uint32_t rep_log = min(5u, uint32_t(31 - __clz(uint32_t(FZ_NODE_WORDS) >> vh0.ans_size_log)));
    const uint32_t cells = (1u << vh0.ans_size_log) << rep_log;
    for (uint32_t i = tid; i < cells; i += FZ_THREADS) sm.node[i] = sm.pro.node_plain[i >> rep_log];
  }
  __syncthreads();  // q, nodes, base in place; the prologue scratch (aliased by ring, stage and windows) is dead
  if (sm.not_narrow) {
    if (tid == 0) { statuses[blockIdx.x] = 0xffffffffu; d_cls[blockIdx.x] = 1; }
    return;
  }
  const uint32_t n = sm.hdr.n;
  const uint32_t n_out = task.out_offset >= out_len ? 0u : uint32_t(min(uint64_t(n), out_len - task.out_offset));
  const uint32_t nb_total = n_batches_of(n), nb_out = n_batches_of(n_out);
  // an index that does not cover this chunk's batches cannot be walked (a stale or foreign index)
  if (task.entries_offset > index_len || uint64_t(nb_total) * sizeof(BatchEntry) > index_len - task.entries_offset) {
    if (tid == 0) { statuses[blockIdx.x] = ST_INVALID_ARGUMENT; d_cls[blockIdx.x] = CLS_DONE; }
    return;
  }
  const uint32_t K = vh0.delta_order;
  if (K <= 1) {
    if (tid < FZ_RING) {
      sm.link[tid][0] = tid == 0 ? sm.moment0 : 0;
      sm.link[tid][1] = (K == 1 && tid == 0) ? 1u : 0u;
    }
  } else {
    if (tid < FZ_MRING) sm.mo.m_flag[tid] = tid == 0 ? 1u : 0u;
    if (tid < int(K)) sm.mo.mvec[0][tid] = sm.hdr.moments[0][tid];
  }
  __syncthreads();
  // the walkers' warp slots rotate with the CTA so that the CTAs of an SM do not all put them on the same schedulers
  const int role = (warp + FZ_WARPS - int((blockIdx.x * FZ_WALKERS) & uint32_t(FZ_WARPS - 1))) & (FZ_WARPS - 1);  // 0 .. FZ_WALKERS - 1: walkers, the rest: decoders
  if (role < FZ_WALKERS) {
    const BatchEntry* entries = reinterpret_cast<const BatchEntry*>(index_base + task.entries_offset);
    const uint32_t rep_log = min(5u, uint32_t(31 - __clz(uint32_t(FZ_NODE_WORDS) >> vh0.ans_size_log)));
    fused_walker(sm, src, chunk_bit0, entries, nb_out, var_stored_n(n, K), vh0.ans_size_log, rep_log, role, lane);
  } else {
    const int d = role - FZ_WALKERS;
    switch (K) {
      case 0: fused_decoder<L, 0>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
      case 1: fused_decoder<L, 1>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
      case 2: fused_decoder<L, 2>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
      case 3: fused_decoder<L, 3>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
      case 4: fused_decoder<L, 4>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
      case 5: fused_decoder<L, 5>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
      case 6: fused_decoder<L, 6>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
      default: fused_decoder<L, 7>(sm, fp, src, task, chunk_bit0, out, n, n_out, d, lane); break;
    }
  }
  __syncthreads();
  if (tid == 0) { statuses[blockIdx.x] = sm.err; d_cls[blockIdx.x] = uint8_t(CLS_DONE | (K == 0 ? CLS_NARROW0 : K == 1 ? CLS_NARROW1 : CLS_NARROWK)); }
}

}  // namespace pcob200
