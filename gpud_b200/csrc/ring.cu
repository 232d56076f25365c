// ring.cu — device-resident counter-sample ring and the fused windowed aggregates (kernels K1-K4 of SURVEY.md §2.2).
//
// Data layout in HBM (per GPU):
//   ring      f64 [F][CAP]      field-major: one field's samples are contiguous in time, so a window of W samples
//                               is one 8·W-byte contiguous run -> 128-bit coalesced loads, one warp per window.
//   results   f64 [F][n_windows] x {min,max,mean,ema,p99}, u32 [F][n_windows] n_over
//   part      f64 [n_windows][F] per-window EMA partial sums (transposed so the carry scan reads coalesced)
//
// Roofline: every kernel here is HBM-bound; the fused reduce reads each sample exactly once (8 B / sample,
// SURVEY.md §8d) and writes 44 B per window.  No tensor cores: there is no contraction on this path.
//
// Reference seams replaced (the reference has no windowed aggregation at all, SURVEY.md §0):
//   sample sink     pkg/metrics/scraper/prometheus.go:28-81 + pkg/metrics/store/sqlite.go:108-164
//   threshold `>`   components/accelerator/nvidia/temperature/component.go:228,240
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include <algorithm>

#include "internal.h"
#include "ring_drain.h"

namespace {

constexpr int kMaxWindow = 1024;      // 32 lanes x 32 elements held in registers
#ifndef GPUD_WARPS_PER_BLOCK
#define GPUD_WARPS_PER_BLOCK 8
#endif
constexpr int kWarpsPerBlock = GPUD_WARPS_PER_BLOCK;
constexpr int kCandMax = 64;
constexpr unsigned kFull = 0xffffffffu;
constexpr size_t kStageBytes = 32u << 20;   // pinned staging buffers (x2)

struct WinParams {
  const double* ring;
  int64_t cap, start, count;
  int W, F, nw;
  int q_num, q_den;
  const double* thr;   // [F]
  const double* pw;    // [127]: (1-alpha)^e for e = -63..63
  const double* pwl;   // [32]: (1-alpha)^(W - 32 l - 32) (in-place kernel)
  double q64;          // (1-alpha)^64
  double alpha;
  double* out_min;
  double* out_max;
  double* out_mean;
  double* out_p99;
  uint32_t* out_nover;
  double* part;        // [F][nw] per-window EMA partial sums
  int do_select;       // 0: skip the order statistic (range reduce uses the radix select instead)
  int k_full;          // k-th largest rank of a full window (m == W), precomputed on the host
  double inv_w;        // 1.0 / W
  int n_list;          // > 0: process only windows w_list[0..n_list) of every field (generic instantiation)
  int w_list[2];
  int w_skip[2];       // windows the specialised launch leaves to the generic one (-1 = none)
  // RANGE instantiations only (whole-range order statistic, select.cu): the pass classifies every sample against the field's
  // pivot pair lo <= hi and parks the keys strictly between them in the field's list
  const double* piv;           // [F][2]: lo, hi
  uint4* w_cls;                // [F][nw]: per window {keys above hi, keys == hi, keys == lo, keys strictly inside}
  unsigned long long* lists;   // [F][list_cap] totalOrder keys strictly inside (lo, hi), any order
  unsigned* fill;              // [F] list fill counters (may run past list_cap: overflow is detected by the reader)
  unsigned list_cap;
};

// ---------------------------------------------------------------------------------------------
// K1: append.  src [n][F] row-major (one row per poll) -> ring [F][CAP] at columns (head + i) % CAP.
// 32x32 tile transpose through shared memory: reads coalesced along F, writes coalesced along time.
// ---------------------------------------------------------------------------------------------
// T = the caller's sample type: double, or a raw NVML / DCGM counter type widened here exactly like Go's float64(v)
// (round-to-nearest-even for 64-bit integers above 2^53).
// The same kernel keeps the SAMPLE RING: every column whose index is smp_half modulo 2^smp_shift is also stored at
// sample[f][col >> smp_shift] - a systematic sample of at most 8192 keys per field that is always current, so the whole-range order
// statistic (select.cu) gets its pivots from 64 KB of contiguous memory per field instead of 8192 scattered 32-byte sectors.
template <typename T>
__global__ void __launch_bounds__(256) k_ring_append(const T* __restrict__ src, double* __restrict__ ring, int64_t n, int F,
                                                      int64_t cap, int64_t head, double* __restrict__ sample, int smp_shift, int64_t smp_half, int64_t smp_slots) {
  __shared__ double tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  const int64_t tiles_f = (F + 31) / 32;
  const int64_t tiles_n = (n + 31) / 32;
  for (int64_t t = blockIdx.x; t < tiles_f * tiles_n; t += gridDim.x) {
    const int64_t tn = t / tiles_f, tf = t - tn * tiles_f;
    const int64_t r0 = tn * 32, f0 = tf * 32;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t r = r0 + ty + 8 * k, f = f0 + tx;
      if (r < n && f < F) tile[ty + 8 * k][tx] = (double)__ldcs(src + r * F + f);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t f = f0 + ty + 8 * k, r = r0 + tx;
      if (r < n && f < F) {
        int64_t col = head + r;
        col = col >= cap ? col % cap : col;
        const double val = tile[tx][ty + 8 * k];
        ring[f * cap + col] = val;
        if ((col & ((1ll << smp_shift) - 1)) == smp_half) sample[f * smp_slots + (col >> smp_shift)] = val;
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// warp primitives.  Keys are kept as (hi, lo) 32-bit halves so every compare / select is one 32-bit instruction.
// ---------------------------------------------------------------------------------------------
struct K64 { unsigned hi, lo; };
// acc += (a > b) for IEEE doubles: DSETP and one predicated integer add
__device__ __forceinline__ void count_gt_f64(unsigned& acc, double a, double b) {
  asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %1, %2;\n\t@p add.u32 %0, %0, 1;\n\t}" : "+r"(acc) : "d"(a), "d"(b));   // DSETP + predicated add
}
// RANGE pass: above += (x > hi); otherwise, when x >= lo, set `bit` in mask.  NaN fails both compares (the caller guards +NaN).
__device__ __forceinline__ void classify_f64(unsigned& above, unsigned& mask, double x, double lo, double hi, unsigned bit) {
  asm("{\n\t.reg .pred p, q;\n\tsetp.gt.f64 p, %2, %4;\n\t@p add.u32 %0, %0, 1;\n\tsetp.ge.and.f64 q, %2, %3, !p;\n\t@q or.b32 %1, %1, %5;\n\t}"
      : "+r"(above), "+r"(mask) : "d"(x), "d"(lo), "d"(hi), "r"(bit));
}
// acc -= (o > v) for unsigned words through the borrow flag (sub.cc / subc pair): two integer instructions, no predicate
__device__ __forceinline__ void count_gt_u32_neg(unsigned& acc, unsigned o, unsigned v) {
  unsigned t;
  asm("sub.cc.u32 %1, %2, %3;\n\tsubc.u32 %0, %0, 0;" : "+r"(acc), "=r"(t) : "r"(v), "r"(o));
}
__device__ __forceinline__ bool k_gt(unsigned ah, unsigned al, unsigned bh, unsigned bl) { return ah > bh || (ah == bh && al > bl); }

__device__ __forceinline__ K64 warp_max_k64(unsigned hi, unsigned lo) {
  // two REDUX passes instead of ten shuffles: max of the high words, then max of the low words among the winners
  K64 r;
  r.hi = __reduce_max_sync(kFull, hi);
  r.lo = __reduce_max_sync(kFull, hi == r.hi ? lo : 0u);
  return r;
}
__device__ __forceinline__ K64 warp_min_k64(unsigned hi, unsigned lo) {
  K64 r;
  r.hi = __reduce_min_sync(kFull, hi);
  r.lo = __reduce_min_sync(kFull, hi == r.hi ? lo : 0xffffffffu);
  return r;
}
__device__ __forceinline__ double k64_to_f64(K64 k) {
  const unsigned m = (k.hi & 0x80000000u) ? 0x80000000u : 0xffffffffu;   // inverse of the totalOrder key map
  const unsigned lo = (k.hi & 0x80000000u) ? k.lo : ~k.lo;
  return __hiloint2double((int)(k.hi ^ m), (int)lo);
}
// bitonic sort across the 32 lanes, descending, on (hi, lo)
__device__ __forceinline__ void warp_sort_desc_k64(unsigned& hi, unsigned& lo, int lane) {
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const unsigned oh = __shfl_xor_sync(kFull, hi, j), ol = __shfl_xor_sync(kFull, lo, j);
      const bool keep_max = (((lane & k) == 0) == ((lane & j) == 0));
      const bool take = keep_max == k_gt(oh, ol, hi, lo);
      hi = take ? oh : hi;
      lo = take ? ol : lo;
    }
  }
}

// rank -= (o > c) for 64-bit keys given as (hi, lo) halves: one borrow chain, no predicates
__device__ __forceinline__ void count_gt_k64_neg(unsigned& acc, unsigned oh, unsigned ol, unsigned ch, unsigned cl) {
  unsigned t;
  asm("sub.cc.u32 %1, %2, %3;\n\tsubc.cc.u32 %1, %4, %5;\n\tsubc.u32 %0, %0, 0;" : "+r"(acc), "=r"(t) : "r"(cl), "r"(ol), "r"(ch), "r"(oh));
}
// The window is parked in shared memory as RAW doubles (pass 1 spends no ALU on keys).  totalOrder key of raw (h, l):
//   key_hi = h ^ ((h >> 31) | 0x80000000)   (bijection on the high word),   key_lo = l ^ ~sign-extension of key_hi bit 31.
__device__ __forceinline__ unsigned key_hi_of(unsigned raw_hi) { return raw_hi ^ ((unsigned)((int)raw_hi >> 31) | 0x80000000u); }
__device__ __forceinline__ unsigned raw_hi_of(unsigned key_hi) { return key_hi ^ ((key_hi & 0x80000000u) ? 0x80000000u : 0xffffffffu); }
__device__ __forceinline__ unsigned true_lo(unsigned key_hi, unsigned raw_lo) { return raw_lo ^ ~(unsigned)((int)key_hi >> 31); }
__device__ __forceinline__ unsigned long long true_key(unsigned long long raw) {
  const unsigned hi = key_hi_of((unsigned)(raw >> 32));
  return ((unsigned long long)hi << 32) | true_lo(hi, (unsigned)raw);
}
constexpr unsigned long long kPadStored = 0xffffffffffffffffull;   // raw form of the smallest key 0 (-NaN, all ones)

// Candidates sit in shared memory s[0..cnt), cnt <= 32, as RAW doubles.  Returns the k-th largest (k <= cnt) and the maximum.
// rank_i = #{j : c_j > c_i};  the k-th largest is the smallest candidate whose rank is < k.
__device__ __forceinline__ K64 select_from_candidates(uint2* s, int cnt, int k, int lane, K64* mx) {
  const bool mine = lane < cnt;
  uint2 c = mine ? s[lane] : make_uint2(0xffffffffu, 0xffffffffu);   // .x = lo, .y = hi (raw)
  c.y = key_hi_of(c.y);
  c.x = true_lo(c.y, c.x);
  if (mine) s[lane] = c;                                     // the broadcast reads below see true keys
  __syncwarp();
  unsigned nr0 = 0, nr1 = 0, nr2 = 0, nr3 = 0;               // four independent borrow chains
#pragma unroll 1
  for (int j = 0; j < cnt; j += 4) {                         // the list is zero-padded to a multiple of 4; a zero never outranks
    const uint4 o01 = *reinterpret_cast<const uint4*>(s + j), o23 = *reinterpret_cast<const uint4*>(s + j + 2);   // broadcast LDS.128
    count_gt_k64_neg(nr0, o01.y, o01.x, c.y, c.x);
    count_gt_k64_neg(nr1, o01.w, o01.z, c.y, c.x);
    count_gt_k64_neg(nr2, o23.y, o23.x, c.y, c.x);
    count_gt_k64_neg(nr3, o23.w, o23.z, c.y, c.x);
  }
  const unsigned neg_rank = (nr0 + nr1) + (nr2 + nr3);
  *mx = warp_max_k64(mine ? c.y : 0u, mine ? c.x : 0u);
  const bool in = mine && (int)(0u - neg_rank) < k;
  return warp_min_k64(in ? c.y : 0xffffffffu, in ? c.x : 0xffffffffu);
}

// ---------------------------------------------------------------------------------------------
// K2+K4 (+ the per-window part of K3): one warp per (field, window).
//   lane l, register pair j holds chronological elements t = 64 j + 2 l + {0,1} of the window (128-bit coalesced loads).
//   Pass 1 streams the loaded values once: sum, EMA Horner, threshold count, min/max of the key high words, and parks the
//   totalOrder keys in shared memory, row = lane (272-byte rows: conflict-free 128-bit stores and 64-bit row reads).
//   Everything after that is warp-cooperative over ROWS: only the ~k lanes whose maximum can reach the order statistic
//   are revisited, 32 keys per LDS, instead of every lane scanning its 32 registers.
// ALIGNED: the window is one 16-byte aligned run (no wrap) -> 128-bit loads; otherwise 64-bit loads with wrap.
// JF >= 0: compile-time number of fully valid register pairs (= W >> 6); such an instantiation only sees full windows
// (m == W), so the pair loop is straight-line code.  JF = -1: everything is decided at run time (any W, partial windows).
// ---------------------------------------------------------------------------------------------
constexpr int kRowU64 = 34;                                   // 32 keys + 2 pad -> 272-byte rows
constexpr int kKeyBytes = 32 * kRowU64 * 8;                   // key rows
constexpr int kPadRowOff = kKeyBytes;                         // 256 B of kPadStored: the row the padded tail of the row list points at
constexpr int kCandOff = kPadRowOff + 256;                    // candidates (+4 pad slots)
constexpr int kRowListOff = kCandOff + (kCandMax + 4) * 8;    // byte offsets of the flagged rows, 32 + 4 pad entries
constexpr int kCntOff = kRowListOff + 36 * 4;
constexpr int kWarpSmemBytes = kCntOff + 16;
constexpr int kBlockSmemBytes = kWarpsPerBlock * kWarpSmemBytes;

__device__ __forceinline__ int elem_index(int row, int col) { return 64 * (col >> 1) + 2 * row + (col & 1); }   // chronological t

// Append the entries of the flagged rows that pass the bound to cand[] (any order, RAW form).  HI_ONLY: keys whose high
// word is >= Lh (the fast path's bound is (Lh, 0), inclusive), tested on the raw word: key_hi >= Lh  <=>
// (int)(raw ^ X) >= (int)(Lh ^ 0x80000000) with X = 0 for a non-negative bound and 0x7fffffff for a negative one.
// Otherwise: true keys > (Lh, Ll).
// The flagged rows' byte offsets are packed into a list first (padded to a multiple of four with the pad row); then one LDS
// per row gives every lane one key of that row and the few lanes that hold a hit claim a slot with a predicated
// shared-memory atomic - straight-line code, four rows in flight per trip.
// Returns the number of hits (may exceed kCandMax; only the first kCandMax are stored).
// INPLACE: the rows are not stored anywhere - "row r, entry i" is element 64 (i >> 1) + 2 ((r + (i >> 1)) & 31) + (i & 1) of the
// linear window buffer (k_window_reduce_inplace); the row list then holds 16 r and the pad row is reached through a flag bit.
template <bool HI_ONLY, int ROWW = kRowU64, bool INPLACE = false>
__device__ __forceinline__ int gather_rows(unsigned char* wbase, unsigned rows, unsigned Lh, unsigned Ll, int lane, unsigned lt_mask) {
  constexpr int kPadOff = 32 * ROWW * 8, kCndOff = kPadOff + 256, kLstOff = kCndOff + (kCandMax + 4) * 8;   // the scratch follows the rows
  const int n_rows = __popc(rows);
  unsigned* row_off = reinterpret_cast<unsigned*>(wbase + kLstOff);
  if ((rows >> lane) & 1u) row_off[__popc(rows & lt_mask)] = INPLACE ? (unsigned)lane : (unsigned)lane * (ROWW * 8);
  if (lane < 4) row_off[n_rows + lane] = INPLACE ? 0x80000000u : kPadOff;
  __syncwarp();
  const unsigned col = (unsigned)__cvta_generic_to_shared(wbase) + (INPLACE ? (unsigned)((lane >> 1) * 512 + (lane & 1) * 8) : (unsigned)(lane * 8));
  uint2* cand = reinterpret_cast<uint2*>(wbase + kCndOff);
  const unsigned long long Lp = ((unsigned long long)Lh << 32) | Ll;
  const unsigned X = (Lh & 0x80000000u) ? 0u : 0x7fffffffu;
  const int Y = (int)(Lh ^ 0x80000000u);
  int cnt = 0;
  // Hits are compacted with warp ballots (slot = hits so far + hits in lower lanes): no shared-memory atomics, and a class of
  // equal keys that would overflow the candidate list ends the walk after the trip that passes 32 (the caller falls back).
#pragma unroll 1
  for (int i = 0; i < n_rows && cnt <= 32; i += 4) {
    uint4 o4 = *reinterpret_cast<const uint4*>(row_off + i);                         // broadcast
    if (INPLACE) {
      auto at = [&](unsigned r) { return (r & 0x80000000u) ? (unsigned)(kPadOff + lane * 8) - (unsigned)((lane >> 1) * 512 + (lane & 1) * 8) : 16u * ((r + (unsigned)(lane >> 1)) & 31u); };
      o4 = make_uint4(at(o4.x), at(o4.y), at(o4.z), at(o4.w));
    }
    unsigned lo[4], hi[4];
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo[0]), "=r"(hi[0]) : "r"(col + o4.x));
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo[1]), "=r"(hi[1]) : "r"(col + o4.y));
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo[2]), "=r"(hi[2]) : "r"(col + o4.z));
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo[3]), "=r"(hi[3]) : "r"(col + o4.w));
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      bool hit;
      if (HI_ONLY) hit = (int)(hi[q] ^ X) >= Y;
      else hit = true_key(((unsigned long long)hi[q] << 32) | lo[q]) > Lp;
      const unsigned b = __ballot_sync(kFull, hit);
      const int slot = cnt + __popc(b & lt_mask);
      if (hit && slot < kCandMax) cand[slot] = make_uint2(lo[q], hi[q]);
      cnt += __popc(b);
    }
  }
  __syncwarp();
  // zero-pad to a multiple of 4 so the rank loop can run unrolled without a tail
  if (lane < 4 && cnt <= kCandMax) cand[cnt + lane] = make_uint2(0u, 0u);
  __syncwarp();
  return cnt;
}

// k-th largest (1-based, k <= 32) of one 32-bit value per lane, counting multiplicity, through shared memory:
// rank_i = #{j : v_j > v_i};  the answer is the smallest value whose rank is < k.  One STS, eight broadcast LDS.128 and
// 32 independent compares per lane: the same instruction count as a 32-bit bitonic sort without its 15-deep shuffle chain.
__device__ __forceinline__ unsigned warp_kth_largest_smem(unsigned v, int k, unsigned* s32, int lane) {
  s32[lane] = v;
  __syncwarp();
  unsigned n0 = 0, n1 = 0, n2 = 0, n3 = 0;    // minus the number of lanes holding a larger value, four independent chains
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const uint4 o = reinterpret_cast<const uint4*>(s32)[q];
    count_gt_u32_neg(n0, o.x, v); count_gt_u32_neg(n1, o.y, v); count_gt_u32_neg(n2, o.z, v); count_gt_u32_neg(n3, o.w, v);
  }
  const unsigned neg_rank = (n0 + n1) + (n2 + n3);
  __syncwarp();
  return __reduce_min_sync(kFull, (int)(0u - neg_rank) < k ? v : 0xffffffffu);
}

struct WinUnit { int f, w, m; int64_t p0; };
// ---- cp.async.bulk landing (TMA instantiations): one bulk copy per window into the warp's stage buffer, completion on an mbarrier ----
__device__ __forceinline__ void mbar_init(unsigned a, int cnt) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(cnt)); }
__device__ __forceinline__ void mbar_expect(unsigned a, int bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory"); }
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, int bytes, unsigned mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned a, int parity) {
  unsigned ok = 0;
  while (!ok)
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(a), "r"(parity) : "memory");
}
constexpr int kStageBytesTma = 8192;                       // one window of <= 1024 doubles
constexpr int kTmaWarps = 13;                              // 13 x (row area + stage) = 226.7 KB: one CTA per SM
// streaming 128-bit load: read-only path, no L1 allocation, 256-byte L2 sector promotion (measured best of the hints on B200)
__device__ __forceinline__ double2 ld_stream(const double2* p) {
  double2 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
  return r;
}
#ifndef GPUD_PREFETCH_PAIRS
#define GPUD_PREFETCH_PAIRS 16   /* measured: 8 pairs + 3 CTAs/SM = 63 % of roofline, 16 pairs + 2 CTAs/SM = 82 % */
#endif
constexpr int kPrefetchPairs = GPUD_PREFETCH_PAIRS;      // register pairs of the NEXT window loaded under the current post-processing
constexpr int kHotCtasPerSM = kPrefetchPairs < 16 ? 3 : 2;  // 8 pairs in flight fit 80 registers (3 CTAs/SM); all 16 need 128 (2 CTAs/SM)

// TMA: the window lands in a per-warp stage buffer through one cp.async.bulk (UBLKCP) instead of 16 LDG.128 per lane into registers;
// pass 1 reads it with conflict-free LDS.128 and the copy of the next window is issued as soon as pass 1 is done with the buffer.
// Only for the hot shape (ALIGNED, JF >= 0); 13 warps per SM in one CTA (the stage buffers take the room of the second CTA's rows).
template <bool ALIGNED, int JF, bool RANGE, bool TMA = false>
__global__ void __launch_bounds__((TMA ? kTmaWarps : kWarpsPerBlock) * 32, TMA ? 1 : ((ALIGNED && JF >= 0) ? kHotCtasPerSM : 2)) k_window_reduce(const WinParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int WPB = TMA ? kTmaWarps : kWarpsPerBlock;
  constexpr int kPerWarp = kWarpSmemBytes + (TMA ? kStageBytesTma : 0);
  __shared__ __align__(8) unsigned long long s_bars[TMA ? kTmaWarps : 1];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  unsigned char* wbase = smem_raw + (size_t)warp * kPerWarp + (TMA ? kStageBytesTma : 0);     // stage buffer first (128-byte aligned), rows after it
  const unsigned stage_a = (unsigned)__cvta_generic_to_shared(smem_raw + (size_t)warp * kPerWarp);
  const double2* stage2 = reinterpret_cast<const double2*>(smem_raw + (size_t)warp * kPerWarp) + lane;
  const unsigned bar_a = (unsigned)__cvta_generic_to_shared(s_bars + (TMA ? warp : 0));
  int tma_parity = 0;
  if (TMA) {
    if (lane == 0) mbar_init(bar_a, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
  }
  unsigned long long* sk = reinterpret_cast<unsigned long long*>(wbase);                        // [32][kRowU64] key rows
  uint2* cand = reinterpret_cast<uint2*>(wbase + kCandOff);                                     // [kCandMax + 4]
  unsigned* s32 = reinterpret_cast<unsigned*>(cand);                                            // 128 B scratch, reused before the gather
  reinterpret_cast<unsigned long long*>(wbase + kPadRowOff)[lane] = kPadStored;                 // the pad row, written once
  uint4* my_row4 = reinterpret_cast<uint4*>(sk + lane * kRowU64);   // one uint4 = two keys {lo0, hi0, lo1, hi1}
  const int64_t n_units = p.n_list > 0 ? (int64_t)p.F * p.n_list : (int64_t)p.F * p.nw;
  const unsigned lt_mask = (1u << lane) - 1u;

  // (field, slot) advance incrementally: one division per kernel instead of one per window
  const int per_f = p.n_list > 0 ? p.n_list : p.nw;
  const int64_t stride = (int64_t)gridDim.x * WPB;
  const int df = (int)(stride / per_f), ds = (int)(stride - (int64_t)df * per_f);
  int64_t u = (int64_t)blockIdx.x * WPB + warp;
  int uf = (int)(u / per_f), uslot = (int)(u - (int64_t)uf * per_f);

  constexpr int PF = (ALIGNED && JF >= 0) ? kPrefetchPairs : 16;
  double2 v[16];                 // the window in flight: loaded for the NEXT unit while the current one is post-processed
  double thr_next = 0.0, lo_next = 0.0, hi_next = 0.0;
  // fetch the next non-skipped unit of this warp (if any) and issue all of its loads.  Measured alternatives, both slower on
  // B200: choosing the next unit BEFORE pass 1 (its address/threshold registers live through pass 1: 0.79 ms vs 0.70 ms) and
  // issuing each pair's load inside pass 1 right after the pair is consumed (0.72 ms).
  auto fetch = [&](WinUnit& q) -> bool {
    for (;;) {
      if (u >= n_units) return false;
      q.f = uf;
      q.w = p.n_list > 0 ? p.w_list[uslot] : uslot;
      u += stride; uf += df; uslot += ds;
      if (uslot >= per_f) { uslot -= per_f; ++uf; }
      if (p.n_list > 0 || (q.w != p.w_skip[0] && q.w != p.w_skip[1])) break;
    }
    const int64_t c0 = (int64_t)q.w * p.W;
    q.m = JF >= 0 ? p.W : (int)min((int64_t)p.W, p.count - c0);
    q.p0 = p.start + c0;
    if (q.p0 >= p.cap) q.p0 -= p.cap;
    const double* __restrict__ base = p.ring + (int64_t)q.f * p.cap;
    thr_next = __ldg(p.thr + q.f);
    if (RANGE) { lo_next = __ldg(p.piv + 2 * q.f); hi_next = __ldg(p.piv + 2 * q.f + 1); }
    if (TMA) {
      if (lane == 0) {                                               // one 8 W-byte bulk copy; the mbarrier flips when all of it has landed
        mbar_expect(bar_a, q.m * 8);
        bulk_g2s(stage_a, base + q.p0, q.m * 8, bar_a);
      }
    } else if (ALIGNED) {
      const double2* __restrict__ b2 = reinterpret_cast<const double2*>(base + q.p0) + lane;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        if (j >= PF) continue;                                     // the rest is loaded by fetch_rest() at the top of the next trip
        if (JF >= 0 && j < JF) { v[j] = ld_stream(b2 + 32 * j); continue; }
        v[j] = make_double2(0.0, 0.0);
        if (64 * j + 2 * lane < q.m) v[j] = ld_stream(b2 + 32 * j);   // element t0+1 == m is masked in pass 1 (the ring has slack)
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int t0 = 64 * j + 2 * lane;
        v[j] = make_double2(0.0, 0.0);
        if (t0 < q.m) { int64_t a = q.p0 + t0; if (a >= p.cap) a -= p.cap; v[j].x = __ldcs(base + a); }
        if (t0 + 1 < q.m) { int64_t a = q.p0 + t0 + 1; if (a >= p.cap) a -= p.cap; v[j].y = __ldcs(base + a); }
      }
    }
    return true;
  };

  auto fetch_rest = [&](const WinUnit& q) {
    if (PF >= 16 || TMA) return;
    const double2* __restrict__ b2 = reinterpret_cast<const double2*>(p.ring + (int64_t)q.f * p.cap + q.p0) + lane;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      if (j < PF) continue;
      if (JF >= 0 && j < JF) { v[j] = ld_stream(b2 + 32 * j); continue; }
      v[j] = make_double2(0.0, 0.0);
      if (64 * j + 2 * lane < q.m) v[j] = ld_stream(b2 + 32 * j);
    }
  };

  WinUnit cur, nxt;
  bool have = fetch(cur);
  while (have) {
    fetch_rest(cur);
    if (TMA) { mbar_wait(bar_a, tma_parity); tma_parity ^= 1; }      // the window has landed in the stage buffer
    const int f = cur.f, w = cur.w, m = cur.m;
    const int J = (m + 63) >> 6;                     // register pairs that hold at least one valid element
    const int Jfull = JF >= 0 ? JF : (m >> 6);       // register pairs in which every lane's two elements are valid
    const double thr = thr_next;
    const double piv_lo = lo_next, piv_hi = hi_next;
    unsigned abv = 0, inmask = 0;                    // RANGE: keys above the upper pivot; row entries inside [lo, hi] (as doubles)

    // ---- pass 1: consume the loaded registers once ----
    double sum0 = 0.0, sum1 = 0.0, es0 = 0.0, es1 = 0.0;
    unsigned nov = 0;
    // lane extremes of the RAW high words, three running values and no per-element transform: sign-magnitude order means
    //   the largest key is smax(h) when any element is non-negative (smax >= 0), else umin(h);
    //   the smallest key is umax(h) when any element is negative (umax >= 2^31), else umin(h).
    int a_smax = (int)0x80000000;
    unsigned b_umin = 0xffffffffu, c_umax = 0u;
    unsigned lor = 0u;                               // OR of the raw low words: zero = an integer-valued gauge, the high words are the whole key
    double2* my_row2 = reinterpret_cast<double2*>(my_row4);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      if (JF >= 0 ? (j < JF) : (j < Jfull)) {  // whole register pair valid (compile-time when JF >= 0, else warp-uniform)
        if (TMA) v[j] = stage2[32 * j];          // LDS.128, lane-consecutive: conflict-free
        const double x0 = v[j].x, x1 = v[j].y;
        const int h0 = __double2hiint(x0), h1 = __double2hiint(x1);
        sum0 += x0; sum1 += x1;
        es0 = fma(es0, p.q64, x0); es1 = fma(es1, p.q64, x1);
        count_gt_f64(nov, x0, thr);
        count_gt_f64(nov, x1, thr);
        if (RANGE) {
          classify_f64(abv, inmask, x0, piv_lo, piv_hi, 1u << (2 * j));
          classify_f64(abv, inmask, x1, piv_lo, piv_hi, 2u << (2 * j));
        }
        a_smax = max(a_smax, max(h0, h1));
        b_umin = min(b_umin, min((unsigned)h0, (unsigned)h1));
        c_umax = max(c_umax, max((unsigned)h0, (unsigned)h1));
        lor |= (unsigned)__double2loint(x0) | (unsigned)__double2loint(x1);
        my_row2[j] = v[j];                     // STS.128 of the loaded registers, conflict-free (272-byte row stride)
      } else if (JF >= 0 ? (j == JF) : (j < J)) {   // the one partially valid pair
        const int t0 = 64 * j + 2 * lane;
        const bool q0 = t0 < m, q1 = t0 + 1 < m;
        if (TMA) v[j] = stage2[32 * j];          // bytes past the window are stale: masked by q0 / q1
        const double x0 = q0 ? v[j].x : 0.0, x1 = q1 ? v[j].y : 0.0;
        const unsigned h0 = q0 ? (unsigned)__double2hiint(x0) : 0xffffffffu, h1 = q1 ? (unsigned)__double2hiint(x1) : 0xffffffffu;   // padding = kPadStored
        sum0 += x0; sum1 += x1;
        es0 = fma(es0, p.q64, x0); es1 = fma(es1, p.q64, x1);
        if (q0 && x0 > thr) ++nov;
        if (q1 && x1 > thr) ++nov;
        if (RANGE) {
          if (q0) { if (x0 > piv_hi) ++abv; else if (x0 >= piv_lo) inmask |= 1u << (2 * j); }
          if (q1) { if (x1 > piv_hi) ++abv; else if (x1 >= piv_lo) inmask |= 2u << (2 * j); }
        }
        a_smax = max(a_smax, max((int)h0, (int)h1));                       // all-ones is -1: neutral unless every element is negative, and then unused
        b_umin = min(b_umin, min(h0, h1));
        c_umax = max(c_umax, max(q0 ? h0 : 0u, q1 ? h1 : 0u));
        lor |= (q0 ? (unsigned)__double2loint(x0) : 0u) | (q1 ? (unsigned)__double2loint(x1) : 0u);
        my_row4[j] = make_uint4(q0 ? (unsigned)__double2loint(x0) : 0xffffffffu, h0, q1 ? (unsigned)__double2loint(x1) : 0xffffffffu, h1);
      } else {
        my_row4[j] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);     // padding: the smallest key (kPadStored)
      }
    }
    const unsigned rmh = a_smax >= 0 ? (unsigned)a_smax : b_umin;          // raw high word of this lane's largest key
    const unsigned mh = key_hi_of(rmh);
    const bool lane_empty = c_umax == 0u && b_umin == 0xffffffffu;         // no valid element (windows shorter than 64 samples)
    const unsigned nh = lane_empty ? 0xffffffffu : key_hi_of((c_umax & 0x80000000u) ? c_umax : b_umin);
    __syncwarp();

    // ---- the registers are free again: put the next window's loads in flight under the post-processing below ----
    have = fetch(nxt);

    // ---- sums (the two shuffle trees are interleaved) ----
    const int eb = m - 1 - 64 * (J - 1) - 2 * lane;          // exponent of this lane's h=0 element in pair J-1, in [-62, 63]
    double ep = es0 * __ldg(p.pw + (eb + 63)) + es1 * __ldg(p.pw + (eb - 1 + 63));   // EMA partial, weights alpha (1-alpha)^(m-1-t)
    double sum = sum0 + sum1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sum += __shfl_xor_sync(kFull, sum, o);
      ep += __shfl_xor_sync(kFull, ep, o);
    }
    ep *= p.alpha;
    // the positional shortcut's pretest rides on this reduction (no extra warp operation on the common path): bits 16.. count the lanes
    // whose own 32 samples span more than 8 high words or hold a negative one (nov itself is at most 1024)
    const unsigned nov_flags = __reduce_add_sync(kFull, nov + ((mh - nh > 8u || (c_umax & 0x80000000u)) ? 0x10000u : 0u));
    nov = nov_flags & 0xffffu;
    const bool tied_nonneg = (nov_flags >> 16) == 0u;

    // ---- exact minimum: global min of the high words, then the low words of the rows that hold it ----
    // Every raw low word zero (integer readings below 2^21: degrees, %, MHz, MiB, mW): the high words order the window by
    // themselves and a key's low word follows from its sign - no row is revisited for min / max, ties cost nothing.
    const bool lo_zero = __reduce_or_sync(kFull, lor) == 0u;
    K64 wmin;
    wmin.hi = __reduce_min_sync(kFull, nh);
    // ---- positional shortcut: a window that is already in ascending order where it matters ----
    // A monotone counter (NVLink / PCIe replays, ECC, energy: float64 of a u64 that only grows) is the one stream whose high words tie
    // AND whose low words matter: every window went down the 64-bit path below (lane maxima, 64-bit warp sort, two gathers) - 1.24 ms
    // for a ring of such fields against 0.69 for gauges.  But its order statistics are positions: min = first sample, max = last,
    // k-th largest = sample m - k.  That holds for ANY window whose samples before t = m - k lie in [first, T] and whose last k lie in
    // [T, last] (T = sample m - k), all non-negative (so that numeric order is totalOrder and no -0 hides in a tie; NaN fails every
    // compare): checked on the parked rows, 32 LDS.64 and 64 compares per lane.  Tried only where every lane's own samples span at most
    // 8 high words (a flag that rides on the n_over reduction; a gauge with noise spans thousands and pays nothing else).  Measured on 512 x
    // 1 Mi: counters 1.24 -> 0.85 ms, survey mix 0.746 -> 0.718 (91 % of the copy peak), white noise 0.689 -> 0.696.  Variants that lost: the
    // check behind a per-lane pretest read from the rows for EVERY window (gauges +9 %), the check out of line in the 64-bit path only
    // (counters 1.12: the minimum scan and the failed gather stay), a lane pretest between the span test and the loop (no change).
    bool positional = false;
    if (!RANGE && !lo_zero && tied_nonneg && m == p.W && m > 960 && p.k_full >= 1 && p.k_full <= 32) {
      const int tk = m - p.k_full;
      auto at = [&](int t) { return __longlong_as_double((long long)sk[((t & 63) >> 1) * kRowU64 + 2 * (t >> 6) + (t & 1)]); };
      const double e0 = at(0), tv = at(tk), el = at(m - 1);
      bool ok = true;
      const int i_low = tk >= 960 ? 30 : 0;          // the usual case (k <= m - 960): entries 0..29 (t < 960) all lie before sample m - k
#pragma unroll 2
      for (int i = 0; i < i_low; ++i) {
        const double x = __longlong_as_double((long long)sk[lane * kRowU64 + i]);
        ok = ok && e0 <= x && x <= tv;
      }
#pragma unroll 1
      for (int i = i_low; i < 32; ++i) {
        const int t = elem_index(lane, i);
        const double x = __longlong_as_double((long long)sk[lane * kRowU64 + i]);
        const bool in_lo = e0 <= x && x <= tv, in_hi = tv <= x && x <= el;
        if (t < m) ok = ok && (t < tk ? in_lo : in_hi);
      }
      positional = __all_sync(kFull, ok);
    }
    if (positional) {
      const unsigned long long r0 = sk[0];                          // sample 0: row 0, entry 0
      wmin.hi = key_hi_of((unsigned)(r0 >> 32));
      wmin.lo = true_lo(wmin.hi, (unsigned)r0);
    } else if (lo_zero) {
      wmin.lo = true_lo(wmin.hi, 0u);
    } else {
      unsigned rows = __ballot_sync(kFull, nh == wmin.hi);
      unsigned nl = 0xffffffffu;
      const unsigned raw_min_hi = raw_hi_of(wmin.hi);
      if (__popc(rows) > 6) {
        // tie-heavy window (integer readings, flat gauges): most rows hold the minimum high word, so every lane scans its own
        // row instead of the warp visiting the rows one by one
        rows = 0u;
#pragma unroll 4
        for (int i = 0; i < 32; ++i) {
          const unsigned long long kv = sk[lane * kRowU64 + i];
          if ((unsigned)(kv >> 32) == raw_min_hi && elem_index(lane, i) < m) nl = min(nl, true_lo(wmin.hi, (unsigned)kv));
        }
      }
      while (rows) {
        const int row = __ffs(rows) - 1;
        rows &= rows - 1;
        const unsigned long long kv = sk[row * kRowU64 + lane];
        if ((unsigned)(kv >> 32) == raw_min_hi && elem_index(row, lane) < m) nl = min(nl, true_lo(wmin.hi, (unsigned)kv));   // the index test screens padding
      }
      wmin.lo = __reduce_min_sync(kFull, nl);
    }

    K64 ans, wmax;
    ans.hi = ans.lo = 0u;
    uint4 cls = make_uint4(0u, 0u, 0u, 0u);
    if constexpr (!RANGE) {
      // ---- exact order statistic: k-th largest, k = m - ceil(m q) + 1; the maximum falls out of the same candidate set ----
      int k = p.k_full;
      if (JF < 0 && m != p.W) {
        long long r = ((long long)m * p.q_num + p.q_den - 1) / p.q_den;
        r = r < 1 ? 1 : (r > m ? m : r);
        k = m - (int)r + 1;
      }
      bool done = false;
      if (positional) {
        const int tk = m - k, tl = m - 1;
        const unsigned long long ra = sk[((tk & 63) >> 1) * kRowU64 + 2 * (tk >> 6) + (tk & 1)], rl = sk[((tl & 63) >> 1) * kRowU64 + 2 * (tl >> 6) + (tl & 1)];
        ans.hi = key_hi_of((unsigned)(ra >> 32)); ans.lo = true_lo(ans.hi, (unsigned)ra);
        wmax.hi = key_hi_of((unsigned)(rl >> 32)); wmax.lo = true_lo(wmax.hi, (unsigned)rl);
        done = true;
      }
      if (!done && k <= 32) {
        // Lower bound L' = (k-th largest lane maximum of the HIGH words, 0): at least k keys are >= L', so the answer is too.
        // Only rows whose maximum reaches L' can hold keys above it.
        const unsigned Lh = warp_kth_largest_smem(mh, k, s32, lane);
        if (lo_zero) {
          // high words are whole keys: fewer than k lanes lie above Lh; if they hold fewer than k keys above Lh the answer is Lh
          // itself (a tie-heavy gauge: usually no lane lies above and nothing is gathered at all)
          const unsigned rows = __ballot_sync(kFull, mh > Lh);
          const int cnt = rows ? gather_rows<true>(wbase, rows, Lh + 1u, 0u, lane, lt_mask) : 0;
          if (cnt < k) { ans.hi = Lh; ans.lo = true_lo(Lh, 0u); done = true; }
          else if (cnt <= 32) { K64 unused; ans = select_from_candidates(cand, cnt, k, lane, &unused); done = true; }
          if (done) { wmax.hi = __reduce_max_sync(kFull, mh); wmax.lo = true_lo(wmax.hi, 0u); }
        } else {
          // at least k lane maxima reach Lh, so at least k keys pass: the k-th largest of the gathered set is the answer.  A class
          // of equal keys around the bound (a flat non-integer gauge) overflows the list; the gather stops early and the
          // 64-bit-bound path below takes over, where such a class collapses to its value.
          const int cnt = gather_rows<true>(wbase, __ballot_sync(kFull, mh >= Lh), Lh, 0u, lane, lt_mask);
          if (cnt <= 32) {
            ans = select_from_candidates(cand, cnt, k, lane, &wmax);
            done = true;
          }
        }
        __syncwarp();
      }
      if (!done) {
        // exact lane maximum: low words among this lane's own row entries that carry its top high word
        unsigned ml = 0u;
  #pragma unroll 4
        for (int i = 0; i < 32; ++i) {
          const unsigned long long kv = sk[lane * kRowU64 + i];
          if ((unsigned)(kv >> 32) == rmh) ml = max(ml, true_lo(mh, (unsigned)kv));
        }
        wmax = warp_max_k64(mh, ml);
        bool solved = false;
        if (k <= 32) {
          // medium path: exact 64-bit bound L = k-th largest lane maximum; ties collapse here (constant gauges)
          unsigned sh = mh, sl = ml;
          warp_sort_desc_k64(sh, sl, lane);
          const unsigned Lh = __shfl_sync(kFull, sh, k - 1), Ll = __shfl_sync(kFull, sl, k - 1);
          const int cnt = gather_rows<false>(wbase, __ballot_sync(kFull, k_gt(mh, ml, Lh, Ll)), Lh, Ll, lane, lt_mask);
          if (cnt < k) { ans.hi = Lh; ans.lo = Ll; solved = true; }
          else if (cnt <= 32) { K64 unused; ans = select_from_candidates(cand, cnt, k, lane, &unused); solved = true; }
          __syncwarp();
        }
        if (!solved) {
          // always-correct slow path: MSB-first bit search over the keys of this lane's row
          unsigned long long pref = 0ull;
          int kk2 = k;
  #pragma unroll 1
          for (int b = 63; b >= 0; --b) {
            const unsigned long long trial = pref | (1ull << b);
            const unsigned long long himask = ~((1ull << b) - 1ull);
            unsigned c = 0;
  #pragma unroll 4
            for (int i = 0; i < 32; ++i) c += ((true_key(sk[lane * kRowU64 + i]) & himask) == trial) ? 1u : 0u;
            c = __reduce_add_sync(kFull, c);
            if ((int)c >= kk2) pref = trial; else kk2 -= (int)c;
          }
          ans.hi = (unsigned)(pref >> 32);
          ans.lo = (unsigned)pref;
        }
      }
    } else {
      // ---- whole-range pass: no per-window order statistic.  Exact maximum the way the minimum is found, then the samples
      // flagged in pass 1 (lo <= x <= hi as doubles) are classified exactly on their totalOrder keys: above hi (+0 over a -0
      // pivot), == hi, == lo, below lo (-0 under a +0 pivot), and the rest - strictly inside - goes to the field's list.
      wmax.hi = __reduce_max_sync(kFull, mh);
      if (lo_zero) {
        wmax.lo = true_lo(wmax.hi, 0u);
      } else {
        unsigned rows = __ballot_sync(kFull, mh == wmax.hi);
        unsigned ml = 0u;
        const unsigned raw_max_hi = raw_hi_of(wmax.hi);
        if (__popc(rows) > 6) {
          rows = 0u;
#pragma unroll 4
          for (int i = 0; i < 32; ++i) {
            const unsigned long long kv = sk[lane * kRowU64 + i];
            if ((unsigned)(kv >> 32) == raw_max_hi && elem_index(lane, i) < m) ml = max(ml, true_lo(wmax.hi, (unsigned)kv));
          }
        }
        while (rows) {
          const int row = __ffs(rows) - 1;
          rows &= rows - 1;
          const unsigned long long kv = sk[row * kRowU64 + lane];
          if ((unsigned)(kv >> 32) == raw_max_hi && elem_index(row, lane) < m) ml = max(ml, true_lo(wmax.hi, (unsigned)kv));
        }
        wmax.lo = __reduce_max_sync(kFull, ml);
      }
      unsigned n_eh = 0, n_el = 0, n_in = 0;
      if (__any_sync(kFull, inmask != 0u)) {
        const unsigned long long lok = gpud_f64_key((unsigned long long)__double_as_longlong(piv_lo));
        const unsigned long long hik = gpud_f64_key((unsigned long long)__double_as_longlong(piv_hi));
        // equal pivots that are not a zero: lo <= x <= hi as doubles already means key == hi (a tie-heavy gauge: every flagged
        // sample is a copy of the pivot), no need to look at the keys
        const bool all_equal = lok == hik && piv_hi != 0.0;
        if (all_equal) { n_eh = (unsigned)__popc(inmask); inmask = 0u; }
        unsigned mm = inmask;
        while (mm) {
          const int i = __ffs(mm) - 1;
          mm &= mm - 1;
          const unsigned long long key = true_key(sk[lane * kRowU64 + i]);
          const bool inside = key > lok && key < hik;
          abv += key > hik ? 1u : 0u;
          n_eh += key == hik ? 1u : 0u;
          n_el += (key == lok && lok != hik) ? 1u : 0u;
          if (!inside) inmask ^= 1u << i;
        }
        const int c = __popc(inmask);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(kFull, incl, o);
          if (lane >= o) incl += t;
        }
        n_in = (unsigned)__shfl_sync(kFull, incl, 31);
        if (n_in) {
          unsigned base = 0;
          if (lane == 0) base = atomicAdd(p.fill + f, n_in);
          base = __shfl_sync(kFull, base, 0);
          unsigned pos = base + (unsigned)(incl - c);
          unsigned long long* __restrict__ list = p.lists + (int64_t)f * p.list_cap;
          mm = inmask;
          while (mm) {
            const int i = __ffs(mm) - 1;
            mm &= mm - 1;
            if (pos < p.list_cap) list[pos] = true_key(sk[lane * kRowU64 + i]);
            ++pos;
          }
        }
      }
      cls.x = __reduce_add_sync(kFull, abv);
      cls.y = __reduce_add_sync(kFull, n_eh);
      cls.z = __reduce_add_sync(kFull, n_el);
      cls.w = n_in;
    }
    __syncwarp();                            // every lane is done with this window's rows before pass 1 of the next overwrites them

    if (lane == 0) {
      const int64_t o = (int64_t)f * p.nw + w;
      p.out_min[o] = k64_to_f64(wmin);
      p.out_max[o] = k64_to_f64(wmax);
      p.out_mean[o] = (JF >= 0 || m == p.W) ? sum * p.inv_w : sum / (double)m;
      if (!RANGE && p.do_select) p.out_p99[o] = k64_to_f64(ans);
      if (RANGE) p.w_cls[o] = cls;
      p.out_nover[o] = nov;
      p.part[o] = ep;
    }
    cur = nxt;
  }
}

#ifdef GPUD_EXPERIMENT_TMA
// ---------------------------------------------------------------------------------------------
// K2+K4, in-place variant (EXPERIMENT, GPUD_WINDOW_LANDING=inplace): the window lands in the warp's 8 KB buffer through ONE
// cp.async.bulk and is processed where it landed - no register landing zone, no second copy into a row array - so an SM holds 20-24
// warps instead of 16.  The linear buffer dictates the element -> lane map: lane l owns the CONTIGUOUS elements 32 l .. 32 l + 31
// ("row" l = bytes [256 l, 256 l + 256)), which makes a row read (lane i reads entry i) conflict-free as it stands, and pass 1 / the
// own-row scans conflict-free when lane l starts at pair (or entry) l and walks cyclically.  Only full windows of an even W in
// 960 .. 1024 (the hot shape); everything else stays with k_window_reduce.
// ---------------------------------------------------------------------------------------------
#ifndef GPUD_INPLACE_WARPS
#define GPUD_INPLACE_WARPS 20
#endif
constexpr int kIpWarps = GPUD_INPLACE_WARPS;
constexpr int kIpRow = 32;                                        // u64 per row: the window itself
constexpr int kIpPadOff = 32 * kIpRow * 8;                        // 8192
constexpr int kIpCandOff = kIpPadOff + 256;
constexpr int kIpListOff = kIpCandOff + (kCandMax + 4) * 8;
constexpr int kIpWarpBytes = kIpListOff + 36 * 4 + 16;            // 9152

__global__ void __launch_bounds__(kIpWarps * 32, 1) k_window_reduce_inplace(const WinParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long s_bars[kIpWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char* wbase = smem_raw + (size_t)warp * kIpWarpBytes;
  unsigned long long* sk = reinterpret_cast<unsigned long long*>(wbase);                        // [32][32]: element t at sk[t]
  uint2* cand = reinterpret_cast<uint2*>(wbase + kIpCandOff);
  unsigned* s32 = reinterpret_cast<unsigned*>(cand);
  const unsigned stage_a = (unsigned)__cvta_generic_to_shared(wbase);
  const unsigned bar_a = (unsigned)__cvta_generic_to_shared(s_bars + warp);
  const unsigned lt_mask = (1u << lane) - 1u;
  const int m = p.W;                                                                             // every window here is full
  reinterpret_cast<unsigned long long*>(wbase + kIpPadOff)[lane] = kPadStored;                  // the pad row
  for (int t = m + lane; t < 1024; t += 32) sk[t] = kPadStored;                                  // entries past the window: never touched by the copy
  if (lane == 0) mbar_init(bar_a, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  const int per_f = p.nw;
  const int64_t n_units = (int64_t)p.F * p.nw;
  const int64_t stride = (int64_t)gridDim.x * kIpWarps;
  const int df = (int)(stride / per_f), ds = (int)(stride - (int64_t)df * per_f);
  int64_t u = (int64_t)blockIdx.x * kIpWarps + warp;
  int uf = (int)(u / per_f), uslot = (int)(u - (int64_t)uf * per_f);
  double thr_next = 0.0;
  auto fetch = [&](WinUnit& q) -> bool {
    for (;;) {
      if (u >= n_units) return false;
      q.f = uf; q.w = uslot;
      u += stride; uf += df; uslot += ds;
      if (uslot >= per_f) { uslot -= per_f; ++uf; }
      if (q.w != p.w_skip[0] && q.w != p.w_skip[1]) break;
    }
    q.p0 = p.start + (int64_t)q.w * p.W;
    if (q.p0 >= p.cap) q.p0 -= p.cap;
    thr_next = __ldg(p.thr + q.f);
    if (lane == 0) {
      mbar_expect(bar_a, m * 8);
      bulk_g2s(stage_a, p.ring + (int64_t)q.f * p.cap + q.p0, m * 8, bar_a);
    }
    return true;
  };
  // lane l, pair j <-> 16-byte chunk 32 j + ((l + j) & 31): consecutive samples stay spread over the lanes (the pigeonhole bounds need
  // that), pass 1 reads 32 distinct chunks of a 512-byte span per step, and a row's 16 chunks hit every 16-byte bank group twice
  const double a1 = 1.0 - p.alpha;
  const double w_first = __ldg(p.pw + (62 - 2 * lane + 63));        // (1-alpha)^(62 - 2 c) for c = lane: weight of pair 0 inside its 64-block
  const double w_step = __ldg(p.pw + (-2 + 63)), w_wrap = __ldg(p.pw + (62 + 63));   // c -> c + 1: x (1-alpha)^-2; c wraps 31 -> 0: x (1-alpha)^62
  const double tail_w = __ldg(p.pw + (m - 1024 + 63));               // the Horner below weighs sample t by (1-alpha)^(1023 - t)
  auto elem_at = [&](int row, int i) { return 64 * (i >> 1) + 2 * ((row + (i >> 1)) & 31) + (i & 1); };   // chronological index of (row, entry)

  WinUnit cur;
  int parity = 0;
  bool have = fetch(cur);
  while (have) {
    mbar_wait(bar_a, parity);
    parity ^= 1;
    const int f = cur.f, w = cur.w;
    const double thr = thr_next;
    // ---- pass 1 ----
    double sum0 = 0.0, sum1 = 0.0, acc = 0.0, wq = w_first;
    unsigned nov = 0, lor = 0u;
    int a_smax = (int)0x80000000;
    unsigned b_umin = 0xffffffffu, c_umax = 0u;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int c = (lane + j) & 31;
      const bool ok = 64 * j + 2 * c < m;                            // W is even: a pair is valid or not as a whole
      const double2 v = *reinterpret_cast<const double2*>(wbase + 512 * j + 16 * c);
      const double x0 = ok ? v.x : 0.0, x1 = ok ? v.y : 0.0;
      sum0 += x0; sum1 += x1;
      acc = fma(acc, p.q64, fma(x0, a1, x1) * wq);
      wq *= (c == 31) ? w_wrap : w_step;
      if (ok) {
        const int h0 = __double2hiint(x0), h1 = __double2hiint(x1);
        count_gt_f64(nov, x0, thr);
        count_gt_f64(nov, x1, thr);
        a_smax = max(a_smax, max(h0, h1));
        b_umin = min(b_umin, min((unsigned)h0, (unsigned)h1));
        c_umax = max(c_umax, max((unsigned)h0, (unsigned)h1));
        lor |= (unsigned)__double2loint(x0) | (unsigned)__double2loint(x1);
      }
    }
    const double e_lane = acc, lane_w = tail_w;
    const unsigned rmh = a_smax >= 0 ? (unsigned)a_smax : b_umin;
    const unsigned mh = key_hi_of(rmh);
    const bool lane_empty = c_umax == 0u && b_umin == 0xffffffffu;
    const unsigned nh = lane_empty ? 0xffffffffu : key_hi_of((c_umax & 0x80000000u) ? c_umax : b_umin);

    double ep = e_lane * lane_w, sum = sum0 + sum1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sum += __shfl_xor_sync(kFull, sum, o);
      ep += __shfl_xor_sync(kFull, ep, o);
    }
    ep *= p.alpha;
    nov = __reduce_add_sync(kFull, nov);
    const bool lo_zero = __reduce_or_sync(kFull, lor) == 0u;

    // ---- exact minimum ----
    K64 wmin;
    wmin.hi = __reduce_min_sync(kFull, nh);
    if (lo_zero) {
      wmin.lo = true_lo(wmin.hi, 0u);
    } else {
      unsigned rows = __ballot_sync(kFull, nh == wmin.hi);
      unsigned nl = 0xffffffffu;
      const unsigned raw_min_hi = raw_hi_of(wmin.hi);
      if (__popc(rows) > 6) {
        rows = 0u;
#pragma unroll 4
        for (int i = 0; i < 32; ++i) {
          const int t = elem_at(lane, i);
          const unsigned long long kv = sk[t];
          if ((unsigned)(kv >> 32) == raw_min_hi && t < m) nl = min(nl, true_lo(wmin.hi, (unsigned)kv));
        }
      }
      while (rows) {
        const int row = __ffs(rows) - 1;
        rows &= rows - 1;
        const int t = elem_at(row, lane);
        const unsigned long long kv = sk[t];
        if ((unsigned)(kv >> 32) == raw_min_hi && t < m) nl = min(nl, true_lo(wmin.hi, (unsigned)kv));
      }
      wmin.lo = __reduce_min_sync(kFull, nl);
    }

    // ---- exact order statistic + maximum (same scheme as k_window_reduce) ----
    const int k = p.k_full;
    K64 ans, wmax;
    ans.hi = ans.lo = 0u;
    bool done = false;
    if (k <= 32) {
      const unsigned Lh = warp_kth_largest_smem(mh, k, s32, lane);
      if (lo_zero) {
        const unsigned rows = __ballot_sync(kFull, mh > Lh);
        const int cnt = rows ? gather_rows<true, kIpRow, true>(wbase, rows, Lh + 1u, 0u, lane, lt_mask) : 0;
        if (cnt < k) { ans.hi = Lh; ans.lo = true_lo(Lh, 0u); done = true; }
        else if (cnt <= 32) { K64 unused; ans = select_from_candidates(cand, cnt, k, lane, &unused); done = true; }
        if (done) { wmax.hi = __reduce_max_sync(kFull, mh); wmax.lo = true_lo(wmax.hi, 0u); }
      } else {
        const int cnt = gather_rows<true, kIpRow, true>(wbase, __ballot_sync(kFull, mh >= Lh), Lh, 0u, lane, lt_mask);
        if (cnt <= 32) { ans = select_from_candidates(cand, cnt, k, lane, &wmax); done = true; }
      }
      __syncwarp();
    }
    if (!done) {
      unsigned ml = 0u;
#pragma unroll 4
      for (int i = 0; i < 32; ++i) {
        const unsigned long long kv = sk[elem_at(lane, i)];
        if ((unsigned)(kv >> 32) == rmh) ml = max(ml, true_lo(mh, (unsigned)kv));
      }
      wmax = warp_max_k64(mh, ml);
      bool solved = false;
      if (k <= 32) {
        unsigned sh = mh, sl = ml;
        warp_sort_desc_k64(sh, sl, lane);
        const unsigned Lh = __shfl_sync(kFull, sh, k - 1), Ll = __shfl_sync(kFull, sl, k - 1);
        const int cnt = gather_rows<false, kIpRow, true>(wbase, __ballot_sync(kFull, k_gt(mh, ml, Lh, Ll)), Lh, Ll, lane, lt_mask);
        if (cnt < k) { ans.hi = Lh; ans.lo = Ll; solved = true; }
        else if (cnt <= 32) { K64 unused; ans = select_from_candidates(cand, cnt, k, lane, &unused); solved = true; }
        __syncwarp();
      }
      if (!solved) {
        unsigned long long pref = 0ull;
        int kk2 = k;
#pragma unroll 1
        for (int b = 63; b >= 0; --b) {
          const unsigned long long trial = pref | (1ull << b);
          const unsigned long long himask = ~((1ull << b) - 1ull);
          unsigned c = 0;
#pragma unroll 4
          for (int i = 0; i < 32; ++i) c += ((true_key(sk[elem_at(lane, i)]) & himask) == trial) ? 1u : 0u;
          c = __reduce_add_sync(kFull, c);
          if ((int)c >= kk2) pref = trial; else kk2 -= (int)c;
        }
        ans.hi = (unsigned)(pref >> 32);
        ans.lo = (unsigned)pref;
      }
    }
    __syncwarp();                              // every lane is done with the buffer: the next window may land in it
    if (lane == 0) {
      const int64_t o = (int64_t)f * p.nw + w;
      p.out_min[o] = k64_to_f64(wmin);
      p.out_max[o] = k64_to_f64(wmax);
      p.out_mean[o] = sum * p.inv_w;
      if (p.do_select) p.out_p99[o] = k64_to_f64(ans);
      p.out_nover[o] = nov;
      p.part[o] = ep;
    }
    have = fetch(cur);
  }
}

#endif  // GPUD_EXPERIMENT_TMA

// ---------------------------------------------------------------------------------------------
// K3 carry: E_w = (1-alpha)^{m_w} E_{w-1} + P_w, E_{-1} = x[0] (oldest sample).  One 128-thread CTA per field:
// rows of 128 consecutive windows are scanned with a decayed Kogge-Stone prefix (S_t += d^off S_{t-off}), the carry
// crosses rows through shared memory; only the last window can have a different decay.
// SEEDED (the streaming drain): E_{-1} = seed_in[f], the EMA the previous drain ended on, instead of the first sample.  When seed_out
// is set, E of the last window is written there (seed_in may alias it: one thread reads it first and writes it last).
// ---------------------------------------------------------------------------------------------
template <bool SEEDED>
__global__ void __launch_bounds__(128) k_ema_carry(const double* __restrict__ part, const double* __restrict__ ring, int64_t cap,
                                                    int64_t start, int F, int nw, double d_full, double d_last,
                                                    double* __restrict__ out_ema, const double* seed_in, double* seed_out) {
  __shared__ double s_warp[4];
  __shared__ double s_carry;
  const int f = blockIdx.x, t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const double* __restrict__ P = part + (int64_t)f * nw;
  double* __restrict__ O = out_ema + (int64_t)f * nw;
  double dp[6];                              // d^1, d^2, d^4, d^8, d^16, d^32
  dp[0] = d_full;
#pragma unroll
  for (int i = 1; i < 6; ++i) dp[i] = dp[i - 1] * dp[i - 1];
  const double my_pow = pow(d_full, (double)(t + 1));        // d^(t+1): weight of the incoming carry at position t of a row
  const double lane_pow = pow(d_full, (double)(lane + 1));
  if (t == 0) s_carry = SEEDED ? seed_in[f] : ring[(int64_t)f * cap + start];
  __syncthreads();
  const int n_main = nw - 1;                 // windows with the full decay; the last window is folded in afterwards
  for (int row = 0; row * 128 < n_main; ++row) {
    const int w = row * 128 + t;
    double sacc = w < n_main ? __ldg(P + w) : 0.0;
    // inclusive decayed scan inside the warp
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const double o = __shfl_up_sync(kFull, sacc, 1 << i);
      if (lane >= (1 << i)) sacc = fma(dp[i], o, sacc);
    }
    if (lane == 31) s_warp[wid] = sacc;
    __syncthreads();
    // carry of the preceding warps of this row: sum_{v < wid} d^(32 (wid-1-v)) * s_warp[v], applied with d^(lane+1)
    double pre = 0.0;
    for (int v2 = 0; v2 < wid; ++v2) pre = fma(pre, dp[5], s_warp[v2]);
    sacc = fma(lane_pow, pre, sacc);
    const double e = fma(my_pow, s_carry, sacc);
    if (w < n_main) O[w] = e;
    __syncthreads();
    if (w == min(n_main, (row + 1) * 128) - 1) s_carry = e;   // the row's last valid window carries into the next row
    __syncthreads();
  }
  if (t == 0) {
    const double e = fma(d_last, s_carry, __ldg(P + nw - 1));
    O[nw - 1] = e;
    if (seed_out) seed_out[f] = e;
  }
}

}  // namespace

// =================================================================================================
// host side
// =================================================================================================
struct gpud_ring {
  gpud_ctx* ctx = nullptr;
  int dev = 0;
  int F = 0, W = 0;
  int64_t cap = 0;
  double alpha = 0;
  int q_num = 99, q_den = 100;
  int64_t total = 0;
  double* d_ring = nullptr;
  double* d_thr = nullptr;
  double* d_pw = nullptr;
  int64_t nw_max = 0;
  double* d_res[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  uint32_t* d_nover = nullptr;
  double* d_part = nullptr;
  int64_t reduced_nw = -1;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  double* h_stage[2] = {nullptr, nullptr};
  double* d_stage[2] = {nullptr, nullptr};
  cudaEvent_t ev_stage[2] = {nullptr, nullptr};    // d_stage[i] is free again (its append has run)
  cudaEvent_t ev_copied[2] = {nullptr, nullptr};   // the H2D into d_stage[i] has landed
  cudaStream_t copy_stream = nullptr;
  int64_t stage_rows = 0;
  double* d_sample = nullptr;      // [F][smp_slots]: column c with c % 2^smp_shift == 2^smp_shift / 2 lives at slot c >> smp_shift (kept by the append kernel)
  int smp_shift = 0;
  int64_t smp_slots = 0;
  double* d_pwl = nullptr;         // [32]: (1-alpha)^(W - 32 l - 32), the lane weights of the in-place kernel's EMA partial
  int sm_count = 148;
  bool inplace_landing = false, tma_landing = false;   // only ever set in a GPUD_EXPERIMENT_TMA build
  int cta_reserve = 0;           // CTA slots the persistent window grid leaves free for kernels of other streams (gpud_ring_set_cta_reserve)
  double* d_rng[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // range-reduce scratch: per-window min,max,mean,ema,partials
  size_t rng_bytes[5] = {0, 0, 0, 0, 0};
  uint32_t* d_rng_nover = nullptr;
  size_t rng_nover_bytes = 0;
  uint4* d_rng_cls = nullptr;                          // sampled range pass: per-window class counts
  size_t rng_cls_bytes = 0;
  unsigned long long* d_rng_lists = nullptr;           // sampled range pass: per-field lists of the keys between the pivots
  size_t rng_lists_bytes = 0;
  double* d_rng_piv = nullptr;                         // [F][2] pivots, then [F] u32 list fill counters
  size_t rng_piv_bytes = 0;
  cudaEvent_t ev_rng[3] = {nullptr, nullptr, nullptr}; // start / after the range pass / end of the last sampled reduce_range
  bool range_timed = false;
  int range_reasons[GPUD_RANGE_N_OPEN_REASONS] = {0};
  int range_fields_open = 0;                           // fields the last sampled reduce_range handed to the histogram path
  cudaEvent_t ev_k[3] = {nullptr, nullptr, nullptr};   // around the two kernels of the last reduce (bench roofline)
  // streaming drain (gpud_ring_drain): its own scratch, so a drain never changes what gpud_ring_read returns
  int64_t drain_next = 0;                              // first stream window not drained yet
  int64_t ema_window = -1;                             // the window whose EMA d_ema_state holds (-1: none)
  int64_t export_last_ms = INT64_MIN;                  // time the store writer gave the newest window it exported
  int64_t last_timed_ms = INT64_MIN;                   // time of the newest row that came through gpud_ring_push_timed
  std::vector<int64_t> win_ms;                         // [nw_max + 2]: end time of window k at k % size (0 = untimed)
  int64_t dr_chunk = 0;                                // windows per drain launch (the scratch below holds [F][dr_chunk])
  double* d_dr[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // min, max, mean, ema, p99
  uint32_t* d_dr_nover = nullptr;
  double* d_dr_part = nullptr;                         // per-window EMA partials
  double* d_ema_state = nullptr;                       // [F] EMA of window ema_window (committed)
  double* d_ema_pend = nullptr;                        // [F] EMA of the last window of the current peek
};

static int64_t ring_count(const gpud_ring* r) { return std::min(r->total, r->cap); }
static int64_t ring_start(const gpud_ring* r) { return r->total <= r->cap ? 0 : r->total % r->cap; }

extern "C" int32_t gpud_ring_create(gpud_ctx* ctx, int32_t dev, const gpud_ring_cfg* cfg, gpud_ring** out) {
  if (!ctx || !cfg || !out) return GPUD_E_INVALID;
  if (gpud_dev_slot(ctx, dev) < 0) return gpud_fail(ctx, GPUD_E_INVALID, "device %d is not part of this ctx", dev);
  if (cfg->n_fields < 1 || cfg->window < 1 || cfg->window > kMaxWindow || cfg->capacity < cfg->window || (cfg->capacity & 1))
    return gpud_fail(ctx, GPUD_E_INVALID, "ring cfg: need n_fields>=1, 1<=window<=%d, capacity even and >= window", kMaxWindow);
  double alpha = cfg->ema_alpha > 0 ? cfg->ema_alpha : std::min(2.0 / (cfg->window + 1.0), 0.9999);   // SPEC.md: default clamped
  if (!(alpha > 0.0) || alpha > 0.9999) return gpud_fail(ctx, GPUD_E_INVALID, "ema_alpha must be in (0, 0.9999]");
  int qn = cfg->q_num, qd = cfg->q_den;
  if (qn == 0 && qd == 0) { qn = 99; qd = 100; }
  if (qn < 0 || qd <= 0 || qn > qd) return gpud_fail(ctx, GPUD_E_INVALID, "quantile q_num/q_den must satisfy 0 <= num <= den");
  GPUD_CUDA(ctx, cudaSetDevice(dev));
  gpud_ring* r = new gpud_ring();
  r->ctx = ctx; r->dev = dev; r->F = cfg->n_fields; r->W = cfg->window; r->cap = cfg->capacity; r->alpha = alpha;
  r->q_num = qn; r->q_den = qd;
  r->sm_count = ctx->sm_count;
#ifdef GPUD_EXPERIMENT_TMA   /* `make EXPERIMENT_TMA=1`: the two cp.async.bulk landing variants measured in round 2 (profiles/r2/tma_landing_experiment.md) */
  { const char* env = getenv("GPUD_WINDOW_LANDING"); r->tma_landing = env && !strcmp(env, "tma"); r->inplace_landing = env && !strcmp(env, "inplace"); }
#endif
  r->nw_max = (r->cap + r->W - 1) / r->W;
  r->win_ms.assign((size_t)r->nw_max + 2, 0);
  const size_t ring_bytes = (size_t)r->F * r->cap * sizeof(double) + 64;   // slack: the 16-byte load of a window's last odd element
  const size_t res_bytes = (size_t)r->F * r->nw_max * sizeof(double);
  while (((r->cap + (1ll << r->smp_shift) - 1) >> r->smp_shift) > GPUD_RANGE_SAMPLE_MAX) ++r->smp_shift;
  r->smp_slots = (r->cap + (1ll << r->smp_shift) - 1) >> r->smp_shift;
  cudaError_t e = cudaMalloc(&r->d_ring, ring_bytes);
  if (e == cudaSuccess) e = cudaMemsetAsync(r->d_ring, 0, ring_bytes, 0);
  if (e == cudaSuccess) e = cudaMalloc(&r->d_sample, (size_t)r->F * r->smp_slots * sizeof(double));
  if (e == cudaSuccess) e = cudaMemsetAsync(r->d_sample, 0, (size_t)r->F * r->smp_slots * sizeof(double), 0);
  if (e == cudaSuccess) e = cudaMalloc(&r->d_thr, r->F * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&r->d_pw, 127 * sizeof(double));
  for (int i = 0; i < 5 && e == cudaSuccess; ++i) e = cudaMalloc(&r->d_res[i], res_bytes);
  if (e == cudaSuccess) e = cudaMalloc(&r->d_nover, (size_t)r->F * r->nw_max * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc(&r->d_part, res_bytes);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r->own_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r->copy_stream, cudaStreamNonBlocking);
  r->stage_rows = std::max<int64_t>(1, (int64_t)(kStageBytes / (sizeof(double) * r->F)));
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaMallocHost(&r->h_stage[i], (size_t)r->stage_rows * r->F * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&r->d_stage[i], (size_t)r->stage_rows * r->F * sizeof(double));
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r->ev_stage[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&r->ev_copied[i], cudaEventDisableTiming);
  }
  for (int i = 0; i < 3 && e == cudaSuccess; ++i) e = cudaEventCreate(&r->ev_k[i]);
  if (e != cudaSuccess) {
    int32_t rc = gpud_fail(ctx, e == cudaErrorMemoryAllocation ? GPUD_E_NOMEM : GPUD_E_CUDA, "ring_create: %s", cudaGetErrorString(e));
    gpud_ring_destroy(r);
    return rc;
  }
  r->stream = r->own_stream;
  std::vector<double> thr(r->F, INFINITY), pw(127);
  if (cfg->thresholds) std::copy(cfg->thresholds, cfg->thresholds + r->F, thr.begin());
  for (int ex = -63; ex <= 63; ++ex) pw[ex + 63] = pow(1.0 - alpha, (double)ex);
  GPUD_CUDA(ctx, cudaMemcpy(r->d_thr, thr.data(), r->F * sizeof(double), cudaMemcpyHostToDevice));
  GPUD_CUDA(ctx, cudaMemcpy(r->d_pw, pw.data(), 127 * sizeof(double), cudaMemcpyHostToDevice));
  {
    std::vector<double> pwl(32);
    for (int l = 0; l < 32; ++l) pwl[l] = pow(1.0 - alpha, (double)(r->W - 32 * l - 32));
    GPUD_CUDA(ctx, cudaMalloc(&r->d_pwl, 32 * sizeof(double)));
    GPUD_CUDA(ctx, cudaMemcpy(r->d_pwl, pwl.data(), 32 * sizeof(double), cudaMemcpyHostToDevice));
  }
  GPUD_CUDA(ctx, cudaDeviceSynchronize());
  *out = r;
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_destroy(gpud_ring* r) {
  if (!r) return GPUD_E_INVALID;
  cudaSetDevice(r->dev);
  if (r->own_stream) cudaStreamSynchronize(r->own_stream);
  cudaFree(r->d_ring); cudaFree(r->d_sample); cudaFree(r->d_pwl); cudaFree(r->d_thr); cudaFree(r->d_pw); cudaFree(r->d_nover); cudaFree(r->d_part);
  for (auto& p : r->d_res) cudaFree(p);
  for (auto& p : r->d_rng) cudaFree(p);
  cudaFree(r->d_rng_nover);
  cudaFree(r->d_rng_cls); cudaFree(r->d_rng_lists); cudaFree(r->d_rng_piv);
  for (auto& ev : r->ev_rng) if (ev) cudaEventDestroy(ev);
  for (auto& p : r->d_dr) cudaFree(p);
  cudaFree(r->d_dr_nover); cudaFree(r->d_dr_part); cudaFree(r->d_ema_state); cudaFree(r->d_ema_pend);
  for (int i = 0; i < 2; ++i) {
    if (r->h_stage[i]) cudaFreeHost(r->h_stage[i]);
    cudaFree(r->d_stage[i]);
    if (r->ev_stage[i]) cudaEventDestroy(r->ev_stage[i]);
    if (r->ev_copied[i]) cudaEventDestroy(r->ev_copied[i]);
  }
  for (auto& ev : r->ev_k) if (ev) cudaEventDestroy(ev);
  if (r->copy_stream) { cudaStreamSynchronize(r->copy_stream); cudaStreamDestroy(r->copy_stream); }
  if (r->own_stream) cudaStreamDestroy(r->own_stream);
  delete r;
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_set_cta_reserve(gpud_ring* r, int32_t n_ctas) {
  if (!r || n_ctas < 0 || n_ctas >= r->sm_count) return GPUD_E_INVALID;
  r->cta_reserve = n_ctas;
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_set_stream(gpud_ring* r, void* s) {
  if (!r) return GPUD_E_INVALID;
  r->stream = s ? (cudaStream_t)s : r->own_stream;
  return GPUD_OK;
}

static size_t dtype_size(int32_t dt) {
  switch (dt) {
    case GPUD_DT_F64: case GPUD_DT_I64: case GPUD_DT_U64: return 8;
    case GPUD_DT_U32: case GPUD_DT_I32: case GPUD_DT_F32: return 4;
    case GPUD_DT_U16: case GPUD_DT_I16: return 2;
    case GPUD_DT_U8: return 1;
  }
  return 0;
}

static int32_t launch_append(gpud_ring* r, const void* d_rows, int64_t n, int32_t dt) {
  // only the newest CAP rows can survive
  if (n > r->cap) {
    d_rows = (const char*)d_rows + (size_t)(n - r->cap) * r->F * dtype_size(dt);
    r->total += n - r->cap;
    n = r->cap;
  }
  const int64_t head = r->total % r->cap;
  const int64_t tiles = ((r->F + 31) / 32) * ((n + 31) / 32);
  const int grid = (int)std::min<int64_t>(tiles, (int64_t)r->sm_count * 16);
  switch (dt) {
    case GPUD_DT_F64: k_ring_append<double><<<grid, 256, 0, r->stream>>>((const double*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_U32: k_ring_append<uint32_t><<<grid, 256, 0, r->stream>>>((const uint32_t*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_I32: k_ring_append<int32_t><<<grid, 256, 0, r->stream>>>((const int32_t*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_F32: k_ring_append<float><<<grid, 256, 0, r->stream>>>((const float*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_I64: k_ring_append<long long><<<grid, 256, 0, r->stream>>>((const long long*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_U64: k_ring_append<unsigned long long><<<grid, 256, 0, r->stream>>>((const unsigned long long*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_U16: k_ring_append<uint16_t><<<grid, 256, 0, r->stream>>>((const uint16_t*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_I16: k_ring_append<int16_t><<<grid, 256, 0, r->stream>>>((const int16_t*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    case GPUD_DT_U8: k_ring_append<uint8_t><<<grid, 256, 0, r->stream>>>((const uint8_t*)d_rows, r->d_ring, n, r->F, r->cap, head, r->d_sample, r->smp_shift, (1ll << r->smp_shift) >> 1, r->smp_slots); break;
    default: return gpud_fail(r->ctx, GPUD_E_INVALID, "unknown sample dtype %d", dt);
  }
  GPUD_CUDA(r->ctx, cudaGetLastError());
  r->total += n;
  r->reduced_nw = -1;
  return GPUD_OK;
}

// Record the end time of every window the rows [old_total, total) completed: row_ms[i] is the time of row old_total + i, NULL = untimed
// (0).  Only the newest win_ms.size() windows can still be drained (the ring holds at most nw_max of them), so older ones are skipped.
static void stamp_windows(gpud_ring* r, int64_t old_total, const int64_t* row_ms) {
  const int64_t sz = (int64_t)r->win_ms.size();
  const int64_t k_end = r->total / r->W;
  const int64_t k_begin = std::max(old_total / r->W, k_end - sz);
  for (int64_t k = k_begin; k < k_end; ++k) r->win_ms[k % sz] = row_ms ? row_ms[(k + 1) * r->W - 1 - old_total] : 0;
}

extern "C" int32_t gpud_ring_push_device(gpud_ring* r, const double* dev_rows, int64_t n) {
  if (!r || (!dev_rows && n) || n < 0) return GPUD_E_INVALID;
  if (n == 0) return GPUD_OK;
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  const int64_t old_total = r->total;
  const int32_t rc = launch_append(r, dev_rows, n, GPUD_DT_F64);
  stamp_windows(r, old_total, nullptr);
  return rc;
}

static int32_t push_host(gpud_ring* r, const void* host_rows_v, int64_t n, int32_t dt);

extern "C" int32_t gpud_ring_push_raw(gpud_ring* r, const void* host_rows_v, int64_t n, int32_t dt) {
  if (!r || (!host_rows_v && n) || n < 0 || dtype_size(dt) == 0) return GPUD_E_INVALID;
  if (n == 0) return GPUD_OK;
  const int64_t old_total = r->total;
  const int32_t rc = push_host(r, host_rows_v, n, dt);
  stamp_windows(r, old_total, nullptr);
  return rc;
}

extern "C" int32_t gpud_ring_push_timed(gpud_ring* r, const void* host_rows_v, int64_t n, int32_t dt, const int64_t* row_ms) {
  if (!r || (!host_rows_v && n) || (!row_ms && n) || n < 0 || dtype_size(dt) == 0) return GPUD_E_INVALID;
  if (n == 0) return GPUD_OK;
  if (row_ms[0] < r->last_timed_ms)
    return gpud_fail(r->ctx, GPUD_E_INVALID, "push_timed: row time %lld is earlier than the last timed row (%lld)", (long long)row_ms[0], (long long)r->last_timed_ms);
  for (int64_t i = 1; i < n; ++i)
    if (row_ms[i] < row_ms[i - 1]) return gpud_fail(r->ctx, GPUD_E_INVALID, "push_timed: row times decrease at row %lld", (long long)i);
  const int64_t old_total = r->total;
  const int32_t rc = push_host(r, host_rows_v, n, dt);
  if (r->total > old_total) r->last_timed_ms = row_ms[r->total - old_total - 1];
  stamp_windows(r, old_total, row_ms);
  return rc;
}

// the body of gpud_ring_push_raw (arguments checked, n > 0)
static int32_t push_host(gpud_ring* r, const void* host_rows_v, int64_t n, int32_t dt) {
  const size_t esz = dtype_size(dt);
  const char* host_rows = (const char*)host_rows_v;
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  if (n > r->cap) {                      // rows that would be overwritten immediately never cross PCIe
    host_rows += (size_t)(n - r->cap) * r->F * esz;
    r->total += n - r->cap;
    n = r->cap;
  }
  cudaPointerAttributes attr;
  bool pinned = false;
  if (cudaPointerGetAttributes(&attr, host_rows) == cudaSuccess) pinned = attr.type == cudaMemoryTypeHost;
  else cudaGetLastError();
  // the staging pair is sized in bytes for stage_rows rows of doubles: narrower samples move more rows per piece
  const int64_t piece_rows = r->stage_rows * (int64_t)(sizeof(double) / esz);
  // Copies run on their own stream so the H2D of piece k+1 overlaps the append of piece k (PCIe never waits for K1):
  //   copy stream:    wait(free[buf]) -> H2D into d_stage[buf] -> record(copied[buf])
  //   compute stream: wait(copied[buf]) -> append from d_stage[buf] -> record(free[buf])
  int64_t done = 0;
  int buf = 0;
  while (done < n) {
    const int64_t rows = std::min(piece_rows, n - done);
    const size_t bytes = (size_t)rows * r->F * esz;
    const char* src = host_rows + (size_t)done * r->F * esz;
    if (!pinned) {
      GPUD_CUDA(r->ctx, cudaEventSynchronize(r->ev_copied[buf]));   // the previous H2D out of this pinned piece has finished
      gpud_parallel_memcpy(r->h_stage[buf], src, bytes);           // pageable caller memory: stage through pinned
      src = (const char*)r->h_stage[buf];
    }
    GPUD_CUDA(r->ctx, cudaStreamWaitEvent(r->copy_stream, r->ev_stage[buf], 0));   // the append that last read d_stage[buf] is done
    GPUD_CUDA(r->ctx, cudaMemcpyAsync(r->d_stage[buf], src, bytes, cudaMemcpyHostToDevice, r->copy_stream));
    GPUD_CUDA(r->ctx, cudaEventRecord(r->ev_copied[buf], r->copy_stream));
    GPUD_CUDA(r->ctx, cudaStreamWaitEvent(r->stream, r->ev_copied[buf], 0));
    int32_t rc = launch_append(r, r->d_stage[buf], rows, dt);
    if (rc) return rc;
    GPUD_CUDA(r->ctx, cudaEventRecord(r->ev_stage[buf], r->stream));
    done += rows;
    buf ^= 1;
  }
  if (pinned) GPUD_CUDA(r->ctx, cudaStreamSynchronize(r->stream));   // caller may reuse its buffer on return
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_push(gpud_ring* r, const double* host_rows, int64_t n) { return gpud_ring_push_raw(r, host_rows, n, GPUD_DT_F64); }

int gpud_ring_n_fields(const gpud_ring* r) { return r ? r->F : 0; }

extern "C" int32_t gpud_ring_counts(gpud_ring* r, int64_t* total, int64_t* count, int64_t* n_windows) {
  if (!r) return GPUD_E_INVALID;
  const int64_t c = ring_count(r);
  if (total) *total = r->total;
  if (count) *count = c;
  if (n_windows) *n_windows = (c + r->W - 1) / r->W;
  return GPUD_OK;
}


// Launch the window kernel(s).  The bulk goes to the aligned 128-bit instantiation (specialised for the window shape when
// W >> 6 is 15 or 16, i.e. W in 960..1024); the window that wraps the physical end of the ring and a trailing partial
// window go to the generic run-time instantiation, which also serves rings whose start is odd.
#ifdef GPUD_EXPERIMENT_TMA
template <int JF, bool RANGE>
static cudaError_t launch_one_tma(gpud_ring* r, const WinParams& p, int64_t units) {
  constexpr int kSmem = kTmaWarps * (kWarpSmemBytes + kStageBytesTma);
  cudaError_t e = cudaFuncSetAttribute(k_window_reduce<true, JF, RANGE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
  if (e != cudaSuccess) return e;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((units + kTmaWarps - 1) / kTmaWarps, (int64_t)r->sm_count - (r->cta_reserve ? 1 : 0)));
  k_window_reduce<true, JF, RANGE, true><<<grid, kTmaWarps * 32, kSmem, r->stream>>>(p);
  return cudaGetLastError();
}

static cudaError_t launch_inplace(gpud_ring* r, const WinParams& p, int64_t units) {
  constexpr int kSmem = kIpWarps * kIpWarpBytes;
  cudaError_t e = cudaFuncSetAttribute(k_window_reduce_inplace, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
  if (e != cudaSuccess) return e;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((units + kIpWarps - 1) / kIpWarps, (int64_t)r->sm_count - (r->cta_reserve ? 1 : 0)));
  k_window_reduce_inplace<<<grid, kIpWarps * 32, kSmem, r->stream>>>(p);
  return cudaGetLastError();
}

#endif  // GPUD_EXPERIMENT_TMA

template <bool ALIGNED, int JF, bool RANGE>
static cudaError_t launch_one(gpud_ring* r, const WinParams& p, int64_t units) {
  // persistent grid: 2 CTAs of 8 warps per SM, a whole number of waves (148 SMs)
  // 72 KB of dynamic shared memory per CTA (8 warps x (32 x 272 B key rows + candidate list)): opt in above 48 KB
  cudaError_t e = cudaFuncSetAttribute(k_window_reduce<ALIGNED, JF, RANGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kBlockSmemBytes);
  if (e != cudaSuccess) return e;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((units + kWarpsPerBlock - 1) / kWarpsPerBlock, (int64_t)r->sm_count * ((ALIGNED && JF >= 0) ? kHotCtasPerSM : 2) - r->cta_reserve));
  k_window_reduce<ALIGNED, JF, RANGE><<<grid, kWarpsPerBlock * 32, kBlockSmemBytes, r->stream>>>(p);
  return cudaGetLastError();
}

template <bool RANGE>
static int32_t launch_windows(gpud_ring* r, WinParams p) {
  {
    long long rr = ((long long)p.W * p.q_num + p.q_den - 1) / p.q_den;
    rr = rr < 1 ? 1 : (rr > p.W ? p.W : rr);
    p.k_full = p.W - (int)rr + 1;
    p.inv_w = 1.0 / (double)p.W;
  }
  p.n_list = 0;
  p.w_list[0] = p.w_list[1] = -1;
  p.w_skip[0] = p.w_skip[1] = -1;
  const int64_t units = (int64_t)p.F * p.nw;
  if ((p.start & 1) || ((p.W & 1) && p.nw > 1)) {          // some window would start on an odd element: 64-bit loads everywhere
    GPUD_CUDA(r->ctx, (launch_one<false, -1, RANGE>(r, p, units)));
    return GPUD_OK;
  }
  int n_skip = 0;
  const int64_t c_wrap = p.cap - p.start;                 // chronological index of the sample stored at physical column 0
  if (p.start > 0 && c_wrap < p.count && (c_wrap % p.W) != 0) p.w_skip[n_skip++] = (int)(c_wrap / p.W);
  const int jf = p.W >> 6;
  const bool special = (jf == 15 || jf == 16) && p.nw > 1;
  if (special && (p.count % p.W) != 0 && (n_skip == 0 || p.w_skip[0] != p.nw - 1)) p.w_skip[n_skip++] = p.nw - 1;   // trailing partial window
  cudaError_t e;
#ifdef GPUD_EXPERIMENT_TMA
  if (special && r->inplace_landing && !RANGE && (p.W & 1) == 0) e = launch_inplace(r, p, units);
  else if (special && r->tma_landing && jf == 15 && !RANGE) e = launch_one_tma<15, false>(r, p, units);
  else if (special && r->tma_landing && jf == 16) e = launch_one_tma<16, RANGE>(r, p, units);
  else
#endif
  if (special && jf == 15 && !RANGE) e = launch_one<true, 15, false>(r, p, units);   // the range pass always runs W' = 1024 (jf = 16)
  else if (special && jf == 16) e = launch_one<true, 16, RANGE>(r, p, units);
  else e = launch_one<true, -1, RANGE>(r, p, units);
  GPUD_CUDA(r->ctx, e);
  if (n_skip > 0) {
    p.n_list = n_skip;
    p.w_list[0] = p.w_skip[0];
    p.w_list[1] = p.w_skip[1];
    p.w_skip[0] = p.w_skip[1] = -1;
    GPUD_CUDA(r->ctx, (launch_one<false, -1, RANGE>(r, p, (int64_t)p.F * n_skip)));
  }
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_reduce(gpud_ring* r) {
  if (!r) return GPUD_E_INVALID;
  const int64_t count = ring_count(r);
  if (count == 0) return gpud_fail(r->ctx, GPUD_E_STATE, "ring is empty");
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  WinParams p;
  p.ring = r->d_ring; p.cap = r->cap; p.start = ring_start(r); p.count = count;
  p.W = r->W; p.F = r->F; p.nw = (int)((count + r->W - 1) / r->W);
  p.q_num = r->q_num; p.q_den = r->q_den; p.thr = r->d_thr; p.pw = r->d_pw; p.pwl = r->d_pwl;
  p.q64 = pow(1.0 - r->alpha, 64.0); p.alpha = r->alpha;
  p.out_min = r->d_res[GPUD_OP_MIN]; p.out_max = r->d_res[GPUD_OP_MAX]; p.out_mean = r->d_res[GPUD_OP_MEAN];
  p.out_p99 = r->d_res[GPUD_OP_P99]; p.out_nover = r->d_nover; p.part = r->d_part; p.do_select = 1;
  cudaEventRecord(r->ev_k[0], r->stream);
  { int32_t rc = launch_windows<false>(r, p); if (rc) return rc; }
  cudaEventRecord(r->ev_k[1], r->stream);
  const int m_last = (int)(count - (int64_t)(p.nw - 1) * r->W);
  k_ema_carry<false><<<r->F, 128, 0, r->stream>>>(r->d_part, r->d_ring, r->cap, p.start, r->F, p.nw,
                                                        pow(1.0 - r->alpha, (double)r->W), pow(1.0 - r->alpha, (double)m_last),
                                                        r->d_res[GPUD_OP_EMA], nullptr, nullptr);
  GPUD_CUDA(r->ctx, cudaGetLastError());
  cudaEventRecord(r->ev_k[2], r->stream);
  r->reduced_nw = p.nw;
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_kernel_ms(gpud_ring* r, float* reduce_ms, float* carry_ms) {
  if (!r || !reduce_ms || !carry_ms) return GPUD_E_INVALID;
  if (r->reduced_nw < 0) return gpud_fail(r->ctx, GPUD_E_STATE, "no reduce since the last push");
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  GPUD_CUDA(r->ctx, cudaEventSynchronize(r->ev_k[2]));
  GPUD_CUDA(r->ctx, cudaEventElapsedTime(reduce_ms, r->ev_k[0], r->ev_k[1]));
  GPUD_CUDA(r->ctx, cudaEventElapsedTime(carry_ms, r->ev_k[1], r->ev_k[2]));
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_sync(gpud_ring* r) {
  if (!r) return GPUD_E_INVALID;
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  GPUD_CUDA(r->ctx, cudaStreamSynchronize(r->stream));
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_result_ptr(gpud_ring* r, int32_t op, void** dev_ptr) {
  if (!r || !dev_ptr || op < 0 || op >= GPUD_N_OPS) return GPUD_E_INVALID;
  if (r->reduced_nw < 0) return gpud_fail(r->ctx, GPUD_E_STATE, "no reduce since the last push");
  *dev_ptr = op == GPUD_OP_NOVER ? (void*)r->d_nover : (void*)r->d_res[op];
  return GPUD_OK;
}

extern "C" int32_t gpud_ring_read(gpud_ring* r, int32_t op, void* out, int64_t out_bytes) {
  if (!r || !out || op < 0 || op >= GPUD_N_OPS) return GPUD_E_INVALID;
  if (r->reduced_nw < 0) return gpud_fail(r->ctx, GPUD_E_STATE, "no reduce since the last push");
  const size_t el = op == GPUD_OP_NOVER ? sizeof(uint32_t) : sizeof(double);
  const size_t need = (size_t)r->F * r->reduced_nw * el;
  if ((size_t)out_bytes < need) return gpud_fail(r->ctx, GPUD_E_CAPACITY, "need %zu bytes", need);
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  const void* src = op == GPUD_OP_NOVER ? (const void*)r->d_nover : (const void*)r->d_res[op];
  GPUD_CUDA(r->ctx, cudaMemcpyAsync(out, src, need, cudaMemcpyDeviceToHost, r->stream));
  GPUD_CUDA(r->ctx, cudaStreamSynchronize(r->stream));
  return GPUD_OK;
}

// ---- streaming drain: stream-aligned windows, each reduced once, into the drain's own scratch ----
// A drain launches the same window kernel over windows [k0, k0 + n) of the stream: physical start (k0 W) mod CAP, n W samples.  Once the
// ring has wrapped, a window can straddle column CAP-1 -> 0 (CAP mod W != 0) or start on an odd column (odd W); launch_windows sends
// those to the generic instantiation exactly as it does for gpud_ring_reduce.
constexpr int64_t kDrainUnits = 1 << 20;   // (field, window) pairs per drain launch: bounds the scratch at F x chunk x 52 B

static void drain_counts(const gpud_ring* r, int64_t max_windows, gpud_drain_info* info) {
  const int64_t W = r->W, count = ring_count(r);
  const int64_t complete = r->total / W;
  const int64_t k0 = std::max(r->drain_next, (r->total - count + W - 1) / W);
  const int64_t avail = complete - k0;
  info->first_window = k0;
  info->n_windows = std::min(avail, max_windows);
  info->n_lost = k0 - r->drain_next;
  info->n_pending = avail - info->n_windows;
}

int32_t gpud_ring_drain_peek(gpud_ring* r, int64_t max_windows, double* out_f64, uint32_t* out_nover, int64_t* out_ms, gpud_drain_info* info) {
  drain_counts(r, max_windows, info);
  const int64_t k0 = info->first_window, n = info->n_windows;
  if (n == 0) return GPUD_OK;
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  if (!r->d_ema_state) {
    for (auto& p : r->d_dr) { cudaFree(p); p = nullptr; }      // whatever an earlier, failed attempt left
    cudaFree(r->d_dr_nover); cudaFree(r->d_dr_part); cudaFree(r->d_ema_pend);
    r->d_dr_nover = nullptr; r->d_dr_part = r->d_ema_pend = nullptr;
    r->dr_chunk = std::max<int64_t>(1, std::min<int64_t>(r->nw_max, kDrainUnits / r->F));
    const size_t per = (size_t)r->F * r->dr_chunk;
    for (int i = 0; i < 5; ++i) GPUD_CUDA(r->ctx, cudaMalloc(&r->d_dr[i], per * sizeof(double)));
    GPUD_CUDA(r->ctx, cudaMalloc(&r->d_dr_nover, per * sizeof(uint32_t)));
    GPUD_CUDA(r->ctx, cudaMalloc(&r->d_dr_part, per * sizeof(double)));
    GPUD_CUDA(r->ctx, cudaMalloc(&r->d_ema_pend, r->F * sizeof(double)));
    GPUD_CUDA(r->ctx, cudaMalloc(&r->d_ema_state, r->F * sizeof(double)));   // allocated last: its presence means the scratch is complete
  }
  // the EMA continues from the previous drain only when that drain ended on window k0 - 1 (no loss in between)
  const bool carry = k0 > 0 && r->ema_window == k0 - 1;
  const double d_w = pow(1.0 - r->alpha, (double)r->W);
  for (int64_t j0 = 0; j0 < n; j0 += r->dr_chunk) {
    const int64_t nc = std::min(r->dr_chunk, n - j0);
    WinParams p;
    p.ring = r->d_ring; p.cap = r->cap; p.start = ((k0 + j0) * r->W) % r->cap; p.count = nc * r->W;
    p.W = r->W; p.F = r->F; p.nw = (int)nc;
    p.q_num = r->q_num; p.q_den = r->q_den; p.thr = r->d_thr; p.pw = r->d_pw; p.pwl = r->d_pwl;
    p.q64 = pow(1.0 - r->alpha, 64.0); p.alpha = r->alpha;
    p.out_min = r->d_dr[GPUD_OP_MIN]; p.out_max = r->d_dr[GPUD_OP_MAX]; p.out_mean = r->d_dr[GPUD_OP_MEAN];
    p.out_p99 = r->d_dr[GPUD_OP_P99]; p.out_nover = r->d_dr_nover; p.part = r->d_dr_part; p.do_select = 1;
    { int32_t rc = launch_windows<false>(r, p); if (rc) return rc; }
    if (j0 == 0 && !carry)
      k_ema_carry<false><<<r->F, 128, 0, r->stream>>>(r->d_dr_part, r->d_ring, r->cap, p.start, r->F, (int)nc, d_w, d_w, r->d_dr[GPUD_OP_EMA],
                                                       nullptr, r->d_ema_pend);
    else
      k_ema_carry<true><<<r->F, 128, 0, r->stream>>>(r->d_dr_part, r->d_ring, r->cap, p.start, r->F, (int)nc, d_w, d_w, r->d_dr[GPUD_OP_EMA],
                                                      j0 == 0 ? r->d_ema_state : r->d_ema_pend, r->d_ema_pend);
    GPUD_CUDA(r->ctx, cudaGetLastError());
    // only the nc new windows cross PCIe, one strided copy per output straight into the caller's layout
    for (int op = 0; op < 5; ++op)
      GPUD_CUDA(r->ctx, cudaMemcpy2DAsync(out_f64 + ((size_t)op * r->F) * max_windows + j0, (size_t)max_windows * sizeof(double), r->d_dr[op],
                                          (size_t)nc * sizeof(double), (size_t)nc * sizeof(double), (size_t)r->F, cudaMemcpyDeviceToHost, r->stream));
    GPUD_CUDA(r->ctx, cudaMemcpy2DAsync(out_nover + j0, (size_t)max_windows * sizeof(uint32_t), r->d_dr_nover, (size_t)nc * sizeof(uint32_t),
                                        (size_t)nc * sizeof(uint32_t), (size_t)r->F, cudaMemcpyDeviceToHost, r->stream));
  }
  GPUD_CUDA(r->ctx, cudaStreamSynchronize(r->stream));
  if (out_ms) {
    const int64_t sz = (int64_t)r->win_ms.size();
    for (int64_t j = 0; j < n; ++j) out_ms[j] = r->win_ms[(k0 + j) % sz];
  }
  return GPUD_OK;
}

void gpud_ring_drain_commit(gpud_ring* r, const gpud_drain_info* info, int64_t last_export_ms) {
  r->drain_next = info->first_window + info->n_windows;
  if (info->n_windows > 0) {
    // stream-ordered after the peek's carry kernel; both buffers are only ever read by later launches on the same stream
    cudaSetDevice(r->dev);
    cudaMemcpyAsync(r->d_ema_state, r->d_ema_pend, r->F * sizeof(double), cudaMemcpyDeviceToDevice, r->stream);
    r->ema_window = r->drain_next - 1;
  }
  if (last_export_ms != INT64_MIN) r->export_last_ms = last_export_ms;
}

int64_t gpud_ring_drain_last_export(const gpud_ring* r) { return r->export_last_ms; }

extern "C" int32_t gpud_ring_drain(gpud_ring* r, int64_t max_windows, double* out_f64, uint32_t* out_nover, int64_t* out_ms, gpud_drain_info* info) {
  if (!r || !info || max_windows < 0 || (max_windows > 0 && (!out_f64 || !out_nover))) return GPUD_E_INVALID;
  const int32_t rc = gpud_ring_drain_peek(r, max_windows, out_f64, out_nover, out_ms, info);
  if (rc) return rc;
  if (max_windows > 0) gpud_ring_drain_commit(r, info, INT64_MIN);
  return GPUD_OK;
}

// ---- range reduce support (select.cu): the window kernel with W' = 1024 over the newest `n` samples, into scratch ----
// gpud_ring_range_prepare sizes the scratch and fills the view; gpud_ring_range_pass launches the pass (+ the EMA carry) in the
// mode the view names: plain (per-window min / max / mean / EMA partial / n_over) or sampled (the same, plus every sample
// classified against the field's pivot pair and the keys between the pivots parked in the field's list).
static cudaError_t grow(void** ptr, size_t* have, size_t need) {
  if (need <= *have) return cudaSuccess;
  cudaFree(*ptr);
  *ptr = nullptr;
  *have = 0;
  cudaError_t e = cudaMalloc(ptr, need);
  if (e == cudaSuccess) *have = need;
  return e;
}

int32_t gpud_ring_range_prepare(gpud_ring* r, int64_t n, gpud_range_view* v) {
  const int64_t count = ring_count(r);
  if (n <= 0 || n > count) n = count;
  const int Wp = (int)std::min<int64_t>(kMaxWindow, n);
  const int nw = (int)((n + Wp - 1) / Wp);
  const size_t per = (size_t)r->F * nw;
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  for (int i = 0; i < 5; ++i) GPUD_CUDA(r->ctx, grow((void**)&r->d_rng[i], &r->rng_bytes[i], per * sizeof(double)));
  GPUD_CUDA(r->ctx, grow((void**)&r->d_rng_nover, &r->rng_nover_bytes, per * sizeof(uint32_t)));
  const bool sampled = n >= GPUD_RANGE_SAMPLED_MIN;
  const unsigned list_cap = (unsigned)std::min<int64_t>(GPUD_RANGE_LIST_CAP, n);
  if (sampled) {
    GPUD_CUDA(r->ctx, grow((void**)&r->d_rng_cls, &r->rng_cls_bytes, per * sizeof(uint4)));
    GPUD_CUDA(r->ctx, grow((void**)&r->d_rng_lists, &r->rng_lists_bytes, (size_t)r->F * list_cap * sizeof(unsigned long long)));
    GPUD_CUDA(r->ctx, grow((void**)&r->d_rng_piv, &r->rng_piv_bytes, (size_t)r->F * (2 * sizeof(double) + sizeof(unsigned))));
  }
  for (auto& ev : r->ev_rng) if (!ev) GPUD_CUDA(r->ctx, cudaEventCreate(&ev));
  int64_t start = ring_start(r) + (count - n);
  if (start >= r->cap) start -= r->cap;
  v->ring = r->d_ring; v->F = r->F; v->cap = r->cap; v->start = start; v->n = n; v->Wp = Wp; v->nw = nw;
  v->w_min = r->d_rng[0]; v->w_max = r->d_rng[1]; v->w_mean = r->d_rng[2]; v->w_ema = r->d_rng[3]; v->w_nover = r->d_rng_nover;
  v->q_num = r->q_num; v->q_den = r->q_den; v->stream = r->stream; v->ctx = r->ctx; v->dev = r->dev; v->sm_count = r->sm_count;
  v->sampled = sampled ? 1 : 0;
  v->sample = r->d_sample; v->smp_shift = r->smp_shift; v->smp_slots = r->smp_slots;
  v->list_cap = list_cap;
  v->piv = sampled ? r->d_rng_piv : nullptr;
  v->fill = sampled ? reinterpret_cast<unsigned*>(r->d_rng_piv + 2 * (size_t)r->F) : nullptr;
  v->w_cls = sampled ? r->d_rng_cls : nullptr;
  v->lists = sampled ? r->d_rng_lists : nullptr;
  for (int i = 0; i < 3; ++i) v->ev[i] = r->ev_rng[i];
  r->range_timed = false;
  return GPUD_OK;
}

int32_t gpud_ring_range_pass(gpud_ring* r, const gpud_range_view* v) {
  WinParams p;
  p.ring = r->d_ring; p.cap = r->cap; p.start = v->start; p.count = v->n; p.W = v->Wp; p.F = r->F; p.nw = v->nw;
  p.q_num = r->q_num; p.q_den = r->q_den; p.thr = r->d_thr; p.pw = r->d_pw; p.q64 = pow(1.0 - r->alpha, 64.0); p.alpha = r->alpha;
  p.out_min = r->d_rng[0]; p.out_max = r->d_rng[1]; p.out_mean = r->d_rng[2]; p.out_p99 = nullptr; p.out_nover = r->d_rng_nover;
  p.part = r->d_rng[4]; p.do_select = 0;
  p.piv = v->piv; p.w_cls = v->w_cls; p.lists = v->lists; p.fill = v->fill; p.list_cap = v->list_cap;
  { int32_t rc = v->sampled ? launch_windows<true>(r, p) : launch_windows<false>(r, p); if (rc) return rc; }
  const int m_last = (int)(v->n - (int64_t)(v->nw - 1) * v->Wp);
  k_ema_carry<false><<<r->F, 128, 0, r->stream>>>(r->d_rng[4], r->d_ring, r->cap, v->start, r->F, v->nw, pow(1.0 - r->alpha, (double)v->Wp),
                                                        pow(1.0 - r->alpha, (double)m_last), r->d_rng[3], nullptr, nullptr);
  GPUD_CUDA(r->ctx, cudaGetLastError());
  return GPUD_OK;
}

void gpud_ring_range_note(gpud_ring* r, bool sampled, unsigned fields_open, const int* reasons) {
  r->range_timed = sampled;
  r->range_fields_open = (int)fields_open;
  for (int i = 0; i < GPUD_RANGE_N_OPEN_REASONS; ++i) r->range_reasons[i] = reasons[i];
}

extern "C" int32_t gpud_ring_range_stats(gpud_ring* r, float* pass_ms, float* total_ms, int32_t* fields_by_histogram, int32_t* reasons) {
  if (!r || !pass_ms || !total_ms || !fields_by_histogram) return GPUD_E_INVALID;
  if (!r->range_timed) return gpud_fail(r->ctx, GPUD_E_STATE, "the last reduce_range (if any) did not take the sampled single pass");
  GPUD_CUDA(r->ctx, cudaSetDevice(r->dev));
  GPUD_CUDA(r->ctx, cudaEventSynchronize(r->ev_rng[2]));
  GPUD_CUDA(r->ctx, cudaEventElapsedTime(pass_ms, r->ev_rng[0], r->ev_rng[1]));
  GPUD_CUDA(r->ctx, cudaEventElapsedTime(total_ms, r->ev_rng[0], r->ev_rng[2]));
  *fields_by_histogram = r->range_fields_open;
  if (reasons) for (int i = 0; i < GPUD_RANGE_N_OPEN_REASONS; ++i) reasons[i] = r->range_reasons[i];
  return GPUD_OK;
}

void gpud_ring_quantile(gpud_ring* r, int* q_num, int* q_den) { *q_num = r->q_num; *q_den = r->q_den; }
