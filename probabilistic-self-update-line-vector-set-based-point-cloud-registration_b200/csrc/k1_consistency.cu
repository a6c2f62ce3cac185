// k1_consistency.cu -- stage 1: line-vector length-consistency bit mask, edge compaction.
//
// Replaces the reference's O(C^2) line-vector set build and the ScaleInliersSelector pass
// (registration.cc:693-732, :418-434, :756-766).  The reference materialises every line vector
// (~130 B per pair, twice); here a pair costs 10 FP32 lane-operations (5 packed FFMA2 / FADD2 issue slots) + 2 ALU
// instructions and one output BIT.
//
// Arithmetic.  The reference decides   | sqrt(A) - sqrt(B) | <= beta   in FP64 with
// A = |s_j - s_i|^2, B = |t_j - t_i|^2.  With D = A - B, S = A + B this is, for a + b > beta,
//        v := D^2 - 2 beta^2 S + beta^4 = (u^2 - beta^2)((a+b)^2 - beta^2) <= 0 ,   u = |a - b| ,
// a sqrt-free polynomial whose FP32 evaluation error is bounded by  kappa * S  (derivation in
// DESIGN.md "K1 error band").  Every pair with |v| inside that band, or with S <= ~beta^2 (where
// the factor (a+b)^2 - beta^2 may change sign), is re-evaluated in FP64 with the reference's exact
// operation order, so the emitted bits equal the FP64 reference's bit for bit; the number of
// re-evaluated pairs is counted.
//
// Fast path.  A and B are formed in the "norm" form  |s_i|^2 + |s_j|^2 - 2 s_i.s_j  (the squared
// norms travel in the .w lane of the float4 tiles, -2 s_i and the per-row constants are pre-folded in registers;
// see pair_fast / pair_fast2).  That form loses relative accuracy for short line vectors, so its sign is
// trusted only when |v| exceeds ONE uniform threshold t_fast (derivation in DESIGN.md "K1 fast-path
// threshold"; it also covers a + b <= beta, where the polynomial's sign is not the answer); a mask
// word with any pair below it is redone with the accurate difference form above, whose own band
// decides what goes to FP64.
//
// Mapping.  One thread owns R rows (its points live in registers as scalars), the CTA's column tile -- pair-
// interleaved records, so that two neighbouring columns share a 64-bit register pair (see pair_fast2) -- is staged
// in shared memory by a 1-D TMA bulk copy (cp.async.bulk + mbarrier) and read as warp-wide
// broadcasts; a thread accumulates the 32 result bits of a mask word with a funnel shift of v's
// sign bit, so no ballot and no divergence on the fast path.  Words that are only partly live for some row (its
// diagonal, the arrays' end) keep their dead columns out of the doubt test (eval_word_masked).
#include <cuda_runtime.h>

#include <type_traits>

#include <cstdlib>

#include "common.cuh"
#include "engine.cuh"

namespace psulvsb {

namespace {

constexpr int K1_THREADS = 256;
#ifndef K1_COLPAIR_UNROLL
#define K1_COLPAIR_UNROLL 4  // column pairs per unrolled step of the word loop (8 columns, as before)
#endif
#ifndef K1_R4_CTAS
#define K1_R4_CTAS 2  // measured with the packed fast path: 3 CTAs per SM (80 registers, 36 B of spills) 2.19 ms vs 2.05 ms
#endif

// exact FP64 test, reference operation order (registration.cc:425-433, SURVEY appendix A.2)
__device__ __forceinline__ bool exact_consistent(const double* __restrict__ s64, const double* __restrict__ t64, int i,
                                                 int j, double beta) {
  const double sx = dsub(s64[3 * j + 0], s64[3 * i + 0]);
  const double sy = dsub(s64[3 * j + 1], s64[3 * i + 1]);
  const double sz = dsub(s64[3 * j + 2], s64[3 * i + 2]);
  const double tx = dsub(t64[3 * j + 0], t64[3 * i + 0]);
  const double ty = dsub(t64[3 * j + 1], t64[3 * i + 1]);
  const double tz = dsub(t64[3 * j + 2], t64[3 * i + 2]);
  const double a = sqrt(sqnorm3(sx, sy, sz));
  const double b = sqrt(sqnorm3(tx, ty, tz));
  return fabs(dsub(a, b)) <= beta;
}

// FP32 evaluation of one pair: returns v (sign bit set <=> consistent), w = |v| - kappa S', sp = S'
__device__ __forceinline__ void pair_eval(const float4 si, const float4 ti, const float4 sj, const float4 tj,
                                          const K1Consts& c, float& v, float& w, float& sp) {
  const float sx = sj.x - si.x, sy = sj.y - si.y, sz = sj.z - si.z;
  const float tx = tj.x - ti.x, ty = tj.y - ti.y, tz = tj.z - ti.z;
  const float A = fmaf(sz, sz, fmaf(sy, sy, fmaf(sx, sx, -c.half_bias)));
  const float B = fmaf(tz, tz, fmaf(ty, ty, fmaf(tx, tx, -c.half_bias)));
  const float D = A - B;
  sp = A + B;
  const float r = fmaf(c.two_beta2, sp, c.r0);
  v = fmaf(D, D, -r);
  w = fmaf(-c.kappa, sp, fabsf(v));
}

// fast path, norm form: with a = |s_i - s_j|^2 and b = |t_i - t_j|^2 the pair is consistent iff
//   v = (a - b)^2 - (2 beta^2 (a + b) - beta^4) = (a - b - beta^2)^2 - 4 beta^2 b <= 0   (and a + b > beta, see t_fast).
// Column point as (x, y, z, |p|^2).  Row registers: ms = (-2 x, -2 y, -2 z, c1), mt = (-2 x, -2 y, -2 z, c2) with the
// per-row constants c1 = |s_i|^2 - |t_i|^2 - beta^2 and c2 = -4 beta^2 |t_i|^2 folded in, so that with
//   A = |s_j|^2 - 2 s_i.s_j,  B = |t_j|^2 - 2 t_i.t_j   (3 FMA each)
//   u = (A - B) + c1 = a - b - beta^2   (2 FADD),   w = -4 beta^2 B + c2 = -4 beta^2 b   (1 FMA),   v = u u + w   (1 FMA):
// 8 FMA + 2 FADD per pair (adding the row norms per pair and forming a + b cost two more).  Every partial sum stays
// below 9 Cmax^2 and the constants carry two more float roundings of 6 Cmax^2: inside the E, ED, ES of
// make_k1_consts (80 / 172 / 184 mu Cmax^2 against ~41 / ~120 needed; the w term errs by 4 beta^2 E + 60 mu beta^2
// Cmax^2, less than the 2 beta^2 ES + 2 mu (48 beta^2 Cmax^2 + beta^4) budgeted for r); |u| <= |a - b| + beta^2 is
// accounted for in Dlim.
__device__ __forceinline__ float pair_fast(const float4 ms, const float4 mt, const float4 sj, const float4 tj,
                                           const float neg_four_beta2, const float beta4) {
  (void)beta4;
  const float A = fmaf(ms.x, sj.x, fmaf(ms.y, sj.y, fmaf(ms.z, sj.z, sj.w)));
  const float B = fmaf(mt.x, tj.x, fmaf(mt.y, tj.y, fmaf(mt.z, tj.z, tj.w)));
  const float u = (A - B) + ms.w;
  const float w = fmaf(neg_four_beta2, B, mt.w);
  return fmaf(u, u, w);
}

// What the slow path needs, staged once per CTA in shared memory: the path is rare per pair but a cfg-A batch
// takes it for 1.7 % of the mask words, and reading these through the job record (pointer -> point: two
// dependent global loads per call) made it 19 % of the kernel's warp time (ncu source page, long scoreboard).
struct K1Slow {
  K1Consts c;
  const double* src64;
  const double* dst64;
  int n;
};

// Slow path (rare): the mask word of row i, columns cb .. cb+31, redone by the whole warp -- lane b
// takes pair (i, cb + b) in the accurate difference form; what falls inside ITS rigorous band is
// decided in FP64 with the reference's operation order; the 32 verdicts come back as one ballot.
// (si, ti) = the row's packed point, broadcast from its owner lane's registers (.w unused here).
__device__ __noinline__ uint32_t slow_word_coop(const K1Slow& sl, int i, int cb, const float4 si, const float4 ti,
                                                const float4 sj, const float4 tj, unsigned int& nborder) {
  const int lane = threadIdx.x & 31;
  float v, w, sp;
  pair_eval(si, ti, sj, tj, sl.c, v, w, sp);
  bool in = (__float_as_uint(v) >> 31) != 0u;
  const int j = cb + lane;
  if ((!(w > sl.c.w_thr) || !(sp > 0.f)) && j < sl.n && j > i) {
    ++nborder;
    in = exact_consistent(sl.src64, sl.dst64, i, j, sl.c.beta);
  }
  return __ballot_sync(0xffffffffu, in);
}

// Packed FP32 (Blackwell FFMA2, PTX fma.rn.f32x2: two FP32 operations per lane and issue slot).  COLUMNS travel in
// pairs: the tiles are pair-interleaved (common.cuh il_store), one LDS.128 delivers the same coordinate of columns
// (2q, 2q + 1) in an aligned register pair, and a thread's row values enter as scalar broadcasts (ptxas folds a {x, x}
// operand into the instruction's .F32 operand form: no MOV).  Each half is an IEEE round-to-nearest fma: v is bit
// for bit what pair_fast computes.  Why columns and not rows in the halves (r2, profiles/tools/fp32_pipe_probe.cu):
//   * an FFMA2 whose 64-bit operand is the one consecutive instructions share (here: a column pair's coordinate,
//     used by each of the thread's R rows in turn) sustains 0.99 of the FP32 peak; sharing the 32-bit scalar instead
//     (rows packed, what the kernel did before) 0.92, because the register file then delivers 128 instead of 96 bits
//     per lane and instruction;
//   * ALU-pipe instructions are not free beside the FP32 pipe -- each costs ~ 1.6 - 2.3 issue cycles that FFMA2s
//     cannot use -- and with both columns of a result pair in one row the band tracking is ONE three-input FMNMX3 per
//     two pairs instead of two FMNMX;
//   * no half-live register pairs along the diagonal: a dead row costs nothing.
// pair_fast for one row against a column pair: 8 FFMA2 + 2 FFMA2 ((A - B) as fma(B, -1, A) and (.) + c1 as
// fma(., 1, c1): one rounding each, the FADD's value) = 10 packed instructions for two pairs
__device__ __forceinline__ float2 pair_fast2(const float4 ms, const float4 mt, const float4 sa, const float4 sb,
                                             const float4 ta, const float4 tb, const float neg_four_beta2) {
  const float2 A = fma2(bc2(ms.x), make_float2(sa.x, sa.y),
                        fma2(bc2(ms.y), make_float2(sa.z, sa.w), fma2(bc2(ms.z), make_float2(sb.x, sb.y), make_float2(sb.z, sb.w))));
  const float2 B = fma2(bc2(mt.x), make_float2(ta.x, ta.y),
                        fma2(bc2(mt.y), make_float2(ta.z, ta.w), fma2(bc2(mt.z), make_float2(tb.x, tb.y), make_float2(tb.z, tb.w))));
  const float2 u = fma2(fma2(B, bc2(-1.f), A), bc2(1.f), bc2(ms.w));
  const float2 w = fma2(bc2(neg_four_beta2), B, bc2(mt.w));
  return fma2(u, u, w);
}

// the 32 pairs (row r, columns of one mask word) for the first RL of a thread's R rows; cs / ct: the word's 32
// pair-interleaved records
template <int RL, int R>
__device__ __forceinline__ void eval_word(const float4* __restrict__ cs, const float4* __restrict__ ct,
                                          const float4 (&ms)[R], const float4 (&mt)[R], const float two_beta2,
                                          const float beta4, uint32_t (&acc)[R], float (&mv)[R]) {
  (void)beta4;
  constexpr int kUnroll = K1_COLPAIR_UNROLL;
#pragma unroll kUnroll
  for (int q = 15; q >= 0; --q) {
    const float4 sa = cs[2 * q], sb = cs[2 * q + 1];
    const float4 ta = ct[2 * q], tb = ct[2 * q + 1];
#pragma unroll
    for (int r = 0; r < RL; ++r) {
      const float2 v = pair_fast2(ms[r], mt[r], sa, sb, ta, tb, two_beta2);
      acc[r] = __funnelshift_l(__float_as_uint(v.y), acc[r], 1);  // bit 2q + 1 <- sign(v), then bit 2q
      acc[r] = __funnelshift_l(__float_as_uint(v.x), acc[r], 1);
      mv[r] = fminf(mv[r], fminf(fabsf(v.x), fabsf(v.y)));
    }
  }
}

// A word that is only PARTLY live for some row of the warp -- the row's diagonal runs through it, or the arrays end
// inside it: the dead columns' values must not enter the row's running minimum (the self pair j = i alone has
// v = beta^4 <= t_fast: every row's diagonal word went down the slow path, N warp-cooperative redos per registration,
// a fifth of the kernel's instructions on N = 5000 problems).  live[r]: the row's live columns of this word.  Rare (two
// or three words per row): compact loop, not unrolled.
template <int R>
__device__ __forceinline__ void eval_word_masked(const float4* __restrict__ cs, const float4* __restrict__ ct,
                                              const float4 (&ms)[R], const float4 (&mt)[R], const float two_beta2,
                                              const uint32_t (&live)[R], uint32_t (&acc)[R], float (&mv)[R]) {
  uint32_t lv[R];
#pragma unroll
  for (int r = 0; r < R; ++r) lv[r] = live[r];
#pragma unroll 1
  for (int q = 15; q >= 0; --q) {
    const float4 sa = cs[2 * q], sb = cs[2 * q + 1];
    const float4 ta = ct[2 * q], tb = ct[2 * q + 1];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float2 v = pair_fast2(ms[r], mt[r], sa, sb, ta, tb, two_beta2);
      acc[r] = __funnelshift_l(__float_as_uint(v.y), acc[r], 1);
      acc[r] = __funnelshift_l(__float_as_uint(v.x), acc[r], 1);
      const float ay = (lv[r] & 0x80000000u) ? fabsf(v.y) : 3.0e38f;  // column 2q + 1
      const float ax = (lv[r] & 0x40000000u) ? fabsf(v.x) : 3.0e38f;  // column 2q
      mv[r] = fminf(mv[r], fminf(ax, ay));
      lv[r] <<= 2;
    }
  }
}

// Position (in units of 32 rows) of warp w's rows inside row group r of the CTA's row block.  Along the
// diagonal a warp's work in the tile where group r is partially live is 8 - pos words per tile, so the
// positions are permuted per group to give every warp (nearly) the same total over the diagonal tiles of a
// chunk: pos0 + pos1 = 7 for R <= 2, pos0 + pos1 + pos2 in {10, 11} for R >= 3 (identity positions leave
// warp 0 with 8 + 16 + 24 words against 1 + 9 + 17 for warp 7).
template <int R>
__device__ __forceinline__ int k1_warp_pos(int r, int w) {
  static_assert(K1_THREADS == 256, "the position tables are for 8 warps per CTA");
  if (r == 0) return w;
  if (R <= 2) return 7 - w;
  if (r == 1) return (w < 4 ? 7 : 14) - 2 * w;  // 7 5 3 1 6 4 2 0
  if (r == 2) return (w + 4) & 7;               // 4 5 6 7 0 1 2 3
  return 7 - ((w + 4) & 7);
}

// One CTA = a block of TI = 256 R rows x a chunk of `tiles_per_cta` column tiles (TJ columns each),
// starting at the tile that holds the diagonal of the row block; the column tiles stream through a
// K1_STAGES-deep shared-memory ring filled by 1-D TMA bulk copies.  Warps are not coupled by a CTA barrier:
// a warp waits for the "full" mbarrier of its next tile and arrives on the stage's "empty" mbarrier when it
// is done with it; thread 0 refills a stage once all eight warps have left it (with chunks of at most
// K1_STAGES tiles -- the cfg-A batches -- every tile is requested up front and nobody waits for anybody).
// Words that lie entirely below the diagonal inside a live tile are written
// as zeros; tiles entirely below it are not touched (callers that need them defined clear the mask
// first -- psulvsb_consistency_mask does, the engine never reads them).
template <int TJ>
struct K1Ring {
  static constexpr int STAGES = TJ <= 128 ? 8 : (TJ <= 256 ? 4 : 2);  // 32 KB of tiles per CTA
};

// SECT: every job's mask rows start on 32-byte sector boundaries and hold whole tiles (stride % 8 == 0: the engine's
// masks always do) -- a row's eight words of a tile are staged and leave as one sector; otherwise word by word.
template <int R, int TJ, bool SECT>
__global__ void __launch_bounds__(K1_THREADS, (R >= 4 ? K1_R4_CTAS : (R >= 2 ? 3 : 4)))
    k1_mask_kernel(const K1Job* __restrict__ jobs, int tiles_per_cta) {
  const K1Job& job = jobs[blockIdx.z];
  if (!job.active) return;
  const float4* __restrict__ src = job.src;
  const float4* __restrict__ dst = job.dst;
  const int n = job.n, row_begin = job.row_begin, row_end = job.row_end;
  const K1Consts c = job.c;
  uint32_t* __restrict__ mask = job.mask;
  const int stride = job.stride;
  uint32_t* __restrict__ row_counts = job.row_counts;
  unsigned long long* __restrict__ border_count = job.border;
  constexpr int TI = K1_THREADS * R;
  constexpr int WORDS = TJ / 32;
  constexpr int S = K1Ring<TJ>::STAGES;
  constexpr int NWARPS = K1_THREADS / 32;
  constexpr int kGroupSpan = (R == 4) ? 64 : 32;  // rows [grp_row_min[r], + kGroupSpan) hold the warp's rows of group r
  __shared__ __align__(128) float4 cs[S][TJ];
  __shared__ __align__(128) float4 ct[S][TJ];
  __shared__ __align__(8) uint64_t bar[S];        // "full": the tile's bytes have landed
  __shared__ __align__(8) uint64_t bar_empty[S];  // "empty": all warps are done with the stage
  __shared__ __align__(8) K1Slow slow;
  // a lane's words of the current tile, [WORDS][R][32] per warp: a row's WORDS words leave as ONE 32-byte sector
  // (two 16-byte stores) when the tile is done -- word-by-word stores touch a row's sector eight times, four bytes
  // at a time, and L2 fills the partial sectors from DRAM (ncu: 0.49 GB read per cfg-A batch by a kernel that reads
  // nothing but 160 KB of points per registration)
  extern __shared__ __align__(16) uint32_t k1_stage[];
  uint32_t* __restrict__ sw = k1_stage + (threadIdx.x >> 5) * (WORDS * R * 32) + (threadIdx.x & 31);
  static_assert(WORDS == 8, "a tile is one 32-byte sector per row");
  constexpr bool row_sectors = SECT;

  const int row0 = row_begin + blockIdx.y * TI;
  if (row0 >= row_end) return;  // grid is sized for the largest job
  const int n_tiles = (n + TJ - 1) / TJ;
  const int t_begin = row0 / TJ + blockIdx.x * tiles_per_cta;  // first live tile of the row block + chunk
  const int t_end = min(n_tiles, t_begin + tiles_per_cta);
  if (t_begin >= t_end) return;
  const int nt = t_end - t_begin;
  const int tid = threadIdx.x, lane = tid & 31;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
      mbar_init(&bar[s], 1);
      mbar_init(&bar_empty[s], NWARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    slow.c = c;
    slow.src64 = job.src64;
    slow.dst64 = job.dst64;
    slow.n = n;
  }
  // slots past the end of the arrays keep a finite dummy point; their bits are masked off below
  for (int k = tid; k < S * TJ; k += K1_THREADS) {
    (&cs[0][0])[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    (&ct[0][0])[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  auto issue = [&](int k) {  // thread 0: bulk copies of tile t_begin + k into stage k % S
    const int st = k % S;
    const int col0 = (t_begin + k) * TJ;
    const uint32_t bytes = (uint32_t)min(TJ, (int)il_records((size_t)n) - col0) * (uint32_t)sizeof(float4);  // whole column pairs
    // order the generic-proxy accesses of the stage's previous use before the async-proxy writes
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(&bar[st], 2 * bytes);
    tma_load_1d(cs[st], src + col0, bytes, &bar[st]);
    tma_load_1d(ct[st], dst + col0, bytes, &bar[st]);
  };
  if (tid == 0)
    for (int k = 0; k < S && k < nt; ++k) issue(k);

  // row points -> registers, pre-scaled by -2 for the norm form (overlaps the bulk copy)
  float4 ms[R], mt[R];
  int irow[R];
  int grp_row_min[R];  // smallest row of this warp in row group r (warp-uniform, increasing in r)
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if (R == 4) {
      // Two strips of 64 consecutive rows per warp, strip w and strip 15 - w of the block's 16: a lane's packed row
      // pairs (2 l, 2 l + 1) are neighbours, so both halves of an FFMA2 die together along the diagonal (with row
      // groups 256 apart, a half-live pair evaluated its dead row: half of the work in the diagonal tiles of an
      // N = 5000 problem, where they are a third of all tiles, was below the diagonal), and every warp owns the same
      // number of live words over the 4 diagonal tiles of its block (32 - 2 w + 2 + 2 w).
      const int strip = (r < 2) ? (tid >> 5) : 15 - (tid >> 5);
      grp_row_min[r] = row0 + 64 * strip;
      irow[r] = grp_row_min[r] + 2 * lane + (r & 1);
    } else {
      grp_row_min[r] = row0 + r * K1_THREADS + 32 * k1_warp_pos<R>(r, tid >> 5);
      irow[r] = grp_row_min[r] + lane;
    }
    const bool ok = irow[r] < row_end;
    const float4 a = ok ? il_load(src, irow[r]) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 b = ok ? il_load(dst, irow[r]) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float beta2 = 0.5f * c.two_beta2;
    ms[r] = make_float4(-2.f * a.x, -2.f * a.y, -2.f * a.z, (a.w - b.w) - beta2);        // .w = c1
    mt[r] = make_float4(-2.f * b.x, -2.f * b.y, -2.f * b.z, -2.f * c.two_beta2 * b.w);  // .w = c2
  }
  const float two_beta2 = -2.f * c.two_beta2, beta4 = c.beta4, t_fast = c.t_fast;  // (pair_fast takes -4 beta^2)
  const int warp_row_min = grp_row_min[0];  // smallest row this warp owns

  uint32_t cnt[R], row_ok[R];  // row_ok: all ones for a row inside [row_begin, row_end)
#pragma unroll
  for (int r = 0; r < R; ++r) {
    cnt[r] = 0;
    row_ok[r] = (irow[r] < row_end) ? 0xFFFFFFFFu : 0u;
  }
  unsigned int nborder = 0;

  for (int k = 0; k < nt; ++k) {
    const int st = k % S;
    if (tid == 0 && k >= 1 && k + S - 1 < nt) {  // refill the stage of tile k-1 once every warp has left it
      mbar_wait(&bar_empty[(k - 1) % S], ((k - 1) / S) & 1);
      issue(k + S - 1);
    }
    mbar_wait(&bar[st], (k / S) & 1);
    const int col0 = (t_begin + k) * TJ;
    for (int wj = 0; wj < WORDS; ++wj) {
      const int cb = col0 + wj * 32;  // first column of this word
      if (cb >= n) {  // past the last column: the rest of the row's sector is padding
        if (row_sectors) {
          for (int w2 = wj; w2 < WORDS; ++w2)
#pragma unroll
            for (int r = 0; r < R; ++r) sw[(w2 * R + r) * 32] = 0u;
        }
        break;
      }
      if (cb + 31 <= warp_row_min) {  // the word is below the diagonal for every row of this warp
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (row_sectors)
            sw[(wj * R + r) * 32] = 0u;
          else if (irow[r] < row_end)
            mask[(size_t)irow[r] * stride + (cb >> 5)] = 0u;
        }
        continue;
      }
      uint32_t acc[R];
      float mv[R];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        acc[r] = 0u;
        mv[r] = 3.0e38f;
      }
      // row group r of this warp still has live columns in this word iff cb + 31 > its smallest row; the
      // groups die in the order R-1, ..., 0 along the diagonal tiles (grp_row_min increases with r)
      int n_live = 1;
#pragma unroll
      for (int r = 1; r < R; ++r) n_live += (cb + 31 > grp_row_min[r]) ? 1 : 0;
      const float4* cw = &cs[st][wj * 32];
      const float4* tw = &ct[st][wj * 32];
      // partly live for some row of this warp (warp-uniform): the diagonal of one of its row groups runs through the
      // word, or the arrays end inside it
      bool partial = cb + 32 > n;
#pragma unroll
      for (int r = 0; r < R; ++r) partial = partial || (cb <= grp_row_min[r] + kGroupSpan - 1 && cb + 30 >= grp_row_min[r]);
      if (partial) {
        uint32_t lm[R];
        const uint32_t valid = (cb + 32 <= n) ? 0xFFFFFFFFu : ((1u << (n - cb)) - 1u);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int i = irow[r];
          const uint32_t upper = (i < cb) ? 0xFFFFFFFFu : ((i >= cb + 31) ? 0u : (0xFFFFFFFFu << (i - cb + 1)));
          lm[r] = (i < row_end) ? (valid & upper) : 0u;
        }
        eval_word_masked<R>(cw, tw, ms, mt, two_beta2, lm, acc, mv);
      } else if (n_live == R)
        eval_word<R, R>(cw, tw, ms, mt, two_beta2, beta4, acc, mv);
      else if (R == 4)  // (strips of adjacent rows: a pair is live or dead as a whole)
        eval_word<(R == 4 ? 2 : 1), R>(cw, tw, ms, mt, two_beta2, beta4, acc, mv);
      else if (R > 1 && n_live == 1)
        eval_word<1, R>(cw, tw, ms, mt, two_beta2, beta4, acc, mv);
      else if (R > 2 && n_live == 2)
        eval_word<(R > 2 ? 2 : 1), R>(cw, tw, ms, mt, two_beta2, beta4, acc, mv);
      else
        eval_word<(R > 3 ? 3 : 1), R>(cw, tw, ms, mt, two_beta2, beta4, acc, mv);
      // the word's epilogue.  FULL: every column of the word is right of every row of the CTA and inside the arrays (all
      // tiles but the block's diagonal ones and the last): no triangle / tail masks
      auto finish = [&](auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        const uint32_t valid = (FULL || cb + 32 <= n) ? 0xFFFFFFFFu : ((1u << (n - cb)) - 1u);
        uint32_t live[R], word[R];
        bool doubt = false;  // some pair of this lane's R words is one the fast path cannot vouch for
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const int i = irow[r];
          const uint32_t upper =
              (FULL || i < cb) ? 0xFFFFFFFFu : ((i >= cb + 31) ? 0u : (0xFFFFFFFFu << (i - cb + 1)));
          live[r] = FULL ? row_ok[r] : (row_ok[r] & valid & upper);
          word[r] = acc[r] & live[r];
          doubt = doubt || (live[r] != 0u && !(mv[r] > t_fast));
        }
        // rare (1.7 % of the words, but 4 in 10 warp steps see one): ONE vote decides whether the warp leaves the
        // fast lane at all; only then the per-row votes and the warp-cooperative redo
        if (__ballot_sync(0xffffffffu, doubt) != 0u) {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            unsigned int flagged = __ballot_sync(0xffffffffu, live[r] != 0u && !(mv[r] > t_fast));
            while (flagged) {
              const int owner = __ffs(flagged) - 1;
              flagged &= flagged - 1;
              const int oi = __shfl_sync(0xffffffffu, irow[r], owner);
              // the owner's row point back from its pre-scaled registers (x -2 and x -0.5 are exact)
              const float4 si = make_float4(-0.5f * __shfl_sync(0xffffffffu, ms[r].x, owner),
                                            -0.5f * __shfl_sync(0xffffffffu, ms[r].y, owner),
                                            -0.5f * __shfl_sync(0xffffffffu, ms[r].z, owner), 0.f);
              const float4 ti = make_float4(-0.5f * __shfl_sync(0xffffffffu, mt[r].x, owner),
                                            -0.5f * __shfl_sync(0xffffffffu, mt[r].y, owner),
                                            -0.5f * __shfl_sync(0xffffffffu, mt[r].z, owner), 0.f);
              // this lane's column of the word (read only here: the slow path is rare)
              const uint32_t res =
                  slow_word_coop(slow, oi, cb, si, ti, il_load(&cs[st][wj * 32], lane), il_load(&ct[st][wj * 32], lane), nborder);
              if (lane == owner) word[r] = res & live[r];
            }
          }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (row_sectors) {
            sw[(wj * R + r) * 32] = word[r];  // (rows past row_end hold zeros: live == 0)
          } else if (row_ok[r]) {
            mask[(size_t)irow[r] * stride + (cb >> 5)] = word[r];
          }
          cnt[r] += __popc(word[r]);  // (a row past row_end has word == 0)
        }
      };
      if (cb >= row0 + TI && cb + 32 <= n)
        finish(std::true_type());
      else
        finish(std::false_type());
    }
    if (row_sectors) {  // the tile's sector of every row (a lane reads back only what it staged itself)
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (irow[r] < row_end) {
          uint4 lo, hi;
          lo.x = sw[(0 * R + r) * 32];
          lo.y = sw[(1 * R + r) * 32];
          lo.z = sw[(2 * R + r) * 32];
          lo.w = sw[(3 * R + r) * 32];
          hi.x = sw[(4 * R + r) * 32];
          hi.y = sw[(5 * R + r) * 32];
          hi.z = sw[(6 * R + r) * 32];
          hi.w = sw[(7 * R + r) * 32];
          uint4* __restrict__ out = reinterpret_cast<uint4*>(mask + (size_t)irow[r] * stride + (col0 >> 5));
          out[0] = lo;
          out[1] = hi;
        }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&bar_empty[st]);  // this warp is done with stage st
  }
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (irow[r] < row_end && cnt[r] != 0u && row_counts) atomicAdd(&row_counts[irow[r]], cnt[r]);
  if (border_count) {
    unsigned int tot = (unsigned int)warp_sum_int((int)nborder);
    if ((tid & 31) == 0 && tot) atomicAdd(border_count, (unsigned long long)tot);
  }
}

// ------------------------------------------------------------------------------------------
__global__ void pack_points_kernel(const double* __restrict__ pts, int n, double cx, double cy, double cz,
                                   float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = pack_point(pts[3 * i] - cx, pts[3 * i + 1] - cy, pts[3 * i + 2] - cz);
}

// per-point float4 records (psulvsb_pack_points) -> the pair-interleaved records K1 reads (common.cuh il_store)
__global__ void interleave_points_kernel(const float4* __restrict__ in, int n, float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) il_store(out, i, in[i]);
  if (i == n && (n & 1)) il_store(out, n, make_float4(0.f, 0.f, 0.f, 0.f));
}

// mirror the upper triangle into the lower one: one warp per 32x32 bit block (bi >= bj)
__global__ void symmetrize_kernel(uint32_t* __restrict__ mask, int n, int stride, int nblk) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  // warp -> (bi, bj) with bj <= bi
  const long long total = (long long)nblk * (nblk + 1) / 2;
  if (warp >= total) return;
  int bi = (int)((sqrt(8.0 * (double)warp + 1.0) - 1.0) * 0.5);
  while ((long long)bi * (bi + 1) / 2 > warp) --bi;
  while ((long long)(bi + 1) * (bi + 2) / 2 <= warp) ++bi;
  const int bj = warp - (int)((long long)bi * (bi + 1) / 2);
  // source: rows of block bj, word bi
  const int jrow = bj * 32 + lane;
  const uint32_t s = (jrow < n) ? mask[(size_t)jrow * stride + bi] : 0u;
  uint32_t mine = 0u;
#pragma unroll
  for (int b = 0; b < 32; ++b) {
    const uint32_t t = __ballot_sync(0xffffffffu, (s >> b) & 1u);
    if (lane == b) mine = t;
  }
  const int irow = bi * 32 + lane;
  if (irow < n) {
    uint32_t* dstw = &mask[(size_t)irow * stride + bj];
    if (bi == bj)
      *dstw = *dstw | mine;
    else
      *dstw = mine;
  }
}

// exclusive scan of row_counts -> u64 offsets (one CTA per job; n <= a few 10^5)
__global__ void __launch_bounds__(1024) row_scan_kernel(const CompactJob* __restrict__ jobs) {
  const CompactJob& job = jobs[blockIdx.x];
  if (!job.active) return;
  const uint32_t* __restrict__ counts = job.row_counts;
  unsigned long long* __restrict__ offsets = job.offsets;
  const int n = job.n;
  __shared__ unsigned long long part[1024];
  const int tid = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int lo = min(n, tid * per), hi = min(n, lo + per);
  unsigned long long s = 0;
  for (int i = lo; i < hi; ++i) s += counts[i];
  part[tid] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    unsigned long long v = (tid >= off) ? part[tid - off] : 0ull;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  unsigned long long run = part[tid] - s;
  for (int i = lo; i < hi; ++i) {
    offsets[i] = run;
    run += counts[i];
  }
  if (tid == 1023) {
    offsets[n] = part[1023];
    if (job.n_edges) *job.n_edges = part[1023];
  }
}

// one warp per row: emit (i, j) for every set bit j > i, ascending j, at offsets[i], in edge format F
template <class F>
__global__ void compact_edges_kernel(const CompactJob* __restrict__ jobs) {
  const CompactJob& job = jobs[blockIdx.y];
  if (!job.active || !job.edges) return;
  const uint32_t* __restrict__ mask = job.mask;
  const int n = job.n, stride = job.stride;
  const unsigned long long cap = job.cap;
  void* __restrict__ edges = job.edges;
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  // the row's count, offset and first 32 mask words are loaded together, and each step loads the next 32 words before
  // it emits: a warp lives for a few steps, so exposed load latency, not bytes, bounded this pass
  const unsigned int count = job.row_counts ? job.row_counts[row] : 1u;
  const int W = (n + 31) >> 5;
  unsigned long long base = job.offsets[row];
  const uint32_t* __restrict__ mrow = mask + (size_t)row * stride;
  uint32_t next = (row >> 5) + lane < W ? mrow[(row >> 5) + lane] : 0u;
  if (count == 0u) return;  // nothing to emit (or a row another rank owns: its words are not this rank's)
  for (int w0 = row >> 5; w0 < W; w0 += 32) {
    const int w = w0 + lane;
    uint32_t word = next;
    next = (w + 32 < W) ? mrow[w + 32] : 0u;
    const int pc = __popc(word);
    int incl = pc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    unsigned long long pos = base + (unsigned long long)(incl - pc);
    while (word) {
      const int b = __ffs(word) - 1;
      word &= word - 1;
      if (pos < cap) F::store(edges, pos, (unsigned)row, (unsigned)(w * 32 + b));
      ++pos;
    }
    base += (unsigned long long)__shfl_sync(0xffffffffu, incl, 31);
  }
}

}  // namespace

K1Consts make_k1_consts(double beta, double coord_bound) {
  const double mu = 5.9604644775390625e-08;  // 2^-24
  const double cmax = coord_bound > beta ? coord_bound : beta;
  const double b2 = beta * beta;
  double cpad = b2 / 64.0;
  const double need = 32.0 * mu * (b2 + beta * cmax);
  if (need > cpad) cpad = need;
  const double cc = b2 + cpad;
  K1Consts k;
  k.half_bias = (float)(0.5 * cc);
  k.two_beta2 = (float)(2.0 * b2);
  k.r0 = (float)(2.0 * b2 * cc - b2 * b2);
  const double kappa = 384.0 * mu * beta * cmax;  // DESIGN.md "K1 error band": 353 mu beta Cmax, rounded up
  k.kappa = (float)(kappa * 1.0001);
  k.w_thr = (float)(kappa * cc * 1.01 + 1e-30);
  k.beta = beta;
  // fast (norm-form) path, DESIGN.md "K1 fast-path threshold"
  const double C2 = cmax * cmax;
  const double E = 80.0 * mu * C2;                 // |A_c - A*|, |B_c - B*|
  const double ED = 2.0 * E + 12.0 * mu * C2;      // |D_c - D*|
  const double ES = 2.0 * E + 24.0 * mu * C2;      // |S_c - S*|
  const double c0 = ED * ED + 2.0 * b2 * ES + 2.0 * mu * (48.0 * b2 * C2 + b2 * b2);
  const double Dlim = ED + sqrt(ED * ED + 48.0 * b2 * C2 + c0) + b2;  // (+ beta^2: the squared term is a - b - beta^2)
  const double Terr = 2.0 * Dlim * ED + c0;
  k.beta4 = (float)(b2 * b2);
  // a + b <= beta (where the sign of v is not the answer) implies S* <= beta^2, hence v* in
  // [-beta^4, 2 beta^4]: one threshold on |v| covers both the rounding band and that case
  k.t_fast = (float)((Terr + 2.0 * b2 * b2) * 1.05 + 1e-30);
  return k;
}

template <int R, int TJ, bool SECT>
static int launch_k1_variant(cudaStream_t st, const K1Job* d_jobs, int n_jobs, int max_n, int max_rows) {
  constexpr int TI = K1_THREADS * R;
  const int n_tiles = (max_n + TJ - 1) / TJ;
  const int row_blocks = (max_rows + TI - 1) / TI;
  // column tiles per CTA: long-lived CTAs amortise their prologue, but keep the grid many waves deep
  const double live_tiles = 0.55 * (double)n_tiles * row_blocks * n_jobs;
  int tpc = (int)(live_tiles / ((double)sm_count() * 3.0 * 12.0));  // ~12 waves of resident CTAs: short tail
  if (tpc < 1) tpc = 1;
  if (tpc > 16) tpc = 16;
  // whole diagonal blocks per chunk (TI / TJ tiles): the row permutation balances the warps over a block's diagonal tiles
  if (R == 4 && tpc >= 3) tpc = (tpc + 3) / 4 * 4;
  if (tpc > n_tiles) tpc = n_tiles;
  dim3 grid((n_tiles + tpc - 1) / tpc, row_blocks, n_jobs);
  // staging of the mask words: one 32-byte sector per row and tile (static + dynamic shared memory exceed 48 KB for R = 4)
  constexpr int stage_bytes = (K1_THREADS / 32) * (TJ / 32) * R * 32 * (int)sizeof(uint32_t);
  static bool attr_set = false;
  if (!attr_set) {
    PSU_CUDA(cudaFuncSetAttribute(k1_mask_kernel<R, TJ, SECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, stage_bytes));
    attr_set = true;
  }
  k1_mask_kernel<R, TJ, SECT><<<grid, K1_THREADS, stage_bytes, st>>>(d_jobs, tpc);
  PSU_CHECK_LAUNCH("k1_mask_kernel");
  return PSULVSB_OK;
}

int launch_consistency_mask(cudaStream_t st, const K1Job* d_jobs, int n_jobs, int max_n, int max_rows, bool row_sectors) {
  if (n_jobs <= 0 || max_n < 1 || max_rows < 1) return PSULVSB_OK;
  // rows per thread by the amount of work: R = 4 / 2 want enough row blocks x tiles to fill the GPU
  const double pairs = 0.5 * (double)max_rows * max_n * n_jobs;
  // measured on B200 (256-column tiles, dead row groups skipped): R = 4 wins once there is enough work
  // (N = 100k: 0.68-0.72 of the FP32-pipe peak vs 0.63; 256 x 5k-point problems: 0.59 vs 0.57; 64: 0.56 vs 0.55)
  int variant = pairs >= 5.0e8 ? 4 : (pairs >= 1.0e8 ? 2 : 1);
  if (debug_knobs().k1_variant >= 1 && debug_knobs().k1_variant <= 4) variant = debug_knobs().k1_variant;
  // 256-column tiles (measured: half the barrier stalls of 128-column tiles; 512 is no better)
  if (row_sectors) {
    if (variant == 3) return launch_k1_variant<3, 256, true>(st, d_jobs, n_jobs, max_n, max_rows);
    if (variant == 4) return launch_k1_variant<4, 256, true>(st, d_jobs, n_jobs, max_n, max_rows);
    if (variant == 2) return launch_k1_variant<2, 256, true>(st, d_jobs, n_jobs, max_n, max_rows);
    return launch_k1_variant<1, 256, true>(st, d_jobs, n_jobs, max_n, max_rows);
  }
  if (variant == 3) return launch_k1_variant<3, 256, false>(st, d_jobs, n_jobs, max_n, max_rows);
  if (variant == 4) return launch_k1_variant<4, 256, false>(st, d_jobs, n_jobs, max_n, max_rows);
  if (variant == 2) return launch_k1_variant<2, 256, false>(st, d_jobs, n_jobs, max_n, max_rows);
  return launch_k1_variant<1, 256, false>(st, d_jobs, n_jobs, max_n, max_rows);
}

int launch_pack_points(cudaStream_t st, const double* pts, int n, const double center[3], float4* out) {
  if (n <= 0) return PSULVSB_OK;
  const double cx = center ? center[0] : 0.0, cy = center ? center[1] : 0.0, cz = center ? center[2] : 0.0;
  pack_points_kernel<<<(n + 255) / 256, 256, 0, st>>>(pts, n, cx, cy, cz, out);
  PSU_CHECK_LAUNCH("pack_points_kernel");
  return PSULVSB_OK;
}

int launch_interleave_points(cudaStream_t st, const float4* in, int n, float4* out) {
  if (n <= 0) return PSULVSB_OK;
  interleave_points_kernel<<<(n + 1 + 255) / 256, 256, 0, st>>>(in, n, out);
  PSU_CHECK_LAUNCH("interleave_points_kernel");
  return PSULVSB_OK;
}

int launch_symmetrize(cudaStream_t st, uint32_t* mask, int n, int stride) {
  const int nblk = (n + 31) / 32;
  const long long warps = (long long)nblk * (nblk + 1) / 2;
  const long long threads = warps * 32;
  symmetrize_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(mask, n, stride, nblk);
  PSU_CHECK_LAUNCH("symmetrize_kernel");
  return PSULVSB_OK;
}

int launch_compact_edges(cudaStream_t st, const CompactJob* d_jobs, int n_jobs, int max_n, bool scan, bool emit,
                         bool narrow) {
  if (n_jobs <= 0 || max_n < 1) return PSULVSB_OK;
  if (scan) {
    row_scan_kernel<<<n_jobs, 1024, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("row_scan_kernel");
  }
  if (emit) {
    const long long threads = (long long)max_n * 32;
    dim3 grid((unsigned)((threads + 255) / 256), n_jobs);
    if (narrow)
      compact_edges_kernel<EdgeNarrow><<<grid, 256, 0, st>>>(d_jobs);
    else
      compact_edges_kernel<EdgeWide><<<grid, 256, 0, st>>>(d_jobs);
    PSU_CHECK_LAUNCH("compact_edges_kernel");
  }
  return PSULVSB_OK;
}

}  // namespace psulvsb
