// k2_sampler.cu -- stage 2: replayable sampling without replacement from a Philox stream.
//
// The reference draws `count` distinct indices with  do { r = rand() % n; } while (used[r]);
// (registration.cc:852-861, :916-932) -- inherently sequential, with a data-dependent number of
// consumed draws.  The same index sequence is produced in parallel here: draw k (a pure function
// of (seed, domain, event, k)) is accepted iff it is the FIRST occurrence of its value, i.e. iff
// first[v_k] == k where first[v] = min { k : v_k = v }; the r-th accepted draw is output r.
// That is exactly the rejection rule, so the output equals the sequential algorithm's for the same
// stream, and the stream position after the call (draws consumed) is reported for replay.
//
// Long value ranges (three buckets or more) first sort the draws by bucket: the draw kernel appends (k, v - lo) to
// its bucket's list (shared-memory histogram per 1024 draws, one global atomicAdd per bucket and step), so that a
// bucket CTA reads only its own ~max_draws / n_buckets draws instead of walking the whole window once per bucket
// (16 buckets on cfg-A: 10 MB -> 1.5 MB of L2 traffic per registration and sample).  The order inside a list is
// arbitrary, the result is not: first[v] is a minimum and the accept bits are indexed by k.
//
// Two passes, no global table:
//   bucket : the value range [0, n) is cut into buckets of SMP_BW values; CTA (b, job) walks the whole draw
//            window (Philox is cheap: the redundancy buys the removal of every random global access), keeps
//            first[v - lo] = min k for the values of ITS bucket in SHARED memory, and sets bit k of the
//            job's accept bitmask for every draw that is the first occurrence of its value.  The last
//            CTA of a job to finish turns the per-1024-draw popcounts into exclusive prefixes
//            (threadfence reduction, no CTA ever waits on another).
//   emit   : rank = prefix[chunk] + position in chunk -> out[rank]; clears the accept words on the way;
//            optional fused post-processing for the batch engine (endpoint flags / edge gather).
// Jobs whose values fit a shared-memory bitmap skip all of this: one CTA of the bucket launch walks their window in draw
// order (sample_onchip_walk).
// Kernels take device-resident SampleJob arrays (one job per registration in the batch engine,
// whose control kernels rewrite n / count / event between ticks).
#include <cstdlib>
#include <cuda_runtime.h>

#include "common.cuh"
#include "engine.cuh"

namespace psulvsb {

namespace {

constexpr int SMP_THREADS = 256;            // emit pass
constexpr int SMP_CHUNK = SMP_THREADS * 4;  // draws per chunk (one Philox block per thread)
constexpr int SMB_THREADS = 1024;           // bucket pass (one CTA per SM: the table fills shared memory)
constexpr int SMP_BW = 49152;               // values per bucket (192 KB of shared memory)
constexpr int SMP_MAX_LIST_BUCKETS = 512;   // bucket lists are used for 3 .. 512 buckets
constexpr int SMF_THREADS = 256;            // flag pass
constexpr int SMF_MAX_POINTS = 65536 * 8;   // flag pass: largest n_points marked in shared memory (a 64 KB bitmap)
constexpr int SMO_CHUNK = SMB_THREADS * 4;  // on-chip walk: draws per chunk (one Philox block per thread)
constexpr int SMO_HASH = 4096;              // on-chip walk: slots of the in-chunk duplicate table (expected chunk^2 / 2n values)
constexpr unsigned int SMO_LOSE_CAP = SMO_HASH / 2;  // losers per chunk the table takes (load <= 1/2); more: the warp walk
// on-chip budget: value bitmaps of up to 2^20 values (128 KB of shared memory) -- cfg-A's reduced sets (~6.9e5 edges +
// 65 536 of self-update head-room) qualify, cfg-B's (~2e7) do not.  Windows up to 2^20 draws: the rate pairs below
// (1.0, 1.0) need at most ~0.7 n.
constexpr unsigned long long SMO_MAX_N = 1ull << 20;
constexpr unsigned long long SMO_MAX_DRAWS = 1ull << 20;

// layout of the bucket lists for (n, max_draws).  An entry is ONE 32-bit word where that works, (k << w_bits) | (v - lo): the draw
// index takes the bits it needs and the rest addresses the value inside its bucket, so the bucket width shrinks
// from SMP_BW to a power of two when the draw window is long (2^17 draws -> 32 768 values per bucket).  n_buckets
// regions of cap_b entries (mean + 10 sigma + 64 of the uniform draws).  When that would take more than
// SMP_MAX_LIST_BUCKETS buckets, two-word entries (`wide`).  false: lists not applicable / scratch too small -> every
// bucket CTA walks the whole window.
struct ListPlan {
  unsigned int n_buckets, w_bits, width;
  unsigned int wide;  // 1: an entry is TWO words, (v - lo, k): long windows over long ranges (cfg-B: 2.3 M draws out of 2 * 10^7
                      // values), where k and a useful in-bucket offset do not fit one word; buckets of SMP_BW values
  unsigned long long cap_b;
};
__host__ __device__ inline unsigned long long list_cap_for(unsigned long long n, unsigned long long max_draws,
                                                          unsigned long long width) {
  const unsigned long long mean = (max_draws * width + n - 1) / n + 1;
  unsigned long long s = 1;
  while (s * s < mean) ++s;  // ceil(sqrt(mean)), integer: identical on host and device
  return (mean + 10 * s + 64 + 3) & ~3ull;
}
__host__ __device__ inline bool sample_list_plan(unsigned long long n, unsigned long long max_draws,
                                                 unsigned long long blist_cap, ListPlan& p) {
  p.n_buckets = 0;
  p.cap_b = 0;
  p.wide = 0;
  if (max_draws < 2 || n < 3ull * SMP_BW) return false;
  unsigned int k_bits = 1;
  while (((max_draws - 1) >> k_bits) != 0ull) ++k_bits;
  if (k_bits <= 24) {  // (narrower buckets than 256 values are not worth it)
    p.w_bits = 32u - k_bits;
    p.width = (p.w_bits >= 16u) ? (unsigned int)SMP_BW : (1u << p.w_bits);
    const unsigned long long nb = (n + p.width - 1) / p.width;
    if (nb >= 3 && nb <= (unsigned long long)SMP_MAX_LIST_BUCKETS) {
      p.n_buckets = (unsigned int)nb;
      p.cap_b = list_cap_for(n, max_draws, p.width);
      if (nb * p.cap_b <= blist_cap) return true;
    }
  }
  // two-word entries: k in full, buckets of SMP_BW values
  if (k_bits > 32) return false;
  p.w_bits = 32u;
  p.width = (unsigned int)SMP_BW;
  const unsigned long long nbw = (n + SMP_BW - 1) / SMP_BW;
  if (nbw < 3 || nbw > (unsigned long long)SMP_MAX_LIST_BUCKETS) {
    p.n_buckets = 0;
    p.cap_b = 0;
    return false;
  }
  p.n_buckets = (unsigned int)nbw;
  p.cap_b = list_cap_for(n, max_draws, p.width);
  p.wide = 1;
  return 2ull * nbw * p.cap_b <= blist_cap;
}
__device__ __forceinline__ uint32_t list_bucket(uint32_t v, const ListPlan& p) {
  return (p.w_bits >= 16u) ? v / (uint32_t)SMP_BW : v >> p.w_bits;  // (wide entries: w_bits = 32)
}

// (word >> 1) % n with the division replaced by a multiply-high: magic = ceil(2^64 / n) gives the exact
// quotient for every 31-bit dividend (the error term v e / 2^64 < 2^-33 cannot reach the next integer,
// which is at least 1/n > 2^-31 away)
struct FastMod {
  unsigned long long magic;
  uint32_t n;
};
__device__ __forceinline__ FastMod make_fastmod(uint32_t n) {
  FastMod f;
  f.n = n;
  f.magic = n > 1u ? (~0ull / n) + 1ull : 0ull;  // ceil(2^64 / n) (n = 1: everything maps to 0)
  return f;
}
__device__ __forceinline__ uint32_t draw_value(uint32_t word, const FastMod& f) {
  const uint32_t v = word >> 1;
  if (f.n <= 1u) return 0u;
  const uint32_t q = (uint32_t)__umul64hi((unsigned long long)v, f.magic);
  return v - q * f.n;
}

// On-chip path: jobs whose value bitmap fits shared memory (n <= onchip_n) and whose draw window is short are drawn by
// ONE CTA that walks the window in draw order, so "first occurrence" is a bit test against the values accepted so far
// and the rank is a running count.  The (1.0, 1.0) escalation (count = n: ~n (ln n + 10.6) draws) stays with the
// bucket passes, which spread its window over many CTAs.  Identity jobs keep the emit pass's handling.
__host__ __device__ inline bool sample_onchip(const SampleJob& job, unsigned long long onchip_n) {
  return job.n <= onchip_n && job.max_draws <= SMO_MAX_DRAWS && !job.identity && (job.post != 1 || job.vbits != nullptr);
}

__device__ __forceinline__ uint32_t philox_word(const Philox4& o, uint32_t l) {  // o.w[l] without local memory
  return l == 0u ? o.w[0] : l == 1u ? o.w[1] : l == 2u ? o.w[2] : o.w[3];
}

__device__ __forceinline__ uint32_t onchip_hash(uint32_t v) { return (v * 0x9E3779B1u) >> (32 - 12); }  // 12 = log2(SMO_HASH)

// The on-chip walk of one job by one CTA of the bucket launch.  Per chunk of SMO_CHUNK draws (thread t: Philox block
// k0/4 + t, draws k0 + 4t .. k0 + 4t + 3):
//   1. a draw whose value is already in `seen` (accepted in an earlier chunk) is rejected; the others are candidates
//   2. candidates claim their value with atomicOr.  A claim that finds the bit set lost to a draw of the same chunk and
//      enters the value in a small hash table (open addressing); every candidate whose value is in the table takes an
//      atomicMin of k there, only the minimum is accepted.  More than lose_cap losers (n not much larger than the
//      chunk) undo the chunk's claims -- every candidate's bit was clear before it -- and one warp walks the chunk in
//      k order instead.
//   3. block scan of the accepted draws -> ranks, out[rank] = v; accepted draws beyond `count` leave `seen` again.
// smem: [SMO_MAX_N / 32] bitmap words, then the table's [SMO_HASH] keys and [SMO_HASH] minima.
// lose_cap: SMO_LOSE_CAP, or (tests only) less, which forces the warp walk.
__device__ void sample_onchip_walk(const SampleJob& job, uint32_t* __restrict__ smem, unsigned int lose_cap) {
  constexpr uint32_t EMPTY = 0xFFFFFFFFu;  // (never a value: n < 2^31)
  uint32_t* seen = smem;
  uint32_t* hkey = smem + SMO_MAX_N / 32;
  uint32_t* hmin = hkey + SMO_HASH;
  __shared__ unsigned int n_lose_s;
  __shared__ unsigned int wsum[SMB_THREADS / 32];
  __shared__ uint32_t walk_acc[SMO_CHUNK / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const uint32_t n = (uint32_t)job.n;
  const uint32_t nwords = (n + 31u) >> 5;
  for (uint32_t i = tid; i < nwords; i += SMB_THREADS) seen[i] = 0u;
  for (int i = tid; i < SMO_HASH; i += SMB_THREADS) hkey[i] = EMPTY;
  if (job.post == 1)  // endpoint flags are rebuilt by the flag pass
    for (int i = tid; i < job.n_points; i += SMB_THREADS) job.flags[i] = 0;
  if (tid == 0) n_lose_s = 0u;
  const FastMod fm = make_fastmod(n);
  const uint64_t seed = job.seed;
  const uint32_t domain = job.domain, event = job.event;
  const uint32_t md = (uint32_t)job.max_draws, cnt = (uint32_t)job.count;  // (max_draws <= SMO_MAX_DRAWS)
  uint32_t* __restrict__ out = job.out;
  uint32_t taken = 0u;  // accepted draws of the earlier chunks (the same in every thread)
  __syncthreads();
  for (uint32_t k0 = 0u; k0 < md && taken < cnt; k0 += SMO_CHUNK) {
    const uint32_t kt = k0 + 4u * (uint32_t)tid;
    const Philox4 o = philox4x32_10(seed, domain, event, kt >> 2);
    uint32_t v[4];
    unsigned int acc = 0u;
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      v[l] = draw_value(o.w[l], fm);
      if (kt + l < md && !((seen[v[l] >> 5] >> (v[l] & 31u)) & 1u)) acc |= 1u << l;
    }
    __syncthreads();  // every test of the chunk saw only the earlier chunks' values
    int slot[4];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      slot[l] = -1;
      if ((acc >> l) & 1u) {
        const uint32_t bit = 1u << (v[l] & 31u);
        if ((atomicOr(&seen[v[l] >> 5], bit) & bit) && atomicAdd(&n_lose_s, 1u) < lose_cap) {
          uint32_t h = onchip_hash(v[l]);
          while (true) {
            const uint32_t old = atomicCAS(&hkey[h], EMPTY, v[l]);
            if (old == EMPTY) hmin[h] = 0xFFFFFFFFu;
            if (old == EMPTY || old == v[l]) break;
            h = (h + 1u) & (SMO_HASH - 1u);
          }
          slot[l] = (int)h;
        }
      }
    }
    __syncthreads();
    const unsigned int n_lose = n_lose_s;
    if (n_lose > lose_cap) {
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        if (slot[l] >= 0) hkey[slot[l]] = EMPTY;
        if ((acc >> l) & 1u) atomicAnd(&seen[v[l] >> 5], ~(1u << (v[l] & 31u)));
      }
      __syncthreads();
      if (wid == 0)
        for (uint32_t j = 0; j < (uint32_t)SMO_CHUNK; j += 32u) {
          const uint32_t k = k0 + j + lane;
          const uint32_t vk = draw_value(philox_word(philox4x32_10(seed, domain, event, k >> 2), k & 3u), fm);
          const bool c = k < md && !((seen[vk >> 5] >> (vk & 31u)) & 1u);
          const unsigned int peers = __match_any_sync(0xffffffffu, c ? vk : EMPTY);
          const bool first = c && (__ffs(peers) - 1) == lane;  // the lowest k of the value among the 32
          if (first) atomicOr(&seen[vk >> 5], 1u << (vk & 31u));
          const unsigned int b = __ballot_sync(0xffffffffu, first);
          if (lane == 0) walk_acc[j >> 5] = b;
          __syncwarp();
        }
      __syncthreads();
      acc = (walk_acc[(4u * tid) >> 5] >> ((4u * tid) & 31u)) & 0xFu;
    } else if (n_lose > 0u) {
#pragma unroll
      for (int l = 0; l < 4; ++l)
        if ((acc >> l) & 1u) {
          if (slot[l] < 0) {  // (a claim winner: is its value in the table?)
            uint32_t h = onchip_hash(v[l]);
            for (uint32_t key = hkey[h]; key != EMPTY; key = hkey[h]) {
              if (key == v[l]) {
                slot[l] = (int)h;
                break;
              }
              h = (h + 1u) & (SMO_HASH - 1u);
            }
          }
          if (slot[l] >= 0) atomicMin(&hmin[slot[l]], kt + l);
        }
      __syncthreads();
#pragma unroll
      for (int l = 0; l < 4; ++l)
        if (slot[l] >= 0) {
          if (hmin[slot[l]] != kt + l) acc &= ~(1u << l);
          hkey[slot[l]] = EMPTY;  // (every lookup of the chunk is done)
        }
    }
    // ranks: thread order is draw order
    const unsigned int c = __popc(acc);
    unsigned int incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    unsigned int wbase = 0u, total = 0u;
#pragma unroll
    for (int w = 0; w < SMB_THREADS / 32; ++w) {
      const unsigned int s = wsum[w];
      wbase += (w < wid) ? s : 0u;
      total += s;
    }
    if (tid == 0) n_lose_s = 0u;  // (every thread read it before the barrier above)
    uint32_t rank = taken + wbase + (incl - c);
#pragma unroll
    for (int l = 0; l < 4; ++l)
      if ((acc >> l) & 1u) {
        if (rank < cnt) {
          out[rank] = v[l];
          if (rank == cnt - 1u && job.status) job.status[0] = (unsigned long long)(kt + l) + 1ull;  // draws consumed
        } else {
          atomicAnd(&seen[v[l] >> 5], ~(1u << (v[l] & 31u)));  // a first occurrence beyond the sample
        }
        ++rank;
      }
    taken += total;
  }
  if (tid == 0 && taken < cnt && job.status) job.status[0] = 0ull;  // draw budget too small
  if (job.post == 1) {
    __syncthreads();
    for (uint32_t i = tid; i < nwords; i += SMB_THREADS) {  // the job's value bitmap for the flag pass, coalesced
      const uint32_t w = seen[i];
      if (w) job.vbits[i] = w;
    }
  }
}

// optional cache of the draw values (SampleJob::draws, one u32 per draw) so that the bucket CTAs stream
// them instead of re-running Philox; windows longer than draws_cap fall back to recomputation
// list_cap_test: 0, or (tests only) a smaller capacity the lists are filled to, which forces the overflow fallback
__global__ void __launch_bounds__(256) sample_draws_kernel(const SampleJob* __restrict__ jobs, unsigned int list_cap_test,
                                                           unsigned long long onchip_n) {
  const SampleJob& job = jobs[blockIdx.y];
  if (!job.active || job.identity || sample_onchip(job, onchip_n)) return;
  const bool cache = job.draws != nullptr && job.max_draws <= job.draws_cap;
  const unsigned long long nblocks = (job.max_draws + 3) >> 2;
  if ((unsigned long long)blockIdx.x * 256 >= nblocks) return;  // the grid is sized for the longest window of the batch
  __shared__ ListPlan plan_s;
  __shared__ FastMod fm_s;
  __shared__ int lists_s;
  if (threadIdx.x == 0) {  // (a 64-bit division and two short loops: once per CTA, not per thread)
    lists_s = (job.blist != nullptr && sample_list_plan(job.n, job.max_draws, job.blist_cap, plan_s)) ? 1 : 0;
    fm_s = make_fastmod((uint32_t)job.n);
  }
  __syncthreads();
  const ListPlan plan = plan_s;
  const bool lists = lists_s != 0;
  const unsigned int n_buckets = plan.n_buckets;
  const unsigned long long cap_b = plan.cap_b;  // region stride; cap_fill: how far a region may be filled
  const unsigned long long cap_fill = (list_cap_test != 0u && list_cap_test < plan.cap_b) ? list_cap_test : plan.cap_b;
  if (!cache && !lists) return;
  const FastMod fm = fm_s;
  uint4* __restrict__ out = reinterpret_cast<uint4*>(job.draws);
  if (!lists) {
    for (unsigned long long q = (unsigned long long)blockIdx.x * 256 + threadIdx.x; q < nblocks;
         q += (unsigned long long)gridDim.x * 256) {
      const Philox4 o = philox4x32_10(job.seed, job.domain, job.event, q);
      out[q] = make_uint4(draw_value(o.w[0], fm), draw_value(o.w[1], fm), draw_value(o.w[2], fm), draw_value(o.w[3], fm));
    }
    return;
  }
  constexpr int QPT = 4;  // Philox blocks per thread and step: 4096 draws share one round of barriers / global atomics
  // ranks inside a step without shared-memory atomics (a handful of buckets would serialise them): lanes of a warp
  // that hit the same bucket find each other with match.any, the warp keeps private running counts per bucket
  __shared__ unsigned int wh[8][SMP_MAX_LIST_BUCKETS];  // per warp: draws of the step that fell into each bucket
  __shared__ unsigned int base[SMP_MAX_LIST_BUCKETS];   // per bucket: reserved start in the global list
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned int lt_mask = (1u << lane) - 1u;
  const unsigned long long max_draws = job.max_draws;
  for (unsigned long long q0 = (unsigned long long)blockIdx.x * (256 * QPT); q0 < nblocks;
       q0 += (unsigned long long)gridDim.x * (256 * QPT)) {
    uint32_t vv[QPT][4];
    unsigned int rk[QPT][4];
    for (int b = lane; b < (int)n_buckets; b += 32) wh[wid][b] = 0u;
#pragma unroll
    for (int u = 0; u < QPT; ++u) {
      const unsigned long long q = q0 + (unsigned long long)u * 256 + tid;
#pragma unroll
      for (int l = 0; l < 4; ++l) vv[u][l] = 0xFFFFFFFFu;  // no draw
      if (q < nblocks) {
        const Philox4 o = philox4x32_10(job.seed, job.domain, job.event, q);
        uint32_t v4[4];
#pragma unroll
        for (int l = 0; l < 4; ++l) v4[l] = draw_value(o.w[l], fm);
        if (cache) out[q] = make_uint4(v4[0], v4[1], v4[2], v4[3]);  // (the emit pass reads the values back)
#pragma unroll
        for (int l = 0; l < 4; ++l)
          if ((q << 2) + l < max_draws) vv[u][l] = v4[l];
      }
    }
    __syncwarp();
#pragma unroll
    for (int u = 0; u < QPT; ++u)
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        const uint32_t b = (vv[u][l] != 0xFFFFFFFFu) ? list_bucket(vv[u][l], plan) : 0xFFFFFFFFu;
        const unsigned int peers = __match_any_sync(0xffffffffu, b);
        const int leader = __ffs(peers) - 1;
        unsigned int start = 0u;
        if (lane == leader && b != 0xFFFFFFFFu) {
          start = wh[wid][b];
          wh[wid][b] = start + __popc(peers);
        }
        start = __shfl_sync(0xffffffffu, start, leader);
        rk[u][l] = start + __popc(peers & lt_mask);
        __syncwarp();
      }
    __syncthreads();
    // per bucket: total of the step -> one global reservation; per warp: exclusive offset inside it
    for (int bk = tid; bk < (int)n_buckets; bk += 256) {
      unsigned int run = 0u;
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const unsigned int c = wh[w][bk];
        wh[w][bk] = run;
        run += c;
      }
      if (run != 0u) base[bk] = atomicAdd(&job.bcount[bk], run);
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < QPT; ++u) {
      const unsigned long long q = q0 + (unsigned long long)u * 256 + tid;
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        if (vv[u][l] == 0xFFFFFFFFu) continue;
        const uint32_t b = list_bucket(vv[u][l], plan);
        const unsigned long long pos = (unsigned long long)base[b] + wh[wid][b] + rk[u][l];
        if (pos < cap_fill) {
          if (plan.wide)
            reinterpret_cast<uint2*>(job.blist)[(unsigned long long)b * cap_b + pos] =
                make_uint2(vv[u][l] - b * plan.width, (uint32_t)((q << 2) + l));
          else
            job.blist[(unsigned long long)b * cap_b + pos] =
                (uint32_t)((((q << 2) + l) << plan.w_bits) | (unsigned long long)(vv[u][l] - b * plan.width));
        } else
          atomicExch(&job.bcount[SMP_MAX_LIST_BUCKETS], 1u);  // a list overflowed (10 sigma): the bucket pass walks instead
      }
    }
    __syncthreads();  // wh / base are rewritten by the next step
  }
}

__global__ void __launch_bounds__(SMB_THREADS, 1) sample_bucket_kernel(const SampleJob* __restrict__ jobs,
                                                                      unsigned long long onchip_n, unsigned int lose_cap) {
  const SampleJob& job = jobs[blockIdx.y];
  if (!job.active) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  if (sample_onchip(job, onchip_n)) {  // (same launch, no extra one: small registrations are bound by launches)
    if (blockIdx.x == 0) sample_onchip_walk(job, reinterpret_cast<uint32_t*>(smem_raw), lose_cap);
    return;
  }
  uint32_t* table = reinterpret_cast<uint32_t*>(smem_raw);  // [SMP_BW]
  uint32_t* wbm = table + SMP_BW;                            // [SMP_BW / 32] value bitmap of the current bucket
  __shared__ unsigned int ticket_s, sh[SMB_THREADS / 32];
  __shared__ unsigned long long carry_s;
  const int tid = threadIdx.x;
  if (job.post == 1 && blockIdx.x == 0)  // endpoint flags are rebuilt by the emit pass
    for (int i = tid; i < job.n_points; i += SMB_THREADS) job.flags[i] = 0;
  if (job.identity) return;
  const uint32_t n = (uint32_t)job.n;
  const FastMod fm = make_fastmod(n);
  ListPlan plan;
  const bool list_mode = job.blist != nullptr && sample_list_plan(job.n, job.max_draws, job.blist_cap, plan);
  const bool lists = list_mode && __ldcg(job.bcount + SMP_MAX_LIST_BUCKETS) == 0u;  // (no list overflowed)
  const unsigned int n_buckets = lists ? plan.n_buckets : (n + SMP_BW - 1) / SMP_BW;
  if (blockIdx.x >= n_buckets) return;
  const unsigned int n_workers = min(gridDim.x, n_buckets);  // CTAs of this job that take buckets (and a ticket)
  const unsigned long long max_draws = job.max_draws;
  const unsigned long long nblocks = (max_draws + 3) >> 2;
  const bool cached = job.draws != nullptr && max_draws <= job.draws_cap;
  const uint4* __restrict__ dv = reinterpret_cast<const uint4*>(job.draws);
  uint32_t* __restrict__ accept = job.first;  // bit k set <=> draw k is accepted; all zero on entry and on exit
  // post 1 with a value bitmap: bit v set <=> value v is in the sample; the flag pass streams the edge list by it
  uint32_t* __restrict__ vbits = (job.post == 1) ? job.vbits : nullptr;
  auto draws_of = [&](uint32_t q) -> uint4 {
    if (cached) return __ldcg(dv + q);
    const Philox4 o = philox4x32_10(job.seed, job.domain, job.event, q);
    return make_uint4(draw_value(o.w[0], fm), draw_value(o.w[1], fm), draw_value(o.w[2], fm), draw_value(o.w[3], fm));
  };
  if (lists && plan.wide) {
    // two-word entries (v - lo, k): read from the list in each of the three short walks (a bucket holds a few thousand)
    const uint2* __restrict__ lists2 = reinterpret_cast<const uint2*>(job.blist);
    for (uint32_t i = tid; i < plan.width; i += SMB_THREADS) table[i] = 0xFFFFFFFFu;
    for (unsigned int b = blockIdx.x; b < n_buckets; b += gridDim.x) {
      const uint2* __restrict__ list = lists2 + (unsigned long long)b * plan.cap_b;
      const uint32_t cnt = __ldcg(job.bcount + b);
      if (vbits)
        for (uint32_t i = tid; i < (plan.width >> 5); i += SMB_THREADS) wbm[i] = 0u;
      __syncthreads();  // the table is clean (initialisation / the previous bucket's third walk)
      for (uint32_t i = tid; i < cnt; i += SMB_THREADS) {
        const uint2 e = __ldcg(list + i);
        atomicMin(&table[e.x], e.y);
      }
      __syncthreads();
      const uint32_t lo_b = b * plan.width;
      for (uint32_t i = tid; i < cnt; i += SMB_THREADS) {
        const uint2 e = __ldcg(list + i);
        if (table[e.x] == e.y) {
          atomicOr(&accept[e.y >> 5], 1u << (e.y & 31));
          if (vbits) atomicOr(&wbm[e.x >> 5], 1u << (e.x & 31u));
        }
      }
      __syncthreads();
      if (vbits)
        for (uint32_t i = tid; i < (plan.width >> 5); i += SMB_THREADS)
          if (wbm[i] && ((unsigned long long)lo_b + 32ull * i) < job.n) vbits[(lo_b >> 5) + i] = wbm[i];
      for (uint32_t i = tid; i < cnt; i += SMB_THREADS) table[__ldcg(list + i).x] = 0xFFFFFFFFu;
      if (tid == 0) job.bcount[b] = 0u;  // zero on exit, like the accept bitmask
    }
  } else if (lists) {
    // every draw of bucket b sits in its list as (k << w_bits | v - lo).  A thread keeps its entries of the bucket in
    // registers for the three short walks (first occurrence, accept, clean the table) and already has the next
    // bucket's entries in flight while it works: one exposed HBM latency per CTA instead of three per bucket.
    const unsigned int wb = plan.w_bits, wmask = (1u << wb) - 1u;
    for (uint32_t i = tid; i < plan.width; i += SMB_THREADS) table[i] = 0xFFFFFFFFu;
    constexpr int EPT = 8;
    uint32_t cur[EPT], nxt[EPT];
    uint32_t cnt_cur = 0u, cnt_nxt = 0u;
    auto fetch = [&](unsigned int b, uint32_t (&e)[EPT], uint32_t& cnt) {
      const uint32_t* __restrict__ list = job.blist + (unsigned long long)b * plan.cap_b;
      cnt = __ldcg(job.bcount + b);
#pragma unroll
      for (int j = 0; j < EPT; ++j) {
        const uint32_t i = tid + j * SMB_THREADS;
        e[j] = (i < cnt) ? __ldcg(list + i) : 0u;
      }
    };
    unsigned int b = blockIdx.x;
    if (b < n_buckets) fetch(b, cur, cnt_cur);
    for (; b < n_buckets; b += gridDim.x) {
      const unsigned int bn = b + gridDim.x;
      if (bn < n_buckets) fetch(bn, nxt, cnt_nxt);
      const uint32_t* __restrict__ list = job.blist + (unsigned long long)b * plan.cap_b;
      if (vbits)
        for (uint32_t i = tid; i < (plan.width >> 5); i += SMB_THREADS) wbm[i] = 0u;
      __syncthreads();  // the table is clean (initialisation / the previous bucket's third walk)
#pragma unroll
      for (int j = 0; j < EPT; ++j)
        if (tid + j * SMB_THREADS < cnt_cur) atomicMin(&table[cur[j] & wmask], cur[j] >> wb);
      for (uint32_t i = tid + EPT * SMB_THREADS; i < cnt_cur; i += SMB_THREADS) {  // (lists longer than 8192 entries)
        const uint32_t e = __ldcg(list + i);
        atomicMin(&table[e & wmask], e >> wb);
      }
      __syncthreads();
      const uint32_t lo_b = b * plan.width;  // (vbits: which values were drawn; the emit pass removes the few beyond `count`)
#pragma unroll
      for (int j = 0; j < EPT; ++j)
        if (tid + j * SMB_THREADS < cnt_cur) {
          const uint32_t k = cur[j] >> wb;
          if (table[cur[j] & wmask] == k) {
            atomicOr(&accept[k >> 5], 1u << (k & 31));
            if (vbits) atomicOr(&wbm[(cur[j] & wmask) >> 5], 1u << (cur[j] & 31u));
          }
        }
      for (uint32_t i = tid + EPT * SMB_THREADS; i < cnt_cur; i += SMB_THREADS) {
        const uint32_t e = __ldcg(list + i);
        const uint32_t k = e >> wb;
        if (table[e & wmask] == k) {
          atomicOr(&accept[k >> 5], 1u << (k & 31));
          if (vbits) atomicOr(&wbm[(e & wmask) >> 5], 1u << (e & 31u));
        }
      }
      __syncthreads();
      if (vbits)  // the bucket's slice of the value bitmap, written once and coalesced (width is a multiple of 32)
        for (uint32_t i = tid; i < (plan.width >> 5); i += SMB_THREADS)
          if (wbm[i] && ((unsigned long long)lo_b + 32ull * i) < job.n) vbits[(lo_b >> 5) + i] = wbm[i];
#pragma unroll
      for (int j = 0; j < EPT; ++j)
        if (tid + j * SMB_THREADS < cnt_cur) table[cur[j] & wmask] = 0xFFFFFFFFu;
      for (uint32_t i = tid + EPT * SMB_THREADS; i < cnt_cur; i += SMB_THREADS) table[__ldcg(list + i) & wmask] = 0xFFFFFFFFu;
      if (tid == 0) job.bcount[b] = 0u;  // zero on exit, like the accept bitmask
#pragma unroll
      for (int j = 0; j < EPT; ++j) cur[j] = nxt[j];
      cnt_cur = cnt_nxt;
    }
  } else {
  if (list_mode && blockIdx.x == 0)  // a list overflowed: drop them all (zero on exit), walk the window instead
    for (int i = tid; i < SMP_MAX_LIST_BUCKETS; i += SMB_THREADS) job.bcount[i] = 0u;
  for (unsigned int b = blockIdx.x; b < n_buckets; b += gridDim.x) {
    const uint32_t lo = b * (uint32_t)SMP_BW;
    const uint32_t width = min((uint32_t)SMP_BW, n - lo);
    __syncthreads();  // the previous bucket's readers are done with the table
    for (uint32_t i = tid; i < width; i += SMB_THREADS) table[i] = 0xFFFFFFFFu;
    if (vbits)
      for (uint32_t i = tid; i < (uint32_t)(SMP_BW / 32); i += SMB_THREADS) wbm[i] = 0u;
    __syncthreads();
    // walk 1: first occurrence of every value of this bucket (four 16-byte loads in flight per thread:
    // the walk is bound by the latency of the cached draws coming from L2, not by arithmetic)
    const uint32_t nb32 = (uint32_t)nblocks, md32 = (uint32_t)max_draws;  // max_draws < 2^32 (launcher check)
    for (uint32_t q0 = tid; q0 < nb32; q0 += 4 * SMB_THREADS) {
      uint4 d4[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t q = q0 + u * SMB_THREADS;
        d4[u] = q < nb32 ? draws_of(q) : make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t q = q0 + u * SMB_THREADS;
        const uint32_t vv[4] = {d4[u].x, d4[u].y, d4[u].z, d4[u].w};
#pragma unroll
        for (int l = 0; l < 4; ++l) {
          const uint32_t k = (q << 2) + l;
          const uint32_t off = vv[l] - lo;  // 0xFFFFFFFF (no draw) never lands in the bucket: lo + width <= n < 2^31
          if (off < width && k < md32) atomicMin(&table[off], k);
        }
      }
    }
    __syncthreads();
    // walk 2: a draw is accepted iff it is that first occurrence (the cached draw values stream from L2, so
    // walking them twice is cheaper than remembering the matches behind a shared counter)
    for (uint32_t q0 = tid; q0 < nb32; q0 += 4 * SMB_THREADS) {
      uint4 d4[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t q = q0 + u * SMB_THREADS;
        d4[u] = q < nb32 ? draws_of(q) : make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t q = q0 + u * SMB_THREADS;
        const uint32_t vv[4] = {d4[u].x, d4[u].y, d4[u].z, d4[u].w};
        uint32_t bits = 0u;
#pragma unroll
        for (int l = 0; l < 4; ++l) {
          const uint32_t k = (q << 2) + l;
          const uint32_t off = vv[l] - lo;
          if (off < width && k < md32 && table[off] == k) {
            bits |= 1u << l;
            if (vbits) atomicOr(&wbm[off >> 5], 1u << (off & 31u));
          }
        }
        if (bits) atomicOr(&accept[q >> 3], bits << ((q & 7) << 2));
      }
    }
    if (vbits) {
      __syncthreads();
      for (uint32_t i = tid; i < ((width + 31u) >> 5); i += SMB_THREADS)
        if (wbm[i]) vbits[(lo >> 5) + i] = wbm[i];
    }
  }
  }
  // last CTA of this job: per-chunk popcounts of the accept bitmask -> exclusive prefixes
  __threadfence();
  __syncthreads();
  if (tid == 0) ticket_s = atomicAdd(job.ticket, 1u);
  __syncthreads();
  if (ticket_s != n_workers - 1) return;
  __threadfence();
  if (tid == 0) {
    carry_s = 0ull;
    *job.ticket = 0u;  // ready for the next use
    if (job.blist != nullptr) job.bcount[SMP_MAX_LIST_BUCKETS] = 0u;  // every CTA of the job has read the overflow flag
  }
  __syncthreads();
  const unsigned long long nchunks = (max_draws + SMP_CHUNK - 1) / SMP_CHUNK;
  constexpr int WPC = SMP_CHUNK / 32;  // accept words per chunk
  const unsigned long long nwords = (max_draws + 31) >> 5;
  for (unsigned long long c0 = 0; c0 < nchunks; c0 += SMB_THREADS) {
    const unsigned long long ch = c0 + tid;
    unsigned int v = 0;
    if (ch < nchunks)
      for (int w = 0; w < WPC; ++w) {
        const unsigned long long wi = ch * WPC + w;
        if (wi < nwords) v += __popc(__ldcg(accept + wi));
      }
    const int lane = tid & 31, wid = tid >> 5;
    unsigned int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) sh[wid] = incl;
    __syncthreads();
    unsigned int wbase = 0;
#pragma unroll
    for (int w = 0; w < SMB_THREADS / 32; ++w)
      if (w < wid) wbase += sh[w];
    const unsigned long long carry = carry_s;
    if (ch < nchunks) job.chunk_prefix[ch] = carry + wbase + (incl - v);
    __syncthreads();
    if (tid == SMB_THREADS - 1) carry_s = carry + wbase + incl;
    __syncthreads();
  }
  if (tid == 0 && carry_s < job.count && job.status) job.status[0] = 0ull;  // draw budget too small
}

// post 2: basic line vector `rank` of the sample (registration.cc:922-925) as an endpoint pair, v = out[rank]
template <class F>
__device__ __forceinline__ void gather_basic(const SampleJob& job, unsigned long long rank, uint32_t v) {
  const uint2 e = F::load(job.edges, job.via[v]);
  job.gathered[rank] = e;
  if (job.lv_out && rank < job.lv_cap) {
    // the line vector itself, formed here (many warps in flight hide the dependent gathers) instead of in
    // the prologue of the latency-bound GNC-TLS kernel; same operations as its load_lv8
    const double2* pa = reinterpret_cast<const double2*>(job.pts8 + 8 * (size_t)e.x);
    const double2* pb = reinterpret_cast<const double2*>(job.pts8 + 8 * (size_t)e.y);
    const double2 a0 = __ldg(pa), a1 = __ldg(pa + 1), a2 = __ldg(pa + 2);
    const double2 b0 = __ldg(pb), b1 = __ldg(pb + 1), b2 = __ldg(pb + 2);
    double* __restrict__ o = job.lv_out + rank;
    const size_t st = (size_t)job.lv_cap;
    __stcg(o, b0.x - a0.x);
    __stcg(o + st, b0.y - a0.y);
    __stcg(o + 2 * st, b1.x - a1.x);
    __stcg(o + 3 * st, b1.y - a1.y);
    __stcg(o + 4 * st, b2.x - a2.x);
    __stcg(o + 5 * st, b2.y - a2.y);
  }
}

template <class F>
__global__ void __launch_bounds__(SMP_THREADS) sample_emit_kernel(const SampleJob* __restrict__ jobs,
                                                                  unsigned long long onchip_n) {
  const SampleJob& job = jobs[blockIdx.y];
  if (!job.active) return;
  __shared__ unsigned int sh[SMP_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned long long count = job.count;
  uint32_t* __restrict__ out = job.out;
  if (sample_onchip(job, onchip_n)) {  // the on-chip pass placed out[]: the basic subset's gathers, indexed by rank
    if (job.post != 2 || (job.status && __ldcg(job.status) == 0ull)) return;  // (a failed sample has no full out[])
    for (unsigned long long r = (unsigned long long)blockIdx.x * SMP_THREADS + tid; r < count;
         r += (unsigned long long)gridDim.x * SMP_THREADS)
      gather_basic<F>(job, r, __ldcg(out + r));
    return;
  }
  if (job.identity) {  // registration.cc:839-847: the sample is the whole set, in order
    for (unsigned long long r = (unsigned long long)blockIdx.x * SMP_THREADS + tid; r < count;
         r += (unsigned long long)gridDim.x * SMP_THREADS) {
      out[r] = (uint32_t)r;
      if (job.post == 1) {
        const uint2 e = F::load(job.edges, r);
        job.flags[e.x] = 1;
        job.flags[e.y] = 1;
      } else if (job.post == 2) {
        job.gathered[r] = F::load(job.edges, job.via[r]);
      }
    }
    if (blockIdx.x == 0 && tid == 0 && job.status) job.status[0] = 1ull;  // nothing drawn; non-zero = success
    return;
  }
  const FastMod fm = make_fastmod((uint32_t)job.n);
  const unsigned long long max_draws = job.max_draws;
  const unsigned long long nchunks = (max_draws + SMP_CHUNK - 1) / SMP_CHUNK;
  const unsigned long long nwords = (max_draws + 31) >> 5;
  const bool cached = job.draws != nullptr && max_draws <= job.draws_cap;
  uint32_t* __restrict__ accept = job.first;
  for (unsigned long long ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const unsigned long long q = ch * SMP_THREADS + tid;  // Philox block: draws 4q .. 4q+3, bits of ONE accept word
    const unsigned long long wi = q >> 3;
    const uint32_t word = (wi < nwords) ? __ldcg(accept + wi) : 0u;
    const uint32_t bits = (word >> ((q & 7) << 2)) & 0xFu;
    const unsigned int c = __popc(bits);
    unsigned int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) sh[wid] = incl;
    __syncthreads();  // also: every thread of the chunk has read its accept word
    unsigned int wbase = 0;
#pragma unroll
    for (int w = 0; w < SMP_THREADS / 32; ++w)
      if (w < wid) wbase += sh[w];
    if ((q & 7) == 0 && wi < nwords && word != 0u) accept[wi] = 0u;  // leave the bitmask clear for the next use
    unsigned long long rank = job.chunk_prefix[ch] + wbase + (incl - c);
    if (bits) {
      uint32_t vv[4];
      if (cached) {
        const uint4 d4 = __ldcg(reinterpret_cast<const uint4*>(job.draws) + q);
        vv[0] = d4.x; vv[1] = d4.y; vv[2] = d4.z; vv[3] = d4.w;
      } else {
        const Philox4 o = philox4x32_10(job.seed, job.domain, job.event, q);
#pragma unroll
        for (int l = 0; l < 4; ++l) vv[l] = draw_value(o.w[l], fm);
      }
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        if ((bits >> l) & 1u) {
          if (rank < count) {
            const uint32_t v = vv[l];
            out[rank] = v;
            if (job.post == 1 && !job.vbits) {
              // src_sampled/dst_sampled = unique endpoints of the sampled line vectors
              // (registration.cc:870-894); only the SET matters downstream, kept as per-point flags
              const uint2 e = F::load(job.edges, v);
              job.flags[e.x] = 1;
              job.flags[e.y] = 1;
            } else if (job.post == 2) {
              gather_basic<F>(job, rank, v);
            }
            if (rank == count - 1 && job.status) job.status[0] = (q << 2) + l + 1;  // draws consumed
          } else if (job.post == 1 && job.vbits) {
            // a first occurrence beyond the count-th accepted draw: not part of the sample
            atomicAnd(&job.vbits[vv[l] >> 5], ~(1u << (vv[l] & 31u)));
          }
          ++rank;
        }
      }
    }
    __syncthreads();
  }
}

// post 1 with a value bitmap: endpoint flags of the sampled edges (registration.cc:870-894) by STREAMING the edge list in
// value order -- a lane takes one 32-value row at a time, skips the rows without a sampled value and reads the others
// coalesced -- instead of one random gather (a 64-byte HBM atom) per sampled edge.  Clears the bitmap.
// The endpoints are marked in a shared-memory bitmap of the job's points (n_points <= onchip_points, the bitmap's
// capacity; larger jobs store their flags directly): cfg-A marks ~30 endpoints per point, so each CTA then writes every marked point's flag
// once -- 16-byte stores where 16 neighbours are all marked -- instead of two scattered byte stores per sampled edge.
// Few CTAs per job keep that write-out small.  flags must be 16-byte aligned.
template <class F>
__global__ void __launch_bounds__(SMF_THREADS) sample_flag_kernel(const SampleJob* __restrict__ jobs, int onchip_points) {
  const SampleJob& job = jobs[blockIdx.y];
  if (!job.active || job.identity || job.post != 1 || !job.vbits) return;
  extern __shared__ uint32_t pbits[];  // [ceil(n_points / 32)] endpoint bitmap
  const int tid = threadIdx.x;
  const bool onchip = job.n_points <= onchip_points;
  const int pwords = (job.n_points + 31) >> 5;
  if (onchip) {
    for (int i = tid; i < pwords; i += SMF_THREADS) pbits[i] = 0u;
    __syncthreads();
  }
  uint8_t* __restrict__ flags = job.flags;
  auto mark = [&](uint32_t p) {
    if (!onchip) {
      flags[p] = 1;
      return;
    }
    const uint32_t bit = 1u << (p & 31u);
    if (!(pbits[p >> 5] & bit)) atomicOr(&pbits[p >> 5], bit);  // (most points are marked early on: a read, no atomic)
  };
  const unsigned long long nwords = (job.n + 31) >> 5;
  const unsigned long long threads = (unsigned long long)gridDim.x * SMF_THREADS;
  const void* __restrict__ edges = job.edges;
  // a lane owns one 32-value row (its bitmap word) per step and walks the set bits four at a time, loads first
  for (unsigned long long wi = (unsigned long long)blockIdx.x * SMF_THREADS + tid; wi < nwords; wi += threads) {
    uint32_t word = __ldcg(job.vbits + wi);
    if (!word) continue;
    job.vbits[wi] = 0u;  // zero on exit
    const unsigned long long row = wi * 32;
    while (word) {
      uint2 e[4];
      int m = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (word) {
          const int bit = __ffs(word) - 1;
          word &= word - 1;
          e[j] = F::load(edges, row + bit);
          m = j + 1;
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < m) {
          mark(e[j].x);
          mark(e[j].y);
        }
    }
  }
  if (!onchip) return;
  __syncthreads();
  // write-out: a lane takes 32 points (32 bytes of flags); only marked points are written (other CTAs of the job
  // write theirs, the bucket pass zeroed the flags)
  for (int w = tid; w < pwords; w += SMF_THREADS) {
    const uint32_t bits = pbits[w];
    if (!bits) continue;
    uint8_t* __restrict__ f = flags + 32 * (size_t)w;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t half = (bits >> (16 * h)) & 0xFFFFu;
      if (half == 0xFFFFu) {
        reinterpret_cast<uint4*>(f)[h] = make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
        continue;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t nib = (half >> (4 * q)) & 0xFu;
        uint8_t* __restrict__ g = f + 16 * h + 4 * q;
        if (nib == 0xFu)
          *reinterpret_cast<uint32_t*>(g) = 0x01010101u;
        else
#pragma unroll
          for (int l = 0; l < 4; ++l)
            if ((nib >> l) & 1u) g[l] = 1;
      }
    }
  }
}

__global__ void philox_fill_kernel(uint64_t seed, uint32_t domain, uint32_t event, unsigned long long first_k,
                                   unsigned long long count, uint32_t* __restrict__ out) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = philox_rand31(seed, domain, event, first_k + i);
}

}  // namespace

unsigned long long sample_default_max_draws(unsigned long long n, unsigned long long count) {
  return sample_max_draws_formula(n, count);
}

// entries of bucket-list scratch (SampleJob::blist) that make the lists usable for (n, max_draws); 0: not applicable
unsigned long long sample_list_entries(unsigned long long n, unsigned long long max_draws) {
  ListPlan p;
  if (!sample_list_plan(n, max_draws, ~0ull, p)) return 0;
  return (unsigned long long)p.n_buckets * p.cap_b * (p.wide ? 2ull : 1ull);  // in 32-bit words
}
unsigned long long sample_list_counters() { return SMP_MAX_LIST_BUCKETS + 4; }

unsigned long long sample_chunk_slots(unsigned long long max_draws) { return (max_draws + SMP_CHUNK - 1) / SMP_CHUNK + 1; }

// 32-bit words of the accept bitmask (SampleJob::first) a job with n values / max_draws draws needs
unsigned long long sample_table_words(unsigned long long n, unsigned long long max_draws) {
  (void)n;  // (it once was a per-value table)
  return (max_draws + 31) / 32 + 8;
}

bool sample_onchip_bound(unsigned long long n_bound) { return n_bound <= SMO_MAX_N; }

// n_bound: upper bound of SampleJob::n over the jobs (sizes the bucket grid, and selects the on-chip pass: every job
// of the launch whose n and window fit it is drawn there, the others by the bucket passes)
int launch_sample(cudaStream_t st, const SampleJob* d_jobs, int n_jobs, unsigned long long max_draws_bound,
                  unsigned long long n_bound, int flag_points, bool narrow) {
  if (n_jobs <= 0) return PSULVSB_OK;
  static bool attr_set = false;
  const size_t smem = (size_t)SMP_BW * 4 + (size_t)SMP_BW / 8;  // first-occurrence table + the bucket's value bitmap
  static_assert(SMO_MAX_N / 8 + 8 * SMO_HASH <= (size_t)SMP_BW * 4 + SMP_BW / 8, "the on-chip walk shares the bucket pass's shared memory");
  const int fsmem_max = SMF_MAX_POINTS / 8;
  if (!attr_set) {
    PSU_CUDA(cudaFuncSetAttribute(sample_bucket_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    PSU_CUDA(cudaFuncSetAttribute(sample_flag_kernel<EdgeWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, fsmem_max));
    PSU_CUDA(cudaFuncSetAttribute(sample_flag_kernel<EdgeNarrow>, cudaFuncAttributeMaxDynamicSharedMemorySize, fsmem_max));
    attr_set = true;
  }
  const unsigned long long nchunks = (max_draws_bound + SMP_CHUNK - 1) / SMP_CHUNK;
  unsigned long long gx = nchunks;
  const unsigned long long cap = (unsigned long long)(sm_count() * 16) / (unsigned long long)(n_jobs < 64 ? n_jobs : 64) + 1;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  const unsigned int list_cap_test = (unsigned int)debug_knobs().sample_list_cap_test;  // tests: list-overflow fallback
  const unsigned long long onchip_n = sample_onchip_bound(n_bound) ? n_bound : 0ull;
  const unsigned int lose_cap = (list_cap_test != 0u && list_cap_test < SMO_LOSE_CAP) ? list_cap_test : SMO_LOSE_CAP;
  sample_draws_kernel<<<dim3((unsigned)gx, (unsigned)n_jobs), 256, 0, st>>>(d_jobs, list_cap_test, onchip_n);
  PSU_CHECK_LAUNCH("sample_draws_kernel");
  // bucket CTAs: one per SM at a time; a CTA walks several buckets when the batch alone fills the GPU
  unsigned long long nb = (n_bound + SMP_BW - 1) / SMP_BW;
  if (nb < 1) nb = 1;
  unsigned long long bx = ((unsigned long long)sm_count() * 3ull + (unsigned long long)n_jobs - 1) / (unsigned long long)n_jobs;
  if (bx > nb) bx = nb;
  if (bx < 1) bx = 1;
  sample_bucket_kernel<<<dim3((unsigned)bx, (unsigned)n_jobs), SMB_THREADS, smem, st>>>(d_jobs, onchip_n, lose_cap);
  PSU_CHECK_LAUNCH("sample_bucket_kernel");
  if (narrow)
    sample_emit_kernel<EdgeNarrow><<<dim3((unsigned)gx, (unsigned)n_jobs), SMP_THREADS, 0, st>>>(d_jobs, onchip_n);
  else
    sample_emit_kernel<EdgeWide><<<dim3((unsigned)gx, (unsigned)n_jobs), SMP_THREADS, 0, st>>>(d_jobs, onchip_n);
  PSU_CHECK_LAUNCH("sample_emit_kernel");
  if (flag_points > 0) {
    // CTAs of 256 lanes x one 32-value row each.  Each writes out the flags of all points it marked (C / 16 stores when
    // they are dense), so a job gets a few CTAs, not hundreds: 8 per job at 296 jobs (measured on cfg-A: half as many
    // took 1.92 instead of 1.81 ms per step, the lanes over the list count for more than the write-out)
    unsigned long long fx = (n_bound + 32ull * SMF_THREADS - 1) / (32ull * SMF_THREADS);
    const unsigned long long fcap = ((unsigned long long)sm_count() * 16 + (unsigned long long)n_jobs - 1) / (unsigned long long)n_jobs;
    if (fx > fcap) fx = fcap;
    if (fx < 1) fx = 1;
    const int onchip_points = flag_points <= SMF_MAX_POINTS ? flag_points : 0;
    const size_t fsmem = (size_t)(onchip_points + 31) / 32 * 4;
    if (narrow)
      sample_flag_kernel<EdgeNarrow><<<dim3((unsigned)fx, (unsigned)n_jobs), SMF_THREADS, fsmem, st>>>(d_jobs, onchip_points);
    else
      sample_flag_kernel<EdgeWide><<<dim3((unsigned)fx, (unsigned)n_jobs), SMF_THREADS, fsmem, st>>>(d_jobs, onchip_points);
    PSU_CHECK_LAUNCH("sample_flag_kernel");
  }
  return PSULVSB_OK;
}

int launch_philox_fill(cudaStream_t st, uint64_t seed, uint32_t domain, uint32_t event, unsigned long long first_k,
                       unsigned long long count, uint32_t* out) {
  if (count == 0) return PSULVSB_OK;
  philox_fill_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(seed, domain, event, first_k, count, out);
  PSU_CHECK_LAUNCH("philox_fill_kernel");
  return PSULVSB_OK;
}

}  // namespace psulvsb
