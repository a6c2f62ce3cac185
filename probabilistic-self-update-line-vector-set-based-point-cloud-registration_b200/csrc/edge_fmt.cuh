// edge_fmt.cuh -- how the batch engine stores the reduced set (JobCtl::edges): one endpoint pair (i, j) per line vector.
//
// A registration whose working set (C plus the self-update head-room, i.e. Ccap) has at most 65 536 points stores an
// edge as ONE 32-bit word (i << 16) | j; larger ones keep a uint2.  The list is streamed whole by the compaction and by
// the L sample's flag pass, so its bytes are what those passes cost (DESIGN.md section 8).  The format is a property
// of the engine's arena only: the stage entry points of the C ABI, the sharded edge exchange and the lists handed to
// the GNC-TLS and clique kernels (JobCtl::basic_edges / pruned_edges) are uint2 always.
//
// Kernels that touch the list take the format as a template parameter (EdgeWide / EdgeNarrow); load() returns the
// pair unpacked, so the code behind it is the same for both.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace psulvsb {

struct EdgeWide {
  using T = uint2;
  __device__ __forceinline__ static uint2 load(const void* p, unsigned long long k) {
    return static_cast<const uint2*>(p)[k];
  }
  __device__ __forceinline__ static void store(void* p, unsigned long long k, unsigned int i, unsigned int j) {
    static_cast<uint2*>(p)[k] = make_uint2(i, j);
  }
};

struct EdgeNarrow {
  using T = uint32_t;
  __device__ __forceinline__ static uint2 load(const void* p, unsigned long long k) {
    const uint32_t e = static_cast<const uint32_t*>(p)[k];
    return make_uint2(e >> 16, e & 0xFFFFu);
  }
  __device__ __forceinline__ static void store(void* p, unsigned long long k, unsigned int i, unsigned int j) {
    static_cast<uint32_t*>(p)[k] = (i << 16) | j;
  }
};

constexpr long long kEdgeNarrowMaxPoints = 65536;  // point indices < 2^16

// the format of a registration whose working set holds at most ccap points
inline bool edge_narrow_fits(long long ccap) { return ccap <= kEdgeNarrowMaxPoints; }
inline size_t edge_bytes(bool narrow) { return narrow ? sizeof(EdgeNarrow::T) : sizeof(EdgeWide::T); }

}  // namespace psulvsb
