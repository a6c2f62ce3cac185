// Host-side check of the reduced-set edge format rule (csrc/edge_fmt.cuh): which working-set sizes get 4-byte edges,
// the bytes per edge the engine's arena takes, and that packing keeps (i, j) and the row-major order.
#include <cstdio>
#include <cstdlib>

#include "edge_fmt.cuh"

using namespace psulvsb;

static int fails = 0;
#define CHECK(c)                                          \
  do {                                                    \
    if (!(c)) {                                           \
      std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #c); \
      ++fails;                                            \
    }                                                     \
  } while (0)

static uint32_t pack(uint32_t i, uint32_t j) { return (i << 16) | j; }

int main() {
  CHECK(edge_narrow_fits(1));
  CHECK(edge_narrow_fits(5000));
  CHECK(edge_narrow_fits(65535));
  CHECK(edge_narrow_fits(65536));
  CHECK(!edge_narrow_fits(65537));
  CHECK(!edge_narrow_fits(100000));
  CHECK(edge_bytes(true) == 4 && edge_bytes(false) == 8);
  CHECK(sizeof(EdgeNarrow::T) == 4 && sizeof(EdgeWide::T) == 8);
  // arena bytes of a cfg-A registration (6.3e5 edges): half of the 8-byte list
  const unsigned long long cap = 630000ull;
  CHECK(cap * edge_bytes(edge_narrow_fits(5000)) == 2520000ull);
  CHECK(cap * edge_bytes(edge_narrow_fits(100000)) == 5040000ull);
  // the largest indices survive, and row-major order (i, then j) is the order of the packed words
  CHECK((pack(65535, 65534) >> 16) == 65535u && (pack(65535, 65534) & 0xFFFFu) == 65534u);
  CHECK(pack(3, 65535) < pack(4, 0) && pack(4, 0) < pack(4, 1));
  if (fails) return 1;
  std::printf("edge format ok\n");
  return 0;
}
