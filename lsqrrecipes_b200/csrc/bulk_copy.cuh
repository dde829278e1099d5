// Bulk global -> shared copies (cp.async.bulk, SASS UBLKCP) that complete on shared-memory mbarriers (SASS SYNCS), sm_90+ PTX,
// and the 2-deep tile ring of the tiled consensus kernels built from them.
#pragma once
#include <cstddef>
#include <cstdint>

namespace lsqr {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// makes the initialised barriers visible to the bulk-copy unit; the block synchronises before anyone else uses them
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// The 2-deep tile ring of the tiled consensus kernels: tiles [t0, t1) of the D rows soa[d * ld + t * TILE ...] pass through two
// shared-memory buffers (ring: 2 * D * TILE elements, bars: two mbarriers), one tile ahead of the readers.  Thread tid == 0
// initialises the barriers and issues one bulk copy per row.  Every thread of the block runs
//   ring.start();
//   for (uint32_t t = t0; t < t1; t++) { const T* tile = ring.wait(t); /* row d at tile[d * TILE] */ ring.release(); }
// and release() synchronises the block, so a buffer is refilled only when everyone is done with it.  restart() instead of start()
// walks the tiles once more.  (The loop stays with the
// caller: with the tile body in a lambda, ptxas allocates the fp64 kernel's registers differently.)
template <int D, int TILE, class T>
struct TileRing {
  static constexpr uint32_t kTileBytes = (uint32_t)(TILE * sizeof(T));
  const T* soa;
  size_t ld;
  uint32_t t0, t1;
  T* ring;
  uint64_t* bars;
  int tid;
  uint32_t phase0 = 0, phase1 = 0;

  __device__ __forceinline__ void issue(uint32_t t, int buf) {
    T* dst = buf ? ring + D * TILE : ring;
    mbar_expect_tx(&bars[buf], kTileBytes * D);
#pragma unroll
    for (int d = 0; d < D; d++) bulk_g2s(dst + d * TILE, soa + (size_t)d * ld + (size_t)t * TILE, kTileBytes, &bars[buf]);
  }
  __device__ __forceinline__ void start() {
    if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
    __syncthreads();
    if (tid == 0 && t0 < t1) issue(t0, 0);
  }
  // walks [t0, t1) again with the initialised barriers (their phases carry on); every thread has released the last tile
  __device__ __forceinline__ void restart() {
    if (tid == 0 && t0 < t1) issue(t0, 0);
  }
  // issues tile t + 1 into the other buffer, then waits for tile t
  __device__ __forceinline__ const T* wait(uint32_t t) {
    const int buf = (t - t0) & 1;
    if (tid == 0 && t + 1 < t1) issue(t + 1, buf ^ 1);
    if (buf) { mbar_wait(&bars[1], phase1); phase1 ^= 1; } else { mbar_wait(&bars[0], phase0); phase0 ^= 1; }
    return buf ? ring + D * TILE : ring;
  }
  __device__ __forceinline__ void release() { __syncthreads(); }
};

}  // namespace lsqr
