// mbar.cuh — split block barrier (arrive now, wait later) on a shared-memory mbarrier object.
// __syncthreads() makes every warp idle until the slowest one has published its values; with
// arrive / wait a thread signals "my values are published", keeps computing what does not need the
// neighbours, and only then waits — the barrier latency hides behind useful fp64 work.
#pragma once
#include <cstdint>

// the kernel's dynamic shared memory (the host emulator of tests/emu/ substitutes its own buffer)
#ifndef MARLPDE_DYN_SMEM
#define MARLPDE_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#endif

// kernel launch (the host emulator runs the blocks of the grid one after the other)
#ifdef MARLPDE_HOST_EMU
#define MARLPDE_LAUNCH(kernel, grid, block, smem, stream, ...) \
  ::simt::run_grid((int)(grid), (int)(block), (size_t)(smem), [&]() { kernel(__VA_ARGS__); })
#else
#define MARLPDE_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif

namespace marlpde {

#ifdef MARLPDE_HOST_EMU   // tests/emu/: kernel control logic on the host, test infrastructure only
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) { ::simt::mbar_init(bar, count); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { ::simt::mbar_arrive(bar); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) { ::simt::mbar_wait(bar, parity); }
#else
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// release semantics at CTA scope: shared-memory writes made before the arrive are visible after the wait
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  unsigned done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
#endif

}  // namespace marlpde
