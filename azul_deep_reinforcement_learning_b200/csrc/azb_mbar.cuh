// azb_mbar.cuh -- shared-memory mbarrier PTX wrappers (device only), used by the rotating rollout kernel (azb.cu) and the
// tensor-core kernels (azb_tc.cuh).  `bar` is a shared-window byte address.
#pragma once
#include <stdint.h>

namespace azb {

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// suspends the thread until the phase of the given parity has completed (try_wait: acquire at CTA scope)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
// one arrival (release at CTA scope): what the thread wrote before it is visible to the thread whose wait it completes
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

}  // namespace azb
