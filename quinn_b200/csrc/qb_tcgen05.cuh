// The tcgen05 and mbarrier primitives that every tensor-core kernel is built from (qb_tc.cuh, qb_tc3.cuh, qb_tcg.cuh,
// qb_tg8.cuh), and the bounded mbarrier waits, which the layer-streamed path (qb_stream.cuh) uses as well.  Device code
// only.  These instructions are written out here and nowhere else, so a change to one of them reaches every path: compare
// the SASS of the whole library before and after.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t qb_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

#define QB_R16(v) "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), \
                  "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
#define QB_W16(v) "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), \
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
#define QB_RW16(v) "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), \
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])

// ---- tensor memory: this thread's lane, 16 or 8 consecutive 32-bit columns from taddr
__device__ __forceinline__ void qb_tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 :: "r"(taddr), QB_R16(v) : "memory");
}
__device__ __forceinline__ void qb_tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void qb_tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : QB_W16(v) : "r"(taddr) : "memory");
}
// the registers are operands of the wait so that no use of them can be scheduled before it
__device__ __forceinline__ void qb_tmem_ld_wait16(uint32_t (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" : QB_RW16(v) :: "memory");
}
__device__ __forceinline__ void qb_tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- fences: tcgen05 operations around a thread synchronisation; generic-proxy shared-memory writes before the tensor
// core (async proxy) reads them
__device__ __forceinline__ void qb_tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void qb_tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void qb_fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- mbarriers (shared-memory addresses)
__device__ __forceinline__ void qb_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void qb_mbar_inval(uint32_t bar) { asm volatile("mbarrier.inval.shared::cta.b64 [%0];" :: "r"(bar) : "memory"); }
// makes the initialisations above visible to the other threads and to the async proxy
__device__ __forceinline__ void qb_mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void qb_mbar_arrive(uint32_t bar) {
    asm volatile("{ .reg .b64 st; mbarrier.arrive.shared::cta.b64 st, [%0]; }" :: "r"(bar) : "memory");
}

// ---- bounded waits for phase `parity` of an mbarrier: a lost arrival traps instead of hanging the GPU.  try_wait with a
// suspend-time hint sleeps until the phase completes or the hint (20 us) expires; without one it returns at once.
// Timed: traps after 20 s of wall-clock time (%globaltimer, so that a context that is merely preempted or time-sliced for a
// while does not trip it).  HINT = false polls: the layer-streamed path's weight ring.
template <bool HINT = true>
__device__ __forceinline__ void qb_mbar_wait_timed(uint32_t bar, uint32_t parity) {
    unsigned long long t0 = 0;
    for (uint32_t it = 0;; ++it) {
        uint32_t ok;
        if constexpr (HINT)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.b32 %0, 1, 0, p; }"
                         : "=r"(ok) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
        else
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.b32 %0, 1, 0, p; }"
                         : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
        if ((it & 1023u) == 1023u) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 20000000000ULL) __trap();
        }
    }
}
// Counted, with the 20 us hint: 2^20 tries, then trap.  No state beyond its counter: the timed loop, inlined or called,
// made ptxas shuffle the live register arrays of the warp-specialised tile loops around it.
__device__ __forceinline__ void qb_mbar_wait_counted(uint32_t bar, uint32_t parity) {
#pragma unroll 1
    for (int it = 0; it < (1 << 20); ++it) {
        uint32_t ok;
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.b32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
        if (ok) return;
    }
    __trap();
}
// Counted spin, no hint: 2^28 polls, then trap.  For the fp16-split gradient kernel's issue warp, where every hand-over
// is on the critical path of the tile loop.
__device__ __forceinline__ void qb_mbar_spin(uint32_t bar, uint32_t parity) {
#pragma unroll 1
    for (int it = 0; it < (1 << 28); ++it) {
        uint32_t ok;
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.b32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();
}

// ---- tensor-memory allocation.  Start-up, all threads of the block: warp 0 allocates `cols` columns (their base address
// lands in the shared word at smem + slot_off) and gives up the allocation permit; thread 0 initialises the NB mbarriers
// at smem + bar_off[i] with arrival counts count[i] (QB_MBAR_BLOCK: one per thread of the block).  Returns the base
// address once both are visible to every thread.
enum : uint32_t { QB_MBAR_BLOCK = 0 };
template <int NB>
__device__ __forceinline__ uint32_t qb_tc_start(unsigned char* smem, uint32_t slot_off, uint32_t cols, const uint32_t (&bar_off)[NB],
                                                const uint32_t (&count)[NB]) {
    if ((threadIdx.x >> 5) == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(qb_smem_u32(smem + slot_off)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (threadIdx.x == 0) {
        const uint32_t b = qb_smem_u32(smem);
#pragma unroll
        for (int i = 0; i < NB; ++i) qb_mbar_init(b + bar_off[i], count[i] == QB_MBAR_BLOCK ? (uint32_t)blockDim.x : count[i]);
        qb_mbar_init_fence();
    }
    qb_tc_fence_before();
    __syncthreads();
    qb_tc_fence_after();
    return *reinterpret_cast<volatile uint32_t*>(smem + slot_off);
}
// thread 0, between two block barriers, once every phase of the previous evaluation has completed: the mbarriers at
// smem + bar_off[i] start again at parity 0, with arrival counts count[i]
template <int NB>
__device__ __forceinline__ void qb_mbar_reset(unsigned char* smem, const uint32_t (&bar_off)[NB], const uint32_t (&count)[NB]) {
    const uint32_t b = qb_smem_u32(smem);
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        qb_mbar_inval(b + bar_off[i]);
        qb_mbar_init(b + bar_off[i], count[i]);
    }
    qb_mbar_init_fence();
}
// all threads, at the end of the kernel: warp 0 frees the columns once every thread's tcgen05 operations are done
__device__ __forceinline__ void qb_tc_stop(uint32_t tmem, uint32_t cols) {
    qb_tc_fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(cols) : "memory");
}

// ---- MMA issue
__device__ __forceinline__ bool qb_elect() {
    uint32_t e;
    asm volatile("{ .reg .pred p; elect.sync _|p, 0xffffffff; selp.b32 %0, 1, 0, p; }" : "=r"(e) :: "memory");
    return e != 0;
}
// the mbarrier receives one arrival when every tcgen05 operation this thread issued before has completed
__device__ __forceinline__ void qb_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
// shared-memory matrix descriptor, as two 32-bit words: lo = start address and leading-dimension byte offset; hi = stride-
// dimension byte offset, the fixed version bit and the layout type (0: no swizzle, 1: 128-byte swizzle with 32-byte atoms)
__device__ __forceinline__ uint32_t qb_desc_lo(uint32_t saddr, uint32_t lbo) { return ((saddr >> 4) & 0x3FFFu) | ((lbo >> 4) << 16); }
__device__ __forceinline__ uint32_t qb_desc_hi(uint32_t sbo, uint32_t layout) { return (sbo >> 4) | (1u << 14) | (layout << 29); }

// One tcgen05.mma, issued by one thread: D (tensor memory at d) = A x B, plus D when the accumulate flag is set;
// kind::f16 (F16) or kind::tf32.  B is the shared-memory descriptor {b_lo, b_hi}; A is the descriptor {a_lo, a_hi} (_ss)
// or sits in tensor memory at a (_ts).  The flag is the register acc (!= 0: accumulate) or, where the issue loop knows
// it at compile time, the immediate ACC: ptxas schedules the two forms differently.
#define QB_MMA_SS(KIND, FLAG) asm volatile("{ .reg .pred p; .reg .b64 da, db; setp.ne.b32 p, %6, 0; mov.b64 da, {%1, %2}; " \
    "mov.b64 db, {%3, %4}; tcgen05.mma.cta_group::1.kind::" KIND " [%0], da, db, %5, p; }" \
    :: "r"(d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), FLAG : "memory")
#define QB_MMA_TS(KIND, FLAG) asm volatile("{ .reg .pred p; .reg .b64 db; setp.ne.b32 p, %5, 0; mov.b64 db, {%2, %3}; " \
    "tcgen05.mma.cta_group::1.kind::" KIND " [%0], [%1], db, %4, p; }" \
    :: "r"(d), "r"(a), "r"(b_lo), "r"(b_hi), "r"(idesc), FLAG : "memory")
template <bool F16>
__device__ __forceinline__ void qb_mma_ss(uint32_t d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                          uint32_t acc) {
    if constexpr (F16) QB_MMA_SS("f16", "r"(acc)); else QB_MMA_SS("tf32", "r"(acc));
}
template <bool F16, bool ACC>
__device__ __forceinline__ void qb_mma_ss(uint32_t d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc) {
    if constexpr (F16) QB_MMA_SS("f16", "n"(ACC ? 1 : 0)); else QB_MMA_SS("tf32", "n"(ACC ? 1 : 0));
}
template <bool F16>
__device__ __forceinline__ void qb_mma_ts(uint32_t d, uint32_t a, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t acc) {
    if constexpr (F16) QB_MMA_TS("f16", "r"(acc)); else QB_MMA_TS("tf32", "r"(acc));
}
template <bool F16, bool ACC>
__device__ __forceinline__ void qb_mma_ts(uint32_t d, uint32_t a, uint32_t b_lo, uint32_t b_hi, uint32_t idesc) {
    if constexpr (F16) QB_MMA_TS("f16", "n"(ACC ? 1 : 0)); else QB_MMA_TS("tf32", "n"(ACC ? 1 : 0));
}
#undef QB_MMA_SS
#undef QB_MMA_TS

// ---- fp16 hi / lo operand splits (kind::f16 "3 x FP16" products)
__device__ __forceinline__ uint32_t qb_pack_f16(float lo_elem, float hi_elem) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_elem), "f"(lo_elem));
    return r;
}
// (x0, x1) -> fp16 pair `hi` (round to nearest) and the fp16 pair of the NEGATED remainders hi - x (the mixed-precision
// subtract takes the fp16 operand first; the sign is absorbed by a negated copy of the other operand's hi tile)
__device__ __forceinline__ void qb_split_f16_nlo(float x0, float x1, uint32_t& hi, uint32_t& nlo) {
    hi = qb_pack_f16(x0, x1);
    float d0, d1;       // hi - x, exactly: one instruction per element
    asm("{ .reg .b16 a, b; mov.b32 {a, b}, %2; sub.rn.f32.f16 %0, a, %3; sub.rn.f32.f16 %1, b, %4; }"
        : "=f"(d0), "=f"(d1) : "r"(hi), "f"(x0), "f"(x1));
    nlo = qb_pack_f16(d0, d1);
}
// the same with the remainders lo = x - hi
__device__ __forceinline__ void qb_split_f16(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    uint32_t nlo;
    qb_split_f16_nlo(x0, x1, hi, nlo);
    lo = nlo ^ 0x80008000u;
}
#endif  // __CUDACC__
