// kin_umma.cuh -- the one inline-PTX layer over tcgen05 (UMMA), TMEM, mbarriers, named barriers and bulk copies for sm_100a.
// Every tensor-core kernel of the library takes its wrappers from here; the operand-format pieces of one flavour live next to
// their kernel (fp16: kin_tc16.cuh, tf32: kin_route_tc.cu).
//
// bf16 operand tiles are [rows][64 bf16] = 128-byte rows, SWIZZLE_128B (16-byte chunk c of row r lives at chunk c ^ (r & 7)),
// 1024-byte aligned.  The same tile serves as
//   * a K-major operand   (rows = M or N index, the 64 columns = K; one MMA consumes K = 16 = 32 bytes of every row), and
//   * an MN-major operand (rows = K index, the 64 columns = M or N; one MMA consumes 16 rows = two 1024-byte atoms),
// which is what lets the activation tiles written for the forward GEMMs feed the sample-reduction (weight-gradient) GEMMs
// without a transpose.  Both descriptor forms and the M = 64 TMEM lane map (row m -> lane m % 16 + 32 * (m / 16)) were
// checked on a B200 with tools/umma_mn_bf16_test.cu.
#pragma once

#include <cstdint>

namespace kin {
namespace umma {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// byte offset of 16-byte chunk `chunk` (8 bf16) of row `row` in a SWIZZLE_128B tile
__device__ __forceinline__ int sw_chunk(int row, int chunk) { return row * 128 + ((chunk ^ (row & 7)) << 4); }
// byte offset of element (row, col)
__device__ __forceinline__ int sw_elem(int row, int col) { return sw_chunk(row, col >> 3) + ((col & 7) << 1); }

// shared-memory descriptors: start >> 4 | LBO >> 4 << 16 | SBO >> 4 << 32 | version 1 << 46 | SWIZZLE_128B (2) << 61
__device__ __forceinline__ unsigned long long desc_k(unsigned saddr) {       // K-major: 8-row groups 1024 B apart
    return (unsigned long long)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ unsigned long long desc_mn(unsigned saddr) {      // MN-major: 8-row K groups 1024 B apart
    return (unsigned long long)((saddr >> 4) & 0x3FFFu) | (1024ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor, kind::f16: D fp32, A/B bf16; a_mn / b_mn select MN-major operands
__host__ __device__ constexpr unsigned idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (a_mn ? (1u << 15) : 0u) | (b_mn ? (1u << 16) : 0u) | ((unsigned)(N >> 3) << 17) |
           ((unsigned)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_bf16(unsigned tmem_d, unsigned long long da, unsigned long long db, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
// the same MMA with the A operand in tensor memory (lane = row, each 32-bit column = two consecutive K elements, 8 columns per K = 16
// step): the tensor core fetches only B from shared memory
__device__ __forceinline__ void mma_bf16_ts(unsigned tmem_d, unsigned a_taddr, unsigned long long db, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_taddr), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_tf32(unsigned tmem_d, unsigned long long da, unsigned long long db, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on the mbarrier once the MMAs this thread issued have completed
__device__ __forceinline__ void commit(unsigned mbar_saddr) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar_saddr) : "memory");
}

// one lane of a converged warp (the MMA issue is then compiled with uniform-register descriptors instead of per-MMA R2UR chains)
__device__ __forceinline__ bool elect_one() {
    unsigned pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0u;
}
// named barrier `id` over `threads` threads (a multiple of 32)
__device__ __forceinline__ void bar_sync(unsigned id, unsigned threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ void bar_arrive(unsigned id, unsigned threads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

// ---- mbarriers
__device__ __forceinline__ void mbar_init(unsigned saddr, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(saddr), "r"(count) : "memory");
}
// makes the mbarrier.init of this thread visible to the other threads and to the async proxy
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned saddr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(saddr) : "memory");
}
// arrive and announce `bytes` of bulk-copy transactions the phase must also wait for
__device__ __forceinline__ void mbar_expect_tx(unsigned saddr, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(saddr), "r"(bytes) : "memory");
}
// spins until the phase with `parity` has completed
__device__ __forceinline__ void mbar_wait(unsigned saddr, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\tWAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}"
        ::"r"(saddr), "r"(parity) : "memory");
}
// the same wait with a watchdog: a protocol bug traps (the launch fails with an error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait_or_trap(unsigned saddr, unsigned parity) {
    unsigned done = 0u;
    for (unsigned spins = 0u; ; ++spins) {
        asm volatile(
            "{\n\t.reg .pred P1;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, P1;\n\t}"
            : "=r"(done) : "r"(saddr), "r"(parity) : "memory");
        if (done) return;
        if (spins > (1u << 24)) __trap();   // each failed try_wait already suspends for a bounded time: >> seconds
    }
}
// non-blocking-ish probe: returns after at most ~`hint_ns` (the hardware suspends the warp meanwhile, no issue slots burnt)
__device__ __forceinline__ bool mbar_try_wait_hint(unsigned saddr, unsigned parity, unsigned hint_ns) {
    unsigned done;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}"
        : "=r"(done) : "r"(saddr), "r"(parity), "r"(hint_ns) : "memory");
    return done != 0u;
}
// non-blocking probe
__device__ __forceinline__ bool mbar_test_wait(unsigned saddr, unsigned parity) {
    unsigned done;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}"
        : "=r"(done) : "r"(saddr), "r"(parity) : "memory");
    return done != 0u;
}

// ---- fences between the generic proxy, the async proxy (tensor core, bulk copies) and thread synchronisation
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- bulk copies (TMA engine)
// global -> shared, completion counted on the mbarrier as `bytes` transactions
__device__ __forceinline__ void bulk_load(unsigned dst_saddr, const void* src, unsigned bytes, unsigned mbar_saddr) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_saddr), "l"(src), "r"(bytes), "r"(mbar_saddr) : "memory");
}
// shared -> global in this thread's current bulk group; bulk_commit closes the group, bulk_wait_read waits until every committed
// group has READ its shared-memory source (which may then be overwritten)
__device__ __forceinline__ void bulk_store(void* dst, unsigned src_saddr, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_saddr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ---- tensor memory
__device__ __forceinline__ void tmem_alloc(unsigned dst_saddr, unsigned cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_saddr), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(unsigned taddr, unsigned cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}

__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// this thread's 32 / 16 / 8 consecutive fp32 accumulator columns of its own TMEM lane, completed before returning
__device__ __forceinline__ void tmem_ld32(unsigned taddr, float* v) {
    unsigned r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(unsigned taddr, float* v) {
    unsigned r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(unsigned taddr, float* v) {
    unsigned r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr) : "memory");
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// split form: 16 raw accumulator words whose values are valid after tmem_wait16 on the same registers
__device__ __forceinline__ void tmem_ld16_raw(unsigned taddr, unsigned* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
// tcgen05.wait::ld with the loaded registers as in/out operands, so no consumer of them can be scheduled above the wait
__device__ __forceinline__ void tmem_wait16(unsigned* r) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :: "memory");
}

// 32-bit words -> consecutive columns of this thread's TMEM lane (an A operand for the _ts MMAs); tmem_st_wait completes them
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st4(unsigned taddr, unsigned a, unsigned b, unsigned c, unsigned d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void tmem_st8(unsigned taddr, const unsigned* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
// 16 words, completed before returning
__device__ __forceinline__ void tmem_st16(unsigned taddr, const unsigned* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
          "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
    tmem_st_wait();
}

// two floats -> packed bf16x2 (lo in bits 0..15), round to nearest even
__device__ __forceinline__ unsigned pack_bf16(float lo, float hi) {
    unsigned r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float bf16_lo(unsigned p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf16_hi(unsigned p) { return __uint_as_float(p & 0xffff0000u); }
// element (row, col) of a bf16 operand tile <- v rounded to bf16
__device__ __forceinline__ void st_bf16(unsigned char* tile, int row, int col, float v) {
    *reinterpret_cast<unsigned short*>(tile + sw_elem(row, col)) = (unsigned short)(pack_bf16(v, 0.0f) & 0xffffu);
}

__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

}  // namespace umma
}  // namespace kin
