// Shared helpers for libb200ret.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "b200ret.h"

namespace b200 {

constexpr int kNumSMs = 148;   // B200: 2 dies x 74 SMs; grids are sized against the queried count at run time

void set_last_cuda_error(cudaError_t e, const char *where);
void count_launch(unsigned n = 1);
int sm_count();

#define B200_CUDA_TRY(expr)                                   \
    do {                                                      \
        cudaError_t _e = (expr);                              \
        if (_e != cudaSuccess) {                              \
            ::b200::set_last_cuda_error(_e, #expr);           \
            return B200_ERR_CUDA;                             \
        }                                                     \
    } while (0)

// after a <<<>>> launch: catches launch-configuration errors without synchronising
#define B200_LAUNCH_CHECK(name)                               \
    do {                                                      \
        ::b200::count_launch();                               \
        cudaError_t _e = cudaGetLastError();                  \
        if (_e != cudaSuccess) {                              \
            ::b200::set_last_cuda_error(_e, name);            \
            return B200_ERR_CUDA;                             \
        }                                                     \
    } while (0)

// Optional per-stage CUDA events of the calling thread (b200_hamming_map_stage_ms): off unless that entry point arms it.
struct StageMarks {
    static constexpr int kMax = 16;
    cudaEvent_t ev[kMax];
    const char *name[kMax];
    int n = 0;
    bool on = false;
};
StageMarks &stage_marks();
inline void stage_mark(const char *name, cudaStream_t st) {
    StageMarks &m = stage_marks();
    if (m.on && m.n < StageMarks::kMax) {
        m.name[m.n] = name;
        cudaEventRecord(m.ev[m.n++], st);
    }
}

inline cudaStream_t as_stream(b200_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename T>
__host__ __device__ constexpr T ceil_div(T a, T b) {
    return (a + b - 1) / b;
}
template <typename T>
__host__ __device__ constexpr T round_up(T a, T b) {
    return ceil_div(a, b) * b;
}

// ---- order-preserving float -> uint32 key of the k-NN selections: a larger key ranks first.  largest: larger floats get
// larger keys, else smaller floats do.  -0.0 folds into +0.0, so equal scores are ordered by index alone, and NaN gets
// key 0, the worst in either direction (no number maps to 0 or its complement).
__device__ __forceinline__ uint32_t rank_key(float f, bool largest) {
    if (f != f) return 0u;
    const uint32_t u = __float_as_uint(f + 0.f);          // -0.0 + 0.0 = +0.0 (IEEE, round to nearest)
    const uint32_t m = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return largest ? m : ~m;
}
// the score of a key (key 0: NaN; -0.0 comes back as +0.0)
__device__ __forceinline__ float rank_key_inv(uint32_t key, bool largest) {
    if (key == 0u) return __uint_as_float(0x7fffffffu);
    const uint32_t m = largest ? key : ~key;
    return __uint_as_float((m & 0x80000000u) ? (m & 0x7fffffffu) : ~m);
}

// ---- streaming global accesses (read-once inputs / write-once outputs must not pollute L1)
__device__ __forceinline__ uint4 ldg_stream_u4(const void *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_f4(float *p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void stg_stream_f2(float *p, float2 v) {
    asm volatile("st.global.cs.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}

// ---- mbarrier + 1-D bulk copy (TMA engine: cp.async.bulk, SASS UBLKCP)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// global -> shared, 16-byte aligned addresses, size multiple of 16; completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global bulk store (completion tracked by bulk async-groups)
__device__ __forceinline__ void bulk_s2g(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// make generic-proxy smem writes visible to the async proxy (before a bulk store reads them)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace b200
