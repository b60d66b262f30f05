// JPEG decoding on the device (b200_jpeg_decode_u8): Image.open(f).convert("RGB") of Pillow on every file of a ragged
// batch, bit for bit.  The per-sample arithmetic lives in jpeg_core.cuh, the planner in jpeg_plan.h; three launches:
//
//   1. jpeg_entropy_kernel (cooperative): the self-synchronising parallel Huffman decode of Weissenberger & Schmidt
//      ("Accelerating JPEG Decompression on GPUs", 2021).  Every restart interval (the whole scan without restarts) is
//      cut into subsequences of kJpegSubBits bits.  Each subsequence is decoded speculatively from an assumed state
//      (bit position, block of the MCU, coefficient index) to the first symbol boundary past its end; the state found
//      there becomes the next subsequence's entry, which is decoded again when it changed; rounds repeat until every
//      entry equals its predecessor's exit.  The first subsequence of an interval starts in its true state and equality
//      is exact, so at that point every entry is the sequential decoder's.  A grid-wide exclusive scan of each
//      subsequence's block count and per-component DC differences then gives each subsequence its first block and its DC
//      predictors (differences restart at interval boundaries: the prefix at the interval's first subsequence is
//      subtracted), and a last decode stores the dezigzagged int16 coefficients, DC absolute, into per-component planes.
//   2. jpeg_idct_kernel: dequantisation + islow IDCT, 8 threads per block (a column each, then a row each), into
//      per-component uint8 sample planes.
//   3. jpeg_color_kernel: one thread per output pixel: fancy upsampling of the chroma, YCbCr -> RGB, interleaved into the
//      ragged HWC output; pixels of worker-decoded images are copied.
#include <cooperative_groups.h>

#include <vector>

#include "common.cuh"
#include "jpeg_plan.h"

namespace cg = cooperative_groups;

namespace b200 {

__global__ void __launch_bounds__(kJpegThreads, 1) jpeg_entropy_kernel(const JpegArgs a, unsigned *head, unsigned *cta_tot) {
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned s_scan[kJpegThreads][4];
    __shared__ unsigned s_red[4];
    const long long threads = static_cast<long long>(gridDim.x) * kJpegThreads;
    const long long tid = static_cast<long long>(blockIdx.x) * kJpegThreads + threadIdx.x;
    const long long per = (a.n_sub + threads - 1) / threads;
    const long long i0 = tid * per < a.n_sub ? tid * per : a.n_sub, i1 = i0 + per < a.n_sub ? i0 + per : a.n_sub;
    for (long long i = i0; i < i1; ++i) jpeg_sub_init(a, i);
    unsigned round = 0;
    for (;;) {
        for (long long i = i0; i < i1; ++i) jpeg_sub_speculate(a, i);
        grid.sync();
        bool changed = false;
        for (long long i = i0; i < i1; ++i) changed |= jpeg_sub_sync(a, i);
        if (changed) *reinterpret_cast<volatile unsigned *>(head + 1) = round + 1;
        grid.sync();
        ++round;
        if (*reinterpret_cast<volatile unsigned *>(head + 1) != round) break;
    }
    if (tid == 0) head[0] = round;
    // exclusive scan of the sums over all subsequences: thread totals, CTA scan, CTA totals, then the prefix in place
    unsigned loc[4] = {0, 0, 0, 0};
    for (long long i = i0; i < i1; ++i)
        for (int j = 0; j < 4; ++j) loc[j] += a.sums[4 * i + j];
    for (int j = 0; j < 4; ++j) s_scan[threadIdx.x][j] = loc[j];
    __syncthreads();
    for (int d = 1; d < kJpegThreads; d <<= 1) {
        unsigned v[4] = {0, 0, 0, 0};
        if (static_cast<int>(threadIdx.x) >= d)
            for (int j = 0; j < 4; ++j) v[j] = s_scan[threadIdx.x - d][j];
        __syncthreads();
        for (int j = 0; j < 4; ++j) s_scan[threadIdx.x][j] += v[j];
        __syncthreads();
    }
    if (threadIdx.x == kJpegThreads - 1)
        for (int j = 0; j < 4; ++j) cta_tot[4 * blockIdx.x + j] = s_scan[threadIdx.x][j];
    grid.sync();
    if (threadIdx.x < 4) s_red[threadIdx.x] = 0;
    __syncthreads();
    for (unsigned b = threadIdx.x; b < blockIdx.x; b += kJpegThreads)
        for (int j = 0; j < 4; ++j) atomicAdd(&s_red[j], __ldcg(cta_tot + 4 * b + j));
    __syncthreads();
    unsigned run[4];
    for (int j = 0; j < 4; ++j) run[j] = s_red[j] + s_scan[threadIdx.x][j] - loc[j];
    for (long long i = i0; i < i1; ++i)
        for (int j = 0; j < 4; ++j) {
            const unsigned t = a.sums[4 * i + j];
            a.sums[4 * i + j] = run[j];
            run[j] += t;
        }
    grid.sync();
    for (long long i = i0; i < i1; ++i) jpeg_sub_write(a, i);
}

constexpr int kJpegIdctBlocks = kJpegThreads / 8;

__global__ void __launch_bounds__(kJpegThreads) jpeg_idct_kernel(const JpegArgs a) {
    __shared__ int ws[kJpegIdctBlocks][64];
    const int slot = threadIdx.x >> 3, t = threadIdx.x & 7;
    const long long g = static_cast<long long>(blockIdx.x) * kJpegIdctBlocks + slot;
    JpegBlockRef r{};
    if (g < a.n_blocks) {
        r = jpeg_block(a, g);
        jpeg_idct_col(r.coef, r.q, t, ws[slot]);
    }
    __syncthreads();
    if (g < a.n_blocks) {
        uint8_t o[8];
        jpeg_idct_row(ws[slot], t, o);
        uint2 v;
        v.x = o[0] | (o[1] << 8) | (o[2] << 16) | (static_cast<unsigned>(o[3]) << 24);
        v.y = o[4] | (o[5] << 8) | (o[6] << 16) | (static_cast<unsigned>(o[7]) << 24);
        *reinterpret_cast<uint2 *>(r.dst + static_cast<size_t>(t) * r.pitch) = v;
    }
}

__global__ void __launch_bounds__(kJpegThreads) jpeg_color_kernel(const JpegArgs a) {
    const long long p = static_cast<long long>(blockIdx.x) * kJpegThreads + threadIdx.x;
    if (p < a.n_pix) jpeg_out_pixel(a, p);
}

static int jpeg_coop_ctas(long long n_sub) {
    static int per_sm = -1;
    if (per_sm < 0) {
        int v = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, jpeg_entropy_kernel, kJpegThreads, 0) != cudaSuccess) return -1;
        per_sm = v;
    }
    long long ctas = static_cast<long long>(per_sm) * sm_count();
    const long long need = (n_sub + kJpegThreads - 1) / kJpegThreads;
    if (ctas > need) ctas = need;
    if (ctas > kJpegMaxCtas) ctas = kJpegMaxCtas;
    return static_cast<int>(ctas < 1 ? 1 : ctas);
}

}  // namespace b200

using namespace b200;

extern "C" {

size_t b200_jpeg_decode_workspace_bytes(const b200_jpeg_desc *desc_host, const void *tables_host, size_t tables_bytes, int n) {
    JpegPlan p;
    if (n < 1 || jpeg_plan(desc_host, static_cast<const unsigned char *>(tables_host), tables_bytes, n, nullptr, kJpegSubBits, p) != B200_OK)
        return 0;
    return p.bytes;
}

int b200_jpeg_decode_u8(const uint8_t *in, const b200_jpeg_desc *desc_host, const void *tables_host, size_t tables_bytes, int n,
                        uint8_t *out, const long long *out_offsets_host, void *workspace, size_t workspace_bytes,
                        b200_stream_t stream) {
    if (n < 0) return B200_ERR_INVALID_ARG;
    if (n == 0) return B200_OK;
    if (!in || !out || !out_offsets_host) return B200_ERR_INVALID_ARG;
    const unsigned char *tables = static_cast<const unsigned char *>(tables_host);
    JpegPlan p;
    const int rc = jpeg_plan(desc_host, tables, tables_bytes, n, out_offsets_host, kJpegSubBits, p);
    if (rc != B200_OK) return rc;
    if (!workspace || workspace_bytes < p.bytes) return B200_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return B200_ERR_ALIGNMENT;
    std::vector<unsigned char> stage;
    jpeg_stage(p, tables, tables_bytes, stage);
    cudaStream_t st = as_stream(stream);
    uint8_t *ws = static_cast<uint8_t *>(workspace);
    const int ctas = p.n_sub ? jpeg_coop_ctas(p.n_sub) : 0;
    if (ctas < 0) {
        set_last_cuda_error(cudaGetLastError(), "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
        return B200_ERR_CUDA;
    }
    B200_CUDA_TRY(cudaMemsetAsync(ws, 0, p.zero_bytes, st));
    // a pageable-source cudaMemcpyAsync stages the host data before it returns, so `stage` may die at scope exit
    B200_CUDA_TRY(cudaMemcpyAsync(ws + p.off_images, stage.data(), stage.size(), cudaMemcpyHostToDevice, st));
    JpegArgs a = jpeg_args(p, in, out, ws, kJpegSubBits);
    if (p.n_sub) {
        unsigned *head = reinterpret_cast<unsigned *>(ws + p.off_head), *cta_tot = reinterpret_cast<unsigned *>(ws + p.off_cta);
        void *args[] = {&a, &head, &cta_tot};
        B200_CUDA_TRY(cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(jpeg_entropy_kernel), dim3(ctas), dim3(kJpegThreads),
                                                  args, 0, st));
        B200_LAUNCH_CHECK("jpeg_entropy_kernel");
    }
    if (p.n_blocks) {
        jpeg_idct_kernel<<<static_cast<unsigned>((p.n_blocks + kJpegIdctBlocks - 1) / kJpegIdctBlocks), kJpegThreads, 0, st>>>(a);
        B200_LAUNCH_CHECK("jpeg_idct_kernel");
    }
    jpeg_color_kernel<<<static_cast<unsigned>((p.n_pix + kJpegThreads - 1) / kJpegThreads), kJpegThreads, 0, st>>>(a);
    B200_LAUNCH_CHECK("jpeg_color_kernel");
    return B200_OK;
}

}  // extern "C"
