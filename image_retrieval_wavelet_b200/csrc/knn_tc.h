// Host interface of the k-NN's tensor-core scorer (knn_tc.cu), driven by b200_knn_topk (knn.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace b200 {

struct TcMaps {
    CUtensorMap q_hi, q_lo, r_hi, r_lo;
};

// bf16 hi / lo copies of both operands + their tensor maps; `sample` reads every sample_stride-th reference row (a tensor
// map with a longer row stride: no gather pass).
struct TcContext {
    TcMaps full, sample;
    int Q, Dp;
    long long N, Ns;
};

size_t knn_tc_extra_workspace(int Q, long long N, int D);

// Splits both operands into bf16 hi + lo (two launches) and builds the tensor maps.  sample_stride > 0 also builds maps
// over every sample_stride-th reference row.  B200_ERR_UNSUPPORTED when the tensor-map entry point is unavailable.
int knn_tc_prepare(const float *queries, const float *refs, int Q, long long N, int D, void *extra, long long sample_stride,
                   TcContext *ctx, cudaStream_t st);

// One pass of the scorer: sample != 0 scores the sampled reference rows (Ns columns), else all N.  thr == nullptr: the
// score matrix goes to S; otherwise the epilogue filters (see TcFilter in knn_tc.cu).
int knn_tc_scores(const TcContext *ctx, int sample, float *S, long long ldS, const float *thr, unsigned long long *cand,
                  uint32_t *cand_cnt, uint32_t cap, const uint32_t *gate, cudaStream_t st);

}  // namespace b200
