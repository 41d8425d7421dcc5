// Host API of the fused memory-bound kernels (see fused_ops.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pb {

struct OptimHyper {
  int kind;          // 0 ADOPT, 1 DecoupledAdamW, 2 SGD
  int first_step;    // ADOPT: step 0 only seeds v = g^2
  float lr, beta1, beta2, eps;
  float decay;         // multiplicative weight decay factor applied to p (1 = none)
  float clip;          // ADOPT: step^0.25 clamp on the normalised gradient (inf = off)
  float step_size;     // AdamW: lr / (1 - beta1^t)
  float inv_sqrt_bc2;  // AdamW: 1 / sqrt(1 - beta2^t)
};

// pos: optional int32 [T] explicit positions (nullptr = t % S); S is then the number of rows of wpe
void embed_fwd(const int64_t* ids, const void* wte, const void* wpe, void* out, long long T, int S, int d, int V, cudaStream_t st,
               const int* pos = nullptr);
void embed_bwd(const int64_t* ids, const void* dh, float* dwte, float* dwpe, long long T, int S, int d, int V, cudaStream_t st);
void layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, long long T, int d,
                   float eps, cudaStream_t st);
void layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd, const void* dres, void* dx,
                   float* dgamma, float* dbeta, long long T, int d, cudaStream_t st);
void col_reduce(const void* dy, long long ld, const void* x, const float* mean, const float* rstd, float* out_sum, float* out_dot,
                long long T, int d, cudaStream_t st);
void cross_entropy(void* logits, long long ld, const int64_t* targets, long long rows, int V, float grad_scale, bool write_grad,
                   double* stats, float* row_lse, const float* unigram_logp, cudaStream_t st);
void flat_sqnorm(const float* x, long long n, double* out_accum, cudaStream_t st);
void sqrt_finalize(const double* in, float* out, cudaStream_t st);
void axpby(float* acc, const float* x, float a, float b, long long n, cudaStream_t st);
void cast_fp32_to_bf16(const float* src, void* dst, long long n, cudaStream_t st);
void fused_optimizer(float* p, const float* g, float* m, float* v, void* shadow, long long n, const OptimHyper& h,
                     const float* grad_mult, cudaStream_t st);

}  // namespace pb
