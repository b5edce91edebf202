// SHAP kernel weights, the weighted linear surrogate fit (one Adam step per coalition batch) and the
// aggregation of node importances into community scores.
//
// Replaces kernels.py:22-174 (Kernel.compute), wlm.py:132-278 / 441-520 (train_model, regularizer,
// weighted_mse_loss, Adam with weight_decay=1e-2), explainer.py:288-314 (weight_stacking) and
// pathways.py:387-429 (aggregate).  The fit reads the coalition bits straight from the packed
// node-major matrix the masked SpMM uses; the (B, N) float mask of the reference never exists.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace xpgnn {

__device__ __forceinline__ double finite_or_zero(double x) { return (isnan(x) || isinf(x)) ? 0.0 : x; }

// one block per batch of coalitions
__global__ void __launch_bounds__(128) shap_weights_kernel(const int32_t* __restrict__ popcount, int S, int M, int batch,
                                                           const double* __restrict__ tables, const int32_t* __restrict__ table_ptr,
                                                           int n_tables, double* __restrict__ out) {
  __shared__ double red[128];
  __shared__ int decision;
  const int s_lo = blockIdx.x * batch, s_hi = min(S, s_lo + batch);
  const int total = M - 1;  // kernels.py:146
  if (total <= 1000) {      // kernels.py:164-166 -> original_shap_kernel (:82-113)
    for (int s = s_lo + threadIdx.x; s < s_hi; s += blockDim.x) {
      const int k = popcount[s];
      const double choose = tables[k];  // binom(M, k)
      // python_scalar / tensor == reciprocal(tensor) * scalar in torch (two roundings)
      const double kern = (1.0 / (choose * (double)(total + 1 - k) * (double)k)) * (double)total;
      out[s] = finite_or_zero(kern);
    }
    return;
  }
  // approximate_shap_kernel (kernels.py:22-80) with the shrinking reference of :152-162
  for (int t = 0; t < n_tables; ++t) {
    const double* tab = tables + table_ptr[t];
    const int ref = table_ptr[t + 1] - table_ptr[t];
    double part = 0.0;
    for (int s = s_lo + threadIdx.x; s < s_hi; s += blockDim.x) {
      const int k = popcount[s];
      int idx = (int)(long long)__fdiv_rn((float)((long long)k * 1000ll), (float)total);  // int64*1000/int -> fp32
      idx = max(0, min(idx, ref - 1));
      const double choose = ((tab[idx] + 1e-10) * (double)total) / 1000.0;
      const double kern = (1.0 / (choose * (double)k * (double)(total - k))) * (double)total;
      out[s] = kern;
      part += kern;
    }
    red[threadIdx.x] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
      double sum = 0.0;
      for (int i = 0; i < (int)blockDim.x; ++i) sum += red[i];
      // while (sum == 0 and ref > 0): ...; if sum > 0: break; else ref = int(0.9 ref)
      decision = (sum > 0.0) ? 0 : ((sum == 0.0 && t + 1 < n_tables) ? 1 : 0);
    }
    __syncthreads();
    if (!decision) break;
    __syncthreads();
  }
  for (int s = s_lo + threadIdx.x; s < s_hi; s += blockDim.x) out[s] = finite_or_zero(out[s]);
}

// ------------------------------------------------------------------------------------------
// WLM fit
// ------------------------------------------------------------------------------------------
constexpr int kFitChunk = 2048;  // nodes per block in the prediction pass

// partial[chunk][word][lane] = sum_{v in chunk} bit(v, 32*word+lane) * w[v];  abs_part[chunk] = sum |w[v]|
// (the bodies are shared by the single and the batched fit kernels, so that both run the same arithmetic)
__device__ __forceinline__ void wlm_pred_partial_body(const uint32_t* __restrict__ act, int W, int N, int w_lo, int n_words,
                                                      const float* __restrict__ wt, float* __restrict__ partial,
                                                      float* __restrict__ abs_part, int chunk, int word) {
  __shared__ float sm[8][32];
  __shared__ float sabs[8];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int v_lo = chunk * kFitChunk, v_hi = min(N, v_lo + kFitChunk);
  float acc = 0.0f, aabs = 0.0f;
  for (int v = v_lo + wib; v < v_hi; v += 8) {
    const uint32_t bits = act[(int64_t)v * W + w_lo + word];
    const float x = wt[v];
    if ((bits >> lane) & 1u) acc += x;
    if (lane == 0) aabs += fabsf(x);
  }
  sm[wib][lane] = acc;
  if (lane == 0) sabs[wib] = aabs;
  __syncthreads();
  if (wib == 0) {
    float t = 0.0f;
    for (int i = 0; i < 8; ++i) t += sm[i][lane];
    partial[((int64_t)chunk * n_words + word) * 32 + lane] = t;
    if (lane == 0 && word == 0) {
      float a = 0.0f;
      for (int i = 0; i < 8; ++i) a += sabs[i];
      abs_part[chunk] = a;
    }
  }
}

__global__ void __launch_bounds__(256) wlm_pred_partial_kernel(const uint32_t* __restrict__ act, int W, int N, int w_lo, int n_words,
                                                               const float* __restrict__ wt, float* __restrict__ partial,
                                                               float* __restrict__ abs_part) {
  wlm_pred_partial_body(act, W, N, w_lo, n_words, wt, partial, abs_part, blockIdx.x, blockIdx.y);
}

// single block: predictions, residual coefficients dp[j], loss
__device__ __forceinline__ void wlm_residual_body(const float* __restrict__ partial, const float* __restrict__ abs_part, int n_chunks,
                                                  int n_words, int w_lo, int s_lo, int B, int N, const float* __restrict__ y, int64_t ldy,
                                                  const double* __restrict__ kern, int broadcast_y, double l1_lambda,
                                                  float* __restrict__ dp, double* __restrict__ loss_out) {
  extern __shared__ float pred[];  // B floats
  __shared__ double red[256];
  __shared__ double K_sh, ysum_sh;
  for (int j = threadIdx.x; j < B; j += blockDim.x) {
    const int bit = (s_lo + j) - w_lo * 32;
    const int word = bit >> 5, lane = bit & 31;
    float p = 0.0f;
    for (int c = 0; c < n_chunks; ++c) p += partial[((int64_t)c * n_words + word) * 32 + lane];
    pred[j] = p;
  }
  double kpart = 0.0, ypart = 0.0;
  for (int j = threadIdx.x; j < B; j += blockDim.x) {
    kpart += kern[s_lo + j];
    ypart += (double)y[(int64_t)(s_lo + j) * ldy];
  }
  red[threadIdx.x] = kpart;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (int)blockDim.x; ++i) t += red[i];
    K_sh = t;
  }
  __syncthreads();
  red[threadIdx.x] = ypart;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (int)blockDim.x; ++i) t += red[i];
    ysum_sh = t;
  }
  __syncthreads();
  const double K = K_sh;
  const float ysum = (float)ysum_sh;
  double lpart = 0.0;
  for (int j = threadIdx.x; j < B; j += blockDim.x) {
    const double kj = kern[s_lo + j];
    const float p = pred[j];
    if (broadcast_y) {
      // loss = mean_{i,j} k_j (p_j - y_i)^2 / K   (wlm.py:517: (B,) - (B,1) broadcasts to (B,B))
      const float c = (float)((1.0 / K) / ((double)B * (double)B) * kj);
      dp[j] = c * 2.0f * ((float)B * p - ysum);
      if (loss_out) {
        double acc = 0.0;
        for (int i = 0; i < B; ++i) {
          const float d = p - y[(int64_t)(s_lo + i) * ldy];
          acc += kj * (double)(d * d);
        }
        lpart += acc;
      }
    } else {
      const float c = (float)((1.0 / K) / (double)B * kj);
      const float d = p - y[(int64_t)(s_lo + j) * ldy];
      dp[j] = c * 2.0f * d;
      lpart += kj * (double)(d * d);
    }
  }
  if (loss_out) {
    red[threadIdx.x] = lpart;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < (int)blockDim.x; ++i) t += red[i];
      const double cnt = broadcast_y ? (double)B * (double)B : (double)B;
      float a = 0.0f;
      for (int c = 0; c < n_chunks; ++c) a += abs_part[c];
      *loss_out = (t / cnt) / K + l1_lambda * ((double)a / (double)N);
    }
  }
}

__global__ void __launch_bounds__(256) wlm_residual_kernel(const float* __restrict__ partial, const float* __restrict__ abs_part, int n_chunks,
                                                           int n_words, int w_lo, int s_lo, int B, int N, const float* __restrict__ y,
                                                           const double* __restrict__ kern, int broadcast_y, double l1_lambda,
                                                           float* __restrict__ dp, double* __restrict__ loss_out) {
  wlm_residual_body(partial, abs_part, n_chunks, n_words, w_lo, s_lo, B, N, y, 1, kern, broadcast_y, l1_lambda, dp, loss_out);
}

// one thread per node: gradient from the batch bits, L1 subgradient, coupled weight decay, Adam
__device__ __forceinline__ void wlm_adam_body(const uint32_t* __restrict__ act, int W, int N, int s_lo, int B, const float* __restrict__ dp,
                                              float* __restrict__ wt, float* __restrict__ m, float* __restrict__ vv, float l1_over_n,
                                              float wd, float step_size, float bc2_sqrt, float one_minus_b1, float b2,
                                              float one_minus_b2, float eps, int block) {
  extern __shared__ float sdp[];
  for (int j = threadIdx.x; j < B; j += blockDim.x) sdp[j] = dp[j];
  __syncthreads();
  const int v = block * blockDim.x + threadIdx.x;
  if (v >= N) return;
  float g = 0.0f;
  int j = 0;
  while (j < B) {
    const int s = s_lo + j;
    const int word = s >> 5, off = s & 31;
    const int n = min(32 - off, B - j);
    uint32_t bits = act[(int64_t)v * W + word] >> off;
    if (n < 32) bits &= (1u << n) - 1u;
    while (bits) {
      const int b = __ffs(bits) - 1;
      bits &= bits - 1;
      g += sdp[j + b];
    }
    j += n;
  }
  const float x = wt[v];
  g += l1_over_n * (float)((x > 0.0f) - (x < 0.0f));  // d/dw lambda * mean|w|
  g = fmaf(wd, x, g);                                  // Adam(weight_decay=1e-2), wlm.py:478
  float mm = m[v], v2 = vv[v];
  mm = fmaf(g - mm, one_minus_b1, mm);                 // exp_avg.lerp_(grad, 1 - beta1)
  v2 = fmaf(one_minus_b2 * g, g, v2 * b2);             // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
  const float denom = sqrtf(v2) / bc2_sqrt + eps;
  wt[v] = x - step_size * (mm / denom);
  m[v] = mm;
  vv[v] = v2;
}

__global__ void __launch_bounds__(256) wlm_adam_kernel(const uint32_t* __restrict__ act, int W, int N, int s_lo, int B, const float* __restrict__ dp,
                                                       float* __restrict__ wt, float* __restrict__ m, float* __restrict__ vv, float l1_over_n,
                                                       float wd, float step_size, float bc2_sqrt, float one_minus_b1, float b2,
                                                       float one_minus_b2, float eps) {
  wlm_adam_body(act, W, N, s_lo, B, dp, wt, m, vv, l1_over_n, wd, step_size, bc2_sqrt, one_minus_b1, b2, one_minus_b2, eps, blockIdx.x);
}

// ---- batched fit: blockIdx.z picks the surrogate (order[z]: the surrogates still running at this step index)
struct FitDev {
  const uint32_t* act;
  const float* y;
  const double* kern;
  float *w, *m, *v, *partial, *absp, *dp;
  double* losses;
  int n, s, batch, n_chunks;
  float l1_over_n;
};

struct FitStep {
  int s_lo, B, w_lo, n_words;
};

__device__ __forceinline__ FitStep fit_step(const FitDev& q, int step) {
  FitStep t;
  t.s_lo = step * q.batch;
  t.B = min(q.batch, q.s - t.s_lo);
  t.w_lo = t.s_lo / 32;
  t.n_words = (t.s_lo + t.B - 1) / 32 - t.w_lo + 1;
  return t;
}

__global__ void __launch_bounds__(256) wlm_pred_partial_batch_kernel(const FitDev* __restrict__ qs, const int32_t* __restrict__ order, int W,
                                                                     int step) {
  const FitDev q = qs[order[blockIdx.z]];
  const FitStep t = fit_step(q, step);
  if ((int)blockIdx.x >= q.n_chunks || (int)blockIdx.y >= t.n_words) return;
  wlm_pred_partial_body(q.act, W, q.n, t.w_lo, t.n_words, q.w, q.partial, q.absp, blockIdx.x, blockIdx.y);
}

__global__ void __launch_bounds__(256) wlm_residual_batch_kernel(const FitDev* __restrict__ qs, const int32_t* __restrict__ order, int64_t ldy,
                                                                 int step, int broadcast_y, double l1_lambda) {
  const FitDev q = qs[order[blockIdx.x]];
  const FitStep t = fit_step(q, step);
  wlm_residual_body(q.partial, q.absp, q.n_chunks, t.n_words, t.w_lo, t.s_lo, t.B, q.n, q.y, ldy, q.kern, broadcast_y, l1_lambda, q.dp,
                    q.losses ? q.losses + step : nullptr);
}

__global__ void __launch_bounds__(256) wlm_adam_batch_kernel(const FitDev* __restrict__ qs, const int32_t* __restrict__ order, int W, float wd,
                                                             int step, float step_size, float bc2_sqrt, float one_minus_b1, float b2,
                                                             float one_minus_b2, float eps) {
  const FitDev q = qs[order[blockIdx.y]];
  if ((int)(blockIdx.x * blockDim.x) >= q.n) return;  // whole block outside this surrogate (uniform: no barrier skipped)
  const FitStep t = fit_step(q, step);
  wlm_adam_body(q.act, W, q.n, t.s_lo, t.B, q.dp, q.w, q.m, q.v, q.l1_over_n, wd, step_size, bc2_sqrt, one_minus_b1, b2, one_minus_b2,
                eps, blockIdx.x);
}

__global__ void repeat_stats_kernel(const float* __restrict__ w, int times, int N, float* __restrict__ mean, float* __restrict__ sd) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= N) return;
  float s = 0.0f;
  for (int t = 0; t < times; ++t) s += w[(int64_t)t * N + v];
  const float mu = s / (float)times;
  float q = 0.0f;
  for (int t = 0; t < times; ++t) {
    const float d = w[(int64_t)t * N + v] - mu;
    q = fmaf(d, d, q);
  }
  mean[v] = mu;
  sd[v] = sqrtf(q / (float)times);  // torch.std(unbiased=False)
}

__global__ void __launch_bounds__(128) community_mean_kernel(const float* __restrict__ w, const int32_t* __restrict__ com_ptr,
                                                             const int32_t* __restrict__ com_idx, int C, float* __restrict__ score) {
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= C) return;
  const int lo = com_ptr[c], hi = com_ptr[c + 1];
  float s = 0.0f;
  for (int i = lo + lane; i < hi; i += 32) s += w[com_idx[i]];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) score[c] = s / (float)(hi - lo);  // 0/0 -> NaN like torch.mean of an empty selection
}

}  // namespace xpgnn

using namespace xpgnn;

extern "C" {

int xpgnn_shap_weights(const int32_t* popcount, int32_t S, int32_t M, int32_t batch, const double* tables,
                       const int32_t* table_ptr, int32_t n_tables, double* out, void* stream) {
  XP_REQUIRE(popcount && tables && out && S >= 0 && batch > 0 && M >= 1, "bad argument");
  XP_REQUIRE(M - 1 <= 1000 || (table_ptr && n_tables >= 1), "approximate branch needs the reference tables");
  if (S == 0) return 0;
  XP_LAUNCH(shap_weights_kernel, (int)ceil_div(S, batch), 128, 0, (cudaStream_t)stream, popcount, S, M, batch, tables, table_ptr,
            n_tables, out);
  return 0;
}

int xpgnn_wlm_fit(const uint32_t* act, int32_t W, int32_t N, int32_t S, int32_t batch, const float* y, const double* kern,
                  float* w, double lr, double l1_lambda, double weight_decay, int32_t broadcast_y, double* losses,
                  void* stream) {
  XP_REQUIRE(act && y && kern && w && N > 0 && S >= 0 && batch > 0 && (int64_t)W * 32 >= S, "bad argument");
  XP_REQUIRE(batch <= 8192, "batch larger than 8192 coalitions is not supported by the fit kernels");
  if (S == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int n_chunks = (int)ceil_div(N, kFitChunk);
  const int max_words = batch / 32 + 2;
  Scratch partial(st), absp(st), dp(st), mv(st);
  XP_CHECK(partial.alloc(sizeof(float) * (size_t)n_chunks * max_words * 32));
  XP_CHECK(absp.alloc(sizeof(float) * n_chunks));
  XP_CHECK(dp.alloc(sizeof(float) * batch));
  XP_CHECK(mv.alloc(sizeof(float) * 2 * (size_t)N));
  XP_CHECK(cudaMemsetAsync(mv.p, 0, sizeof(float) * 2 * (size_t)N, st));
  float* m = mv.as<float>();
  float* v = m + N;
  const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
  int step = 0;
  for (int s_lo = 0; s_lo < S; s_lo += batch) {
    ++step;
    const int B = std::min(batch, S - s_lo);
    const int w_lo = s_lo / 32, w_hi = (s_lo + B - 1) / 32, n_words = w_hi - w_lo + 1;
    dim3 g1((unsigned)n_chunks, (unsigned)n_words);
    XP_LAUNCH(wlm_pred_partial_kernel, g1, 256, 0, st, act, W, N, w_lo, n_words, w, partial.as<float>(), absp.as<float>());
    XP_LAUNCH(wlm_residual_kernel, 1, 256, sizeof(float) * B, st, partial.as<float>(), absp.as<float>(), n_chunks, n_words, w_lo,
              s_lo, B, N, y, kern, broadcast_y, l1_lambda, dp.as<float>(), losses ? losses + (step - 1) : nullptr);
    const double bc1 = 1.0 - pow(b1, step), bc2 = 1.0 - pow(b2, step);
    XP_LAUNCH(wlm_adam_kernel, (int)ceil_div(N, 256), 256, sizeof(float) * B, st, act, W, N, s_lo, B, dp.as<float>(), w, m, v,
              (float)(l1_lambda / (double)N), (float)weight_decay, (float)(lr / bc1), (float)sqrt(bc2), (float)(1.0 - b1),
              (float)b2, (float)(1.0 - b2), (float)eps);
  }
  return 0;
}

int xpgnn_wlm_fit_batch(const uint32_t* act, int32_t W, const float* y, int64_t ldy, const double* kern, float* w,
                        const xpgnn_fit_query_t* queries_host, int32_t Q, double lr, double l1_lambda, double weight_decay,
                        int32_t broadcast_y, void* stream) {
  XP_REQUIRE(act && y && kern && w && queries_host && Q >= 0 && W > 0 && ldy > 0, "bad argument");
  if (Q == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  // host side: per-surrogate scratch offsets (the same sizes xpgnn_wlm_fit allocates), step counts, launch shapes
  std::vector<FitDev> qs(Q);
  std::vector<int> steps(Q);
  size_t n_partial = 0, n_absp = 0, n_dp = 0, n_mv = 0;
  int max_chunks = 1, max_words = 1, max_batch = 1, max_n = 1, max_steps = 0;
  for (int i = 0; i < Q; ++i) {
    const xpgnn_fit_query_t& d = queries_host[i];
    XP_REQUIRE(d.n > 0 && d.s >= 0 && d.batch > 0 && d.act_off >= 0 && d.y_off >= 0 && d.kern_off >= 0 && d.w_off >= 0,
               "bad surrogate descriptor");
    XP_REQUIRE(d.batch <= 8192, "batch larger than 8192 coalitions is not supported by the fit kernels");
    const int n_chunks = (int)ceil_div(d.n, kFitChunk), words = d.batch / 32 + 2;
    steps[i] = (int)ceil_div(d.s, d.batch);
    n_partial += (size_t)n_chunks * words * 32;
    n_absp += n_chunks;
    n_dp += d.batch;
    n_mv += 2 * (size_t)d.n;
    max_chunks = std::max(max_chunks, n_chunks);
    max_words = std::max(max_words, words);
    max_batch = std::max(max_batch, d.batch);
    max_n = std::max(max_n, d.n);
    max_steps = std::max(max_steps, steps[i]);
  }
  if (max_steps == 0) return 0;
  Scratch partial(st), absp(st), dp(st), mv(st), dq(st), dorder(st);
  XP_CHECK(partial.alloc(sizeof(float) * n_partial));
  XP_CHECK(absp.alloc(sizeof(float) * n_absp));
  XP_CHECK(dp.alloc(sizeof(float) * n_dp));
  XP_CHECK(mv.alloc(sizeof(float) * n_mv));
  XP_CHECK(cudaMemsetAsync(mv.p, 0, sizeof(float) * n_mv, st));
  size_t o_partial = 0, o_absp = 0, o_dp = 0, o_mv = 0;
  for (int i = 0; i < Q; ++i) {
    const xpgnn_fit_query_t& d = queries_host[i];
    FitDev& q = qs[i];
    q.act = act + d.act_off;
    q.y = y + d.y_off;
    q.kern = kern + d.kern_off;
    q.w = w + d.w_off;
    q.m = mv.as<float>() + o_mv;
    q.v = q.m + d.n;
    q.n_chunks = (int)ceil_div(d.n, kFitChunk);
    q.partial = partial.as<float>() + o_partial;
    q.absp = absp.as<float>() + o_absp;
    q.dp = dp.as<float>() + o_dp;
    q.losses = d.losses;
    q.n = d.n;
    q.s = d.s;
    q.batch = d.batch;
    q.l1_over_n = (float)(l1_lambda / (double)d.n);
    o_partial += (size_t)q.n_chunks * (d.batch / 32 + 2) * 32;
    o_absp += q.n_chunks;
    o_dp += d.batch;
    o_mv += 2 * (size_t)d.n;
  }
  // surrogates by step count, longest first: at step index t the first n_active[t] entries still run
  std::vector<int32_t> order(Q);
  for (int i = 0; i < Q; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return steps[a] > steps[b]; });
  XP_CHECK(dq.alloc(sizeof(FitDev) * Q));
  XP_CHECK(dorder.alloc(sizeof(int32_t) * Q));
  XP_CHECK(cudaMemcpyAsync(dq.p, qs.data(), sizeof(FitDev) * Q, cudaMemcpyHostToDevice, st));
  XP_CHECK(cudaMemcpyAsync(dorder.p, order.data(), sizeof(int32_t) * Q, cudaMemcpyHostToDevice, st));
  // the pageable copies above are staged before they return; the host vectors may go out of scope
  const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
  int n_active = Q;
  for (int step = 1; step <= max_steps; ++step) {
    while (n_active > 0 && steps[order[n_active - 1]] < step) --n_active;
    const double bc1 = 1.0 - pow(b1, step), bc2 = 1.0 - pow(b2, step);
    dim3 g1((unsigned)max_chunks, (unsigned)max_words, (unsigned)n_active);
    XP_LAUNCH(wlm_pred_partial_batch_kernel, g1, 256, 0, st, dq.as<FitDev>(), dorder.as<int32_t>(), W, step - 1);
    XP_LAUNCH(wlm_residual_batch_kernel, n_active, 256, sizeof(float) * max_batch, st, dq.as<FitDev>(), dorder.as<int32_t>(), ldy,
              step - 1, broadcast_y, l1_lambda);
    dim3 g3((unsigned)ceil_div(max_n, 256), (unsigned)n_active);
    XP_LAUNCH(wlm_adam_batch_kernel, g3, 256, sizeof(float) * max_batch, st, dq.as<FitDev>(), dorder.as<int32_t>(), W,
              (float)weight_decay, step - 1, (float)(lr / bc1), (float)sqrt(bc2), (float)(1.0 - b1), (float)b2, (float)(1.0 - b2),
              (float)eps);
  }
  return 0;
}

int xpgnn_repeat_stats(const float* weights, int32_t times, int32_t N, float* mean, float* sd, void* stream) {
  XP_REQUIRE(weights && mean && sd && times > 0 && N > 0, "bad argument");
  XP_LAUNCH(repeat_stats_kernel, (int)ceil_div(N, 256), 256, 0, (cudaStream_t)stream, weights, times, N, mean, sd);
  return 0;
}

int xpgnn_community_mean(const float* w, const int32_t* com_ptr, const int32_t* com_idx, int32_t C, float* score,
                         void* stream) {
  XP_REQUIRE(w && com_ptr && com_idx && score && C >= 0, "bad argument");
  if (C == 0) return 0;
  XP_LAUNCH(community_mean_kernel, (int)ceil_div(C, 4), 128, 0, (cudaStream_t)stream, w, com_ptr, com_idx, C, score);
  return 0;
}

}  // extern "C"
