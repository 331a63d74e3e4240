// Segmented learning-to-rank losses, forward + backward in one launch.
// One CTA per candidate group (reactant); the group lives in shared memory, so the
// reference's Python loop of ~14 tiny launches per group (train/loss.py:86-95) becomes a
// single kernel that emits the normalised loss and dL/dscore.
#include <math_constants.h>

#include "rr_common.cuh"

namespace rr {

constexpr int kLossThreads = 256;
constexpr int kMaxGroup = 8192;         // largest group the segmented kernels take (dynamic shared memory: 4 x 4 B x capacity for ListMLE)
constexpr int kDefaultGroupCap = 2048;  // capacity when the caller gives no max_group hint (rr_loss_fwdbwd)
constexpr int kMaxMetricGroup = 8192;   // 128 KB of shared doubles

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// block-wide reductions; `red` is >= 32 floats of shared scratch
__device__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
  if (threadIdx.x < 32) r = warp_sum(r);
  if (threadIdx.x == 0) red[0] = r;
  __syncthreads();
  r = red[0];
  __syncthreads();
  return r;
}
__device__ float block_max(float v, float* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : -CUDART_INF_F;
  if (threadIdx.x < 32) r = warp_max(r);
  if (threadIdx.x == 0) red[0] = r;
  __syncthreads();
  r = red[0];
  __syncthreads();
  return r;
}

// inclusive Hillis-Steele scan over buf[0..n) (left to right), ping-pong with tmp; result in buf
__device__ void block_scan(float* buf, float* tmp, int n) {
  float* in = buf;
  float* out = tmp;
  for (int off = 1; off < n; off <<= 1) {
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = in[i] + (i >= off ? in[i - off] : 0.f);
    float* sw = in;
    in = out;
    out = sw;
  }
  __syncthreads();
  if (in != buf)
    for (int i = threadIdx.x; i < n; i += blockDim.x) buf[i] = in[i];
  __syncthreads();
}

// bitonic sort of (key, id)[0..P), P a power of two, descending by key with ties by ascending id; pad with key -inf and ids >= the
// group size, and the padding sorts last.  Synchronises before and after.
__device__ __forceinline__ void block_sort_desc(float* key, int* id, int P) {
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const int l = i ^ j;
        if (l > i) {
          const bool desc = (i & k) == 0;
          const float ki = key[i], kl = key[l];
          const int ii = id[i], il = id[l];
          const bool i_first = (ki > kl) || (ki == kl && ii < il);  // i should precede l in descending order
          if (desc ? !i_first : i_first) {
            key[i] = kl; key[l] = ki;
            id[i] = il; id[l] = ii;
          }
        }
      }
    }
  __syncthreads();
}

// A block's share of the loss: added into loss[0] with an atomic, or (DET, deterministic mode) stored to loss[block], the partials that
// k_sum_parts then adds in block order.  (A macro, not a function: the default kernels then compile exactly as they did before DET existed.)
#define RR_PUT_LOSS(loss, v)                                          \
  do {                                                                \
    if constexpr (DET) (loss)[blockIdx.y * gridDim.x + blockIdx.x] = (v); \
    else atomicAdd((loss), (v));                                      \
  } while (0)

// ---------------------------------------------------------------------------------------
// ListMLE  (MLEloss loss.py:64-99, LogCumsumExp loss.py:9-61)
// ---------------------------------------------------------------------------------------
// DIS = true: MLEDisLoss (loss.py:102-141) on scores [N,2] = (mean, variance).  Its n x n lower-triangular form reduces to ListMLE of
// z = mean + variance / 2 plus the group mean of the variance:  mean_j( lcse_j(z) - z_j + v_j ).
template <bool DIS, bool DET>
__global__ void __launch_bounds__(kLossThreads) k_listmle(const float* __restrict__ scores, const float* __restrict__ targets,
                                                          const int* __restrict__ seg, float inv_norm, float* __restrict__ loss,
                                                          float* __restrict__ dscore, int cap) {
  extern __shared__ float loss_dyn[];            // key | id | a | b, `cap` entries each (cap = a power of two >= the largest group)
  float* key = loss_dyn;
  int* id = reinterpret_cast<int*>(loss_dyn + cap);
  float* a = loss_dyn + 2 * cap;
  float* b = loss_dyn + 3 * cap;
  __shared__ float red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  if (n > cap) {   // the shared arrays hold `cap` candidates: a larger group poisons the result instead of overrunning them
    for (int i = threadIdx.x; i < n * (DIS ? 2 : 1); i += blockDim.x) dscore[static_cast<size_t>(o) * (DIS ? 2 : 1) + i] = CUDART_NAN_F;
    if (threadIdx.x == 0) RR_PUT_LOSS(loss, CUDART_NAN_F);
    return;
  }
  int P = 1;
  while (P < n) P <<= 1;
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    key[i] = i < n ? targets[o + i] : -CUDART_INF_F;
    id[i] = i;
  }
  // descending by target (ties by index; torch.argsort leaves them unspecified)
  block_sort_desc(key, id, P);
  // x = scores sorted; reuse key[] for x
  float mx = -CUDART_INF_F;
  float vsum = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float x;
    if (DIS) {
      const float v = scores[2 * (o + id[i]) + 1];
      x = scores[2 * (o + id[i])] + 0.5f * v;
      vsum += v;
    } else {
      x = scores[o + id[i]];
    }
    key[i] = x;
    mx = fmaxf(mx, x);
  }
  mx = block_max(mx, red);
  if (DIS) vsum = block_sum(vsum, red);
  // suffix sums of exp(x - m): scan the reversed array
  for (int i = threadIdx.x; i < n; i += blockDim.x) a[i] = expf(key[n - 1 - i] - mx);
  block_scan(a, b, n);  // a[i] = sum_{k >= n-1-i} e_k
  float part = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float suffix = a[n - 1 - i];
    part += (logf(suffix) + mx) - key[i];
    b[i] = 1.f / suffix;
  }
  __syncthreads();
  const float total = block_sum(part, red);
  // prefix sums of 1/suffix  (== exp(m) * cumsum(exp(-lcse)), loss.py:59)
  // a[] is free again after the loop above has been read by everyone (block_sum synchronised)
  for (int i = threadIdx.x; i < n; i += blockDim.x) a[i] = b[i];
  block_scan(a, b, n);
  const float gscale = inv_norm / static_cast<float>(n);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float e = expf(key[i] - mx);
    const float gz = (e * a[i] - 1.f) * gscale;
    if (DIS) {
      dscore[2 * (o + id[i])] = gz;
      dscore[2 * (o + id[i]) + 1] = 0.5f * gz + gscale;
    } else {
      dscore[o + id[i]] = gz;
    }
  }
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, (total + (DIS ? vsum : 0.f)) * gscale);
}

// ---------------------------------------------------------------------------------------
// ListNet@1  (ListnetLoss loss.py:317-352): mean over ALL items (norm = N)
// ---------------------------------------------------------------------------------------
// DIS = true: Listnet_For_Gauss (loss.py:233-272) on scores [N,2] = (mean, variance): with u = mean + variance / 2 its n x n form is
// -p_i log pred_i = p_i (lse(u) - u_i + v_i), averaged over the items of the GROUP and then over groups (inv_norm = 1 / G here).
template <bool DIS, bool DET>
__global__ void __launch_bounds__(kLossThreads) k_listnet(const float* __restrict__ scores, const float* __restrict__ targets,
                                                          const int* __restrict__ seg, float inv_norm, float* __restrict__ loss,
                                                          float* __restrict__ dscore) {
  __shared__ float red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  auto score = [&](int i) { return DIS ? scores[2 * (o + i)] + 0.5f * scores[2 * (o + i) + 1] : scores[o + i]; };
  float ms = -CUDART_INF_F, mt = -CUDART_INF_F;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    ms = fmaxf(ms, score(i));
    mt = fmaxf(mt, targets[o + i]);
  }
  ms = block_max(ms, red);
  mt = block_max(mt, red);
  float zs = 0.f, zt = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    zs += expf(score(i) - ms);
    zt += expf(targets[o + i] - mt);
  }
  zs = block_sum(zs, red);
  zt = block_sum(zt, red);
  const float lzs = logf(zs), izt = 1.f / zt, izs = 1.f / zs;
  const float c = DIS ? inv_norm / static_cast<float>(n) : inv_norm;
  float part = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float ds = score(i) - ms;
    const float p = expf(targets[o + i] - mt) * izt;
    const float gu = (expf(ds) * izs - p) * c;
    if (DIS) {
      const float v = scores[2 * (o + i) + 1];
      part -= p * (ds - lzs - v);
      dscore[2 * (o + i)] = gu;
      dscore[2 * (o + i) + 1] = 0.5f * gu + p * c;
    } else {
      part -= p * (ds - lzs);
      dscore[o + i] = gu;
    }
  }
  part = block_sum(part, red);
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, part * c);
}

// ---------------------------------------------------------------------------------------
// UC-Listwise  (evidential_ranking loss.py:526-554): scores [N,2] = (mean, variance)
// ---------------------------------------------------------------------------------------
template <bool DET>
__global__ void __launch_bounds__(kLossThreads) k_evidential(const float* __restrict__ scores, const float* __restrict__ targets,
                                                             const int* __restrict__ seg, float inv_norm, float* __restrict__ loss,
                                                             float* __restrict__ dscore) {
  __shared__ float red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  float ms = -CUDART_INF_F, mt = -CUDART_INF_F;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    ms = fmaxf(ms, scores[2 * (o + i)]);
    mt = fmaxf(mt, targets[o + i]);
  }
  ms = block_max(ms, red);
  mt = block_max(mt, red);
  float zs = 0.f, zt = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    zs += expf(scores[2 * (o + i)] - ms);
    zt += expf(targets[o + i] - mt);
  }
  zs = block_sum(zs, red);
  zt = block_sum(zt, red);
  const float lzs = logf(zs), lzt = logf(zt);
  float part = 0.f, dsum = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float m = scores[2 * (o + i)], v = scores[2 * (o + i) + 1], t = targets[o + i];
    const float logq = m - ms - lzs, logp = t - mt - lzt;
    const float d = logp - logq;
    part += -logp + 0.5f * d * d / v + 0.5f * logf(2.f * 3.141592653f * v) + fabsf(m - t);
    dsum += d / v;
  }
  part = block_sum(part, red);
  dsum = block_sum(dsum, red);
  const float gscale = inv_norm / static_cast<float>(n);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float m = scores[2 * (o + i)], v = scores[2 * (o + i) + 1], t = targets[o + i];
    const float logq = m - ms - lzs, logp = t - mt - lzt;
    const float d = logp - logq;
    const float sgn = (m > t) ? 1.f : ((m < t) ? -1.f : 0.f);
    dscore[2 * (o + i)] = (expf(logq) * dsum - d / v + sgn) * gscale;
    dscore[2 * (o + i) + 1] = (-0.5f * d * d / (v * v) + 0.5f / v) * gscale;
  }
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, part * gscale);
}

// ---------------------------------------------------------------------------------------
// Listnet_with_uq (loss.py:355-399): positive scores s (softplus head), pred = s / sum(s), p = softmax(t), c_i = log(p_i / pred_i);
//   group loss = (1/n) sum_i p_i c_i  +  coef * mean_i |c_i (s_i - 1)|        (KLDivLoss 'batchmean' of a 1-D input divides by n)
// coef = max_coeff * (epoch / (epochs - 1))^3 is computed by the caller.  Mean over groups.
// ---------------------------------------------------------------------------------------
template <bool DET>
__global__ void __launch_bounds__(kLossThreads) k_listnet_uq(const float* __restrict__ scores, const float* __restrict__ targets,
                                                             const int* __restrict__ seg, float inv_norm, float coef, float* __restrict__ loss,
                                                             float* __restrict__ dscore) {
  __shared__ float red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  float mt = -CUDART_INF_F, ssum = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    mt = fmaxf(mt, targets[o + i]);
    ssum += scores[o + i];
  }
  mt = block_max(mt, red);
  ssum = block_sum(ssum, red);
  float zt = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) zt += expf(targets[o + i] - mt);
  zt = block_sum(zt, red);
  const float lzt = logf(zt), lS = logf(ssum);
  float kl = 0.f, pen = 0.f, sg = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float s = scores[o + i], logp = targets[o + i] - mt - lzt;
    const float c = logp - logf(s) + lS;
    const float res = c * (s - 1.f);
    kl += expf(logp) * c;
    pen += fabsf(res);
    sg += (res > 0.f ? 1.f : (res < 0.f ? -1.f : 0.f)) * (s - 1.f);
  }
  kl = block_sum(kl, red);
  pen = block_sum(pen, red);
  sg = block_sum(sg, red);
  const float gscale = inv_norm / static_cast<float>(n);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float s = scores[o + i], logp = targets[o + i] - mt - lzt;
    const float c = logp - logf(s) + lS;
    const float res = c * (s - 1.f);
    const float sgn = res > 0.f ? 1.f : (res < 0.f ? -1.f : 0.f);
    const float dkl = 1.f / ssum - expf(logp) / s;                          // d/ds_k of sum_i p_i c_i
    const float dpen = sg / ssum + sgn * (c - (s - 1.f) / s);               // d/ds_k of sum_i |c_i (s_i - 1)|
    dscore[o + i] = (dkl + coef * dpen) * gscale;
  }
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, (kl + coef * pen) * gscale);
}

// ---------------------------------------------------------------------------------------
// Dirichlet_uq (loss.py:440-474) on 1-D positive concentrations a: pred = a / S, p = softmax(t),
//   group loss = mean_i( (pred_i - p_i)^2 + pred_i (1 - pred_i) / (S + 1) + coef |log(p_i / pred_i) (a_i - 1)| ),  mean over groups.
// ---------------------------------------------------------------------------------------
template <bool DET>
__global__ void __launch_bounds__(kLossThreads) k_dirichlet_uq(const float* __restrict__ scores, const float* __restrict__ targets,
                                                               const int* __restrict__ seg, float inv_norm, float coef,
                                                               float* __restrict__ loss, float* __restrict__ dscore) {
  __shared__ float red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  float mt = -CUDART_INF_F, S = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    mt = fmaxf(mt, targets[o + i]);
    S += scores[o + i];
  }
  mt = block_max(mt, red);
  S = block_sum(S, red);
  float zt = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) zt += expf(targets[o + i] - mt);
  zt = block_sum(zt, red);
  const float lzt = logf(zt), lS = logf(S);
  float part = 0.f, s_ep = 0.f, s_vp = 0.f, s_v = 0.f, sg = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float a = scores[o + i], logp = targets[o + i] - mt - lzt, p = expf(logp);
    const float pr = a / S;
    const float res = (logp - logf(a) + lS) * (a - 1.f);
    part += (pr - p) * (pr - p) + pr * (1.f - pr) / (S + 1.f) + coef * fabsf(res);
    s_ep += (pr - p) * pr;
    s_vp += (1.f - 2.f * pr) * pr;
    s_v += pr * (1.f - pr);
    sg += (res > 0.f ? 1.f : (res < 0.f ? -1.f : 0.f)) * (a - 1.f);
  }
  part = block_sum(part, red);
  s_ep = block_sum(s_ep, red);
  s_vp = block_sum(s_vp, red);
  s_v = block_sum(s_v, red);
  sg = block_sum(sg, red);
  const float gscale = inv_norm / static_cast<float>(n);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float a = scores[o + i], logp = targets[o + i] - mt - lzt, p = expf(logp);
    const float pr = a / S;
    const float c = logp - logf(a) + lS;
    const float res = c * (a - 1.f);
    const float sgn = res > 0.f ? 1.f : (res < 0.f ? -1.f : 0.f);
    const float derr = 2.f / S * ((pr - p) - s_ep);
    const float dvar = ((1.f - 2.f * pr) - s_vp) / (S * (S + 1.f)) - s_v / ((S + 1.f) * (S + 1.f));
    const float dpen = sg / S + sgn * (c - (a - 1.f) / a);
    dscore[o + i] = (derr + dvar + coef * dpen) * gscale;
  }
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, part * gscale);
}

// ---------------------------------------------------------------------------------------
// evidential_loss_new (loss.py:402-437) AS THE TRAINING LOOP CALLS IT (train_listwise.py:229-260): mu, v, alpha, beta are [N,1] column
// slices of the [N,4] head while targets is [N], so every term broadcasts to an N x N matrix and the reference's loss is
//   mean over (i, j) of  NLL(mu_i, v_i, alpha_i, beta_i; t_j) + lam (|t_j - mu_i| (2 v_i + alpha_i) - 1e-4),
// every reaction's NIG scored against every target of the batch.  Reproduced as is: thread per row i, j tiled across blockIdx.y.
// ---------------------------------------------------------------------------------------
__device__ double digamma_d(double x) {      // x > 0: recurrence up to x >= 6, then the asymptotic series
  double r = 0.0;
  while (x < 6.0) {
    r -= 1.0 / x;
    x += 1.0;
  }
  const double f = 1.0 / (x * x);
  return r + log(x) - 0.5 / x - f * (1.0 / 12.0 - f * (1.0 / 120.0 - f * (1.0 / 252.0 - f * (1.0 / 240.0 - f * (1.0 / 132.0)))));
}
constexpr int kNigRows = 128;
constexpr int kNigCols = 512;
template <bool DET>
__global__ void __launch_bounds__(kNigRows) k_nig_allpairs(int N, const float* __restrict__ scores, const float* __restrict__ targets,
                                                           float inv_norm, float lam, float* __restrict__ loss, float* __restrict__ dscore) {
  __shared__ float ts[kNigCols];
  __shared__ float red[32];
  const int i = blockIdx.x * kNigRows + threadIdx.x;
  const int j0 = blockIdx.y * kNigCols, nj = min(kNigCols, N - j0);
  for (int j = threadIdx.x; j < nj; j += kNigRows) ts[j] = targets[j0 + j];
  __syncthreads();
  float part = 0.f;
  if (i < N) {
    const float4 q = *reinterpret_cast<const float4*>(scores + 4 * static_cast<size_t>(i));
    const float mu = q.x, v = q.y, al = q.z, be = q.w;
    const float om = 2.f * be * (1.f + v), ah = al + 0.5f, w = 2.f * v + al;
    float s_log = 0.f, s_abs = 0.f, g_mu = 0.f, s_inv = 0.f, s_d2inv = 0.f;
    for (int j = 0; j < nj; ++j) {
      const float d = ts[j] - mu;
      const float A = v * d * d + om, rA = 1.f / A;
      s_log += logf(A);
      s_abs += fabsf(d);
      s_inv += rA;
      s_d2inv += d * d * rA;
      g_mu += -2.f * ah * v * d * rA - lam * (d > 0.f ? w : (d < 0.f ? -w : 0.f));
    }
    const float fj = static_cast<float>(nj);
    // row-only terms, once per (row, column tile) with the tile's share of the N columns
    const float lg = static_cast<float>(lgamma(static_cast<double>(al)) - lgamma(static_cast<double>(al) + 0.5));
    const float row = 0.5f * logf(3.14159274101257324f / v) - al * logf(om) + lg - lam * 1e-4f;
    part = fj * row + ah * s_log + lam * w * s_abs;
    const float dpsi = static_cast<float>(digamma_d(static_cast<double>(al)) - digamma_d(static_cast<double>(al) + 0.5));
    const float g_v = fj * (-0.5f / v - al * 2.f * be / om) + ah * (s_d2inv + 2.f * be * s_inv) + 2.f * lam * s_abs;
    const float g_al = fj * (-logf(om) + dpsi) + s_log + lam * s_abs;
    const float g_be = -fj * al / be + ah * 2.f * (1.f + v) * s_inv;
    if constexpr (DET) {   // this column block's partial row gradient; k_nig_dscore_sum adds the blocks in order
      st_f4(dscore + 4 * (static_cast<size_t>(blockIdx.y) * N + i), make_float4(g_mu * inv_norm, g_v * inv_norm, g_al * inv_norm, g_be * inv_norm));
    } else {
      float* dr = dscore + 4 * static_cast<size_t>(i);
      atomicAdd(dr + 0, g_mu * inv_norm);
      atomicAdd(dr + 1, g_v * inv_norm);
      atomicAdd(dr + 2, g_al * inv_norm);
      atomicAdd(dr + 3, g_be * inv_norm);
    }
  }
  part = block_sum(part, red);
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, part * inv_norm);
}

// ---------------------------------------------------------------------------------------
// RankNet 'sum_session'  (train_pairwise.py:98-122): all ordered intra-group pairs
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float softplus_f(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

template <bool DET>
__global__ void __launch_bounds__(kLossThreads) k_ranknet(const float* __restrict__ scores, const float* __restrict__ targets,
                                                          const int* __restrict__ seg, float inv_norm, float sigma, float gfac,
                                                          float* __restrict__ loss, float* __restrict__ dscore, int cap) {
  extern __shared__ float loss_dyn[];            // ss | ts, `cap` entries each
  float* ss = loss_dyn;
  float* ts = loss_dyn + cap;
  __shared__ float red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  if (n > cap) {   // as in k_listmle: NaN, never a shared-memory overrun (direct C-ABI callers bypass the Python-side check)
    for (int i = threadIdx.x; i < n; i += blockDim.x) dscore[o + i] = CUDART_NAN_F;
    if (threadIdx.x == 0) RR_PUT_LOSS(loss, CUDART_NAN_F);
    return;
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    ss[i] = scores[o + i];
    ts[i] = targets[o + i];
  }
  __syncthreads();
  float part = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float si = ss[i], ti = ts[i];
    float g = 0.f;
    for (int j = 0; j < n; ++j) {
      const float d = sigma * (si - ss[j]);
      const float tj = ts[j];
      if (ti > tj) {          // pos pair: C = log(1 + exp(-sigma (s_i - s_j)))
        part += softplus_f(-d);
        g -= sigmoid_f(-d);
      } else if (ti < tj) {   // neg pair: C = log(1 + exp(+sigma (s_i - s_j)))
        part += softplus_f(d);
        g += sigmoid_f(d);
      }
    }
    dscore[o + i] = gfac * sigma * g * inv_norm;
  }
  part = block_sum(part, red);
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, part * inv_norm);
}

// ---------------------------------------------------------------------------------------
// LambdaRank (Burges et al.): RankNet with each pair weighted by |dNDCG@K|, the change of the validation's NDCG (eval.py:460-472: gain
// exp(t), discount 1 / log2(1 + rank)) if the two items swapped places.  Per group, with G_i = exp(t_i - max t) (the shift cancels in every
// NDCG ratio), r_i the 1-based descending rank of s_i with ties by index (the rule of k_rank_metrics) and D(r) = 1 / log2(1 + r) for
// r <= K, else 0:
//   w_ij = |G_i - G_j| |D(r_i) - D(r_j)| / IDCG_K,    L = (1 / norm) sum_{t_i > t_j} w_ij softplus(-sigma (s_i - s_j))
// (each unordered pair once).  w is constant in s, so dL/ds is RankNet's pair gradient times w.  K = n, or with TOP the K of the
// validation's NDCG@25 %: max(1, round_half_even(n / 4)).  A group without an ordered pair adds 0 and gets a zero gradient.
// ---------------------------------------------------------------------------------------
template <bool TOP, bool DET>
__global__ void __launch_bounds__(kLossThreads) k_lambdarank(const float* __restrict__ scores, const float* __restrict__ targets,
                                                             const int* __restrict__ seg, float inv_norm, float sigma,
                                                             float* __restrict__ loss, float* __restrict__ dscore, int cap) {
  extern __shared__ float loss_dyn[];            // ss | gs | key | id, `cap` entries each (cap = a power of two >= the largest group)
  float* ss = loss_dyn;
  float* gs = loss_dyn + cap;
  float* key = loss_dyn + 2 * cap;               // the sorts' keys, then D(r_i) by item
  int* id = reinterpret_cast<int*>(loss_dyn + 3 * cap);
  float* ts = loss_dyn + 3 * cap;                // id[]'s space, after the sorts: the targets
  __shared__ float red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  if (n > cap) {   // as in k_listmle: NaN, never a shared-memory overrun
    for (int i = threadIdx.x; i < n; i += blockDim.x) dscore[o + i] = CUDART_NAN_F;
    if (threadIdx.x == 0) RR_PUT_LOSS(loss, CUDART_NAN_F);
    return;
  }
  int P = 1;
  while (P < n) P <<= 1;
  const int K = TOP ? max(1, __float2int_rn(0.25f * static_cast<float>(n))) : n;    // n / 4 is exact in fp32; _rn rounds half to even
  float mt = -CUDART_INF_F;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    ss[i] = scores[o + i];
    mt = fmaxf(mt, targets[o + i]);
  }
  mt = block_max(mt, red);
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    const float g = i < n ? expf(targets[o + i] - mt) : -CUDART_INF_F;
    if (i < n) gs[i] = g;
    key[i] = g;
    id[i] = i;
  }
  // IDCG_K from the gains in descending order
  block_sort_desc(key, id, P);
  float idcg = 0.f;
  for (int k = threadIdx.x; k < K; k += blockDim.x) idcg += key[k] / log2f(2.f + static_cast<float>(k));
  idcg = block_sum(idcg, red);                   // >= 1: the largest gain is exp(0) at rank 1
  // D(r_i): sort the scores (ties by index: the stable rank) and scatter each position's discount to its item
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    key[i] = i < n ? ss[i] : -CUDART_INF_F;
    id[i] = i;
  }
  block_sort_desc(key, id, P);
  for (int k = threadIdx.x; k < n; k += blockDim.x) key[id[k]] = k < K ? 1.f / log2f(2.f + static_cast<float>(k)) : 0.f;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) ts[i] = targets[o + i];
  __syncthreads();
  // The pair costs span many orders of magnitude (discounts of neighbouring deep ranks differ by ~1e-6): a thread's fp32 running sum of
  // ~n^2 / 512 of them would drop those below its half ulp and come out 3e-5 low at n = 8192, so it is kept in double.  The per-item
  // gradient sums n terms and stays in fp32.
  double part = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float si = ss[i], ti = ts[i], gi = gs[i], di = key[i];
    float g = 0.f;
    for (int j = 0; j < n; ++j) {
      const float d = sigma * (si - ss[j]);
      const float tj = ts[j];
      const float w = fabsf(gi - gs[j]) * fabsf(di - key[j]);
      if (ti > tj) {          // i should rank above j: C = w log(1 + exp(-sigma (s_i - s_j)))
        part += static_cast<double>(w * softplus_f(-d));
        g -= w * sigmoid_f(-d);
      } else if (ti < tj) {   // j should rank above i: the same pair seen from its lower item, gradient only
        g += w * sigmoid_f(d);
      }
    }
    dscore[o + i] = sigma * g * inv_norm / idcg;
  }
  const float total = block_sum(static_cast<float>(part), red);
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, total * inv_norm / idcg);
}

// ---------------------------------------------------------------------------------------
// pointwise: GaussDisLoss (loss.py:144-162), nn.MSELoss (train_listwise.py:166-167), the 'regression_exploss' key (276-281)
// ---------------------------------------------------------------------------------------
template <bool DET>
__global__ void __launch_bounds__(kLossThreads) k_pointwise(int kind, int N, const float* __restrict__ scores, const float* __restrict__ targets,
                                                            float inv_norm, float* __restrict__ loss, float* __restrict__ dscore) {
  __shared__ float red[32];
  float part = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    const float t = targets[i];
    if (kind == RR_LOSS_GAUSS) {
      const float mu = scores[2 * i], v = scores[2 * i + 1];
      const float d = mu - t;
      part += 0.5f * logf(2.f * 3.14159274101257324f) + 0.5f * logf(v) + d * d / (2.f * v);
      dscore[2 * i] = d / v * inv_norm;
      dscore[2 * i + 1] = (0.5f / v - d * d / (2.f * v * v)) * inv_norm;
    } else if (kind == RR_LOSS_LOGNORM) {      // Lognorm, loss.py:165-184: scores = (m, v), both positive
      const float m = scores[2 * i], v = scores[2 * i + 1];
      const float d = logf(m) - t;
      part += 0.5f * logf(2.f * 3.14159274101257324f) + 0.5f * logf(v * (m * m)) + d * d / (2.f * v);
      dscore[2 * i] = (1.f / m + d / (v * m)) * inv_norm;
      dscore[2 * i + 1] = (0.5f / v - d * d / (2.f * v * v)) * inv_norm;
    } else if (kind == RR_LOSS_EXPMSE) {       // mean((exp(t) - exp(s))^2), train_listwise.py:276-281
      const float e = expf(scores[i]);
      const float d = e - expf(t);
      part += d * d;
      dscore[i] = 2.f * d * e * inv_norm;
    } else {
      const float d = scores[i] - t;
      part += d * d;
      dscore[i] = 2.f * d * inv_norm;
    }
  }
  part = block_sum(part, red);
  if (threadIdx.x == 0) RR_PUT_LOSS(loss, part * inv_norm);
}

// deterministic mode: loss[0] = sum of the n block partials (each thread a strided run in order, then the fixed block_sum tree)
__global__ void __launch_bounds__(kLossThreads) k_sum_parts(int n, const float* __restrict__ parts, float* __restrict__ loss) {
  __shared__ float red[32];
  float v = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) v += parts[i];
  v = block_sum(v, red);
  if (threadIdx.x == 0) loss[0] = v;
}
// deterministic mode: dscore[i] = sum over column blocks y = 0, 1, ... of the NIG partials
__global__ void k_nig_dscore_sum(int N, int ny, const float* __restrict__ parts, float* __restrict__ dscore) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    float4 acc = ld_f4(parts + 4 * static_cast<size_t>(i));
    for (int y = 1; y < ny; ++y) acc = f4_add(acc, ld_f4(parts + 4 * (static_cast<size_t>(y) * N + i)));
    st_f4(dscore + 4 * static_cast<size_t>(i), acc);
  }
}

// DET (deterministic mode): every block stores its loss part to scratch (zeroed first: an empty group stores nothing), NIG its per-column-block
// gradient rows too, and k_sum_parts / k_nig_dscore_sum add them in block order.  The scratch is transient (cudaMallocAsync on s).
template <bool DET>
static int loss_launch(int kind, int N, int G, const float* scores, const float* targets, const int* seg_off, float norm, float sigma,
                       float* loss, float* dscore, cudaStream_t s, int max_group) {
  ProfScope prof_scope(KC_LOSS, s);
  RR_REQUIRE(N > 0 && scores && targets && loss && dscore, "loss: NULL argument or N <= 0");
  RR_REQUIRE(norm > 0.f, "loss: norm must be positive (got %g)", norm);
  RR_REQUIRE(max_group <= kMaxGroup, "loss: groups of up to %d candidates are supported (max_group %d)", kMaxGroup, max_group);
  // capacity of the per-group shared arrays of ListMLE / RankNet / LambdaRank: the next power of two >= max_group (the bitonic sort pads to it);
  // without a hint (max_group <= 0) kDefaultGroupCap.  A group larger than the capacity yields NaN, never an overrun.
  int cap = kDefaultGroupCap;
  if (max_group > 0) {
    cap = 64;
    while (cap < max_group) cap <<= 1;
  }
  const float inv = 1.f / norm;
  const dim3 nig_grid((N + kNigRows - 1) / kNigRows, (N + kNigCols - 1) / kNigCols);
  int pw_blocks = (N + kLossThreads - 1) / kLossThreads;
  if (pw_blocks > num_sms() * 4) pw_blocks = num_sms() * 4;
  long long n_parts = 0;
  switch (kind) {
    case RR_LOSS_NIG: n_parts = static_cast<long long>(nig_grid.x) * nig_grid.y; break;
    case RR_LOSS_GAUSS: case RR_LOSS_MSE: case RR_LOSS_LOGNORM: case RR_LOSS_EXPMSE: n_parts = pw_blocks; break;
    default: n_parts = G > 0 ? G : 0; break;
  }
  DetScratch ds;
  float* out = loss;        // where the kernels put their parts
  float* dparts = dscore;   // NIG: where the kernel puts its gradient rows
  if (DET) {
    const long long nig_floats = kind == RR_LOSS_NIG ? 4LL * N * nig_grid.y : 0;
    const long long parts_floats = (n_parts + 3) / 4 * 4;
    RR_TRY(det_scratch(&ds, nullptr, 0, (parts_floats + nig_floats) * static_cast<long long>(sizeof(float)), s));
    out = static_cast<float*>(ds.p);
    dparts = out + parts_floats;
    if (n_parts > 0) RR_CUDA(cudaMemsetAsync(out, 0, n_parts * sizeof(float), s));
  } else {
    RR_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), s));
  }
  switch (kind) {
    case RR_LOSS_LISTMLE:
    case RR_LOSS_LISTNET:
    case RR_LOSS_EVIDENTIAL:
    case RR_LOSS_RANKNET:
    case RR_LOSS_LISTMLE_DIS:
    case RR_LOSS_LISTNET_DIS:
    case RR_LOSS_LISTNET_UQ:
    case RR_LOSS_RANKNET_ACC:
    case RR_LOSS_DIRICHLET_UQ:
    case RR_LOSS_LAMBDARANK:
    case RR_LOSS_LAMBDARANK_TOP:
      RR_REQUIRE(G > 0 && seg_off, "loss: segmented kinds need seg_off and G > 0");
      {
        static PerDeviceOnce attr_set;           // up to 128 KB of dynamic shared memory for groups of up to kMaxGroup candidates
        if (attr_set.need()) {
          RR_CUDA(cudaFuncSetAttribute(k_listmle<false, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kMaxGroup * static_cast<int>(sizeof(float))));
          RR_CUDA(cudaFuncSetAttribute(k_listmle<true, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kMaxGroup * static_cast<int>(sizeof(float))));
          RR_CUDA(cudaFuncSetAttribute(k_ranknet<DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * kMaxGroup * static_cast<int>(sizeof(float))));
          RR_CUDA(cudaFuncSetAttribute(k_lambdarank<false, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kMaxGroup * static_cast<int>(sizeof(float))));
          RR_CUDA(cudaFuncSetAttribute(k_lambdarank<true, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kMaxGroup * static_cast<int>(sizeof(float))));
          attr_set.mark();
        }
      }
      if (kind == RR_LOSS_LISTMLE) k_listmle<false, DET><<<G, kLossThreads, 4 * cap * sizeof(float), s>>>(scores, targets, seg_off, inv, out, dscore, cap);
      else if (kind == RR_LOSS_LISTMLE_DIS) k_listmle<true, DET><<<G, kLossThreads, 4 * cap * sizeof(float), s>>>(scores, targets, seg_off, inv, out, dscore, cap);
      else if (kind == RR_LOSS_LISTNET) k_listnet<false, DET><<<G, kLossThreads, 0, s>>>(scores, targets, seg_off, inv, out, dscore);
      else if (kind == RR_LOSS_LISTNET_DIS) k_listnet<true, DET><<<G, kLossThreads, 0, s>>>(scores, targets, seg_off, inv, out, dscore);
      else if (kind == RR_LOSS_EVIDENTIAL) k_evidential<DET><<<G, kLossThreads, 0, s>>>(scores, targets, seg_off, inv, out, dscore);
      else if (kind == RR_LOSS_DIRICHLET_UQ) k_dirichlet_uq<DET><<<G, kLossThreads, 0, s>>>(scores, targets, seg_off, inv, sigma, out, dscore);
      else if (kind == RR_LOSS_LISTNET_UQ) k_listnet_uq<DET><<<G, kLossThreads, 0, s>>>(scores, targets, seg_off, inv, sigma, out, dscore);
      else if (kind == RR_LOSS_LAMBDARANK) k_lambdarank<false, DET><<<G, kLossThreads, 4 * cap * sizeof(float), s>>>(scores, targets, seg_off, inv, sigma, out, dscore, cap);
      else if (kind == RR_LOSS_LAMBDARANK_TOP) k_lambdarank<true, DET><<<G, kLossThreads, 4 * cap * sizeof(float), s>>>(scores, targets, seg_off, inv, sigma, out, dscore, cap);
      else k_ranknet<DET><<<G, kLossThreads, 2 * cap * sizeof(float), s>>>(scores, targets, seg_off, inv, sigma, kind == RR_LOSS_RANKNET_ACC ? 1.f : 2.f, out, dscore, cap);
      break;
    case RR_LOSS_NIG: {            // norm = N * N (the reference's mean over the broadcast matrix); `sigma` carries lam
      RR_REQUIRE((reinterpret_cast<uintptr_t>(scores) & 15) == 0, "loss: NIG scores must be 16-byte aligned");
      if (!DET) RR_CUDA(cudaMemsetAsync(dscore, 0, sizeof(float) * 4 * static_cast<size_t>(N), s));
      k_nig_allpairs<DET><<<nig_grid, kNigRows, 0, s>>>(N, scores, targets, inv, sigma, out, dparts);
      break;
    }
    case RR_LOSS_GAUSS:
    case RR_LOSS_MSE:
    case RR_LOSS_LOGNORM:
    case RR_LOSS_EXPMSE: {
      k_pointwise<DET><<<pw_blocks, kLossThreads, 0, s>>>(kind, N, scores, targets, inv, out, dscore);
      break;
    }
    default:
      return fail(RR_ERR_INVALID, "unknown loss kind %d", kind);
  }
  RR_LAUNCH_CHECK("loss kernel");
  if (DET) {
    k_sum_parts<<<1, kLossThreads, 0, s>>>(static_cast<int>(n_parts), out, loss);
    RR_LAUNCH_CHECK("k_sum_parts");
    if (kind == RR_LOSS_NIG) {
      int blocks = (N + 255) / 256;
      if (blocks > num_sms() * 4) blocks = num_sms() * 4;
      k_nig_dscore_sum<<<blocks, 256, 0, s>>>(N, static_cast<int>(nig_grid.y), dparts, dscore);
      RR_LAUNCH_CHECK("k_nig_dscore_sum");
    }
  }
  return RR_OK;
}

int loss_fwdbwd(int kind, int N, int G, const float* scores, const float* targets, const int* seg_off, float norm, float sigma,
                float* loss, float* dscore, cudaStream_t s, int max_group) {
  if (deterministic()) return loss_launch<true>(kind, N, G, scores, targets, seg_off, norm, sigma, loss, dscore, s, max_group);
  return loss_launch<false>(kind, N, G, scores, targets, seg_off, norm, sigma, loss, dscore, s, max_group);
}

int loss_max_group() { return kMaxGroup; }

// ---------------------------------------------------------------------------------------
// Per-group ranking metrics of the validation pass (eval.py:475-555 ranking_metrics, 76-177 evaluate_top_scores), one CTA per group:
// the reference pulls every group's scores to the host and sorts them in Python; here the scores never leave the device, only
// RR_METRIC_COLS doubles per group do.  Orders are the reference's stable descending sorts (ties keep the earlier item), expressed
// as ranks:  rank(i) = #{j : x_j > x_i} + #{j < i : x_j == x_i}.  With K = max(1, round_half_even(n * ratio)):
//   [0] predicted top-1 is the true top-1                    [1] |pred top-K  n  true top-K| / K
//   [2] predicted top-1 is inside the true top-K              [3] true top-1 is inside the predicted top-K
//   [4] NDCG@1   [5] the reference's NDCG@2 (both gains at one position, eval.py:544)   [6] NDCG@K   [7] NDCG@all
// NDCG = sum_k exp(target of the item predicted at k) / log2(k + 2)  over the ideal ordering's same sum (eval.py:460-472).
// ---------------------------------------------------------------------------------------
__device__ double block_sum_d(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.0;
  if (threadIdx.x < 32) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  }
  if (threadIdx.x == 0) red[0] = r;
  __syncthreads();
  r = red[0];
  __syncthreads();
  return r;
}
__global__ void __launch_bounds__(kLossThreads) k_rank_metrics(const float* __restrict__ scores, int score_ld, const double* __restrict__ targets,
                                                               const int* __restrict__ seg, int max_group, double ratio, double* __restrict__ out) {
  extern __shared__ double sm_d[];
  __shared__ double red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  double* res = out + static_cast<size_t>(blockIdx.x) * RR_METRIC_COLS;
  if (n <= 0 || n > max_group) {     // empty group: zeros; a group larger than the caller declared (shared memory was sized for max_group): NaN, never an overrun
    if (threadIdx.x < RR_METRIC_COLS) res[threadIdx.x] = n <= 0 ? 0.0 : CUDART_NAN;
    return;
  }
  double* sc = sm_d;
  double* tg = sm_d + n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    sc[i] = static_cast<double>(scores[static_cast<size_t>(o + i) * score_ld]);
    tg[i] = targets[o + i];
  }
  __syncthreads();
  const int K = max(1, static_cast<int>(rint(static_cast<double>(n) * ratio)));     // Python's round(): half to even
  double a[12];
#pragma unroll
  for (int q = 0; q < 12; ++q) a[q] = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double si = sc[i], ti = tg[i];
    int pr = 0, tr = 0;
    for (int j = 0; j < n; ++j) {
      const double sj = sc[j], tj = tg[j];
      pr += (sj > si) || (sj == si && j < i);
      tr += (tj > ti) || (tj == ti && j < i);
    }
    const double e = exp(ti);
    if (pr == 0) {
      a[0] += tr == 0;
      a[2] += tr < K;
      a[4] += e;                                    // gain at predicted position 0
    }
    if (tr == 0) {
      a[3] += pr < K;
      a[5] += e;                                    // ideal gain at position 0
    }
    a[1] += (pr < K && tr < K);
    if (pr < 2) a[6] += e;
    if (tr < 2) a[7] += e;
    const double dp = e / log2(static_cast<double>(pr) + 2.0), dt = e / log2(static_cast<double>(tr) + 2.0);
    if (pr < K) a[8] += dp;
    if (tr < K) a[9] += dt;
    a[10] += dp;
    a[11] += dt;
  }
#pragma unroll
  for (int q = 0; q < 12; ++q) a[q] = block_sum_d(a[q], red);
  if (threadIdx.x == 0) {
    res[0] = a[0];
    res[1] = a[1] / static_cast<double>(K);
    res[2] = a[2];
    res[3] = a[3];
    res[4] = a[4] / a[5];
    res[5] = a[6] / a[7];
    res[6] = a[8] / a[9];
    res[7] = a[10] / a[11];
  }
}

int rank_metrics(int N, int G, const float* scores, int score_ld, const double* targets, const int* seg_off, int max_group, double ratio,
                 double* out, cudaStream_t s) {
  ProfScope prof_scope(KC_LOSS, s);
  RR_REQUIRE(N > 0 && G > 0 && scores && targets && seg_off && out, "rank_metrics: NULL argument or empty input");
  RR_REQUIRE(score_ld >= 1, "rank_metrics: score_ld must be >= 1");
  RR_REQUIRE(ratio > 0.0 && ratio <= 1.0, "rank_metrics: ratio must lie in (0, 1] (got %g)", ratio);
  RR_REQUIRE(max_group >= 1 && max_group <= kMaxMetricGroup, "rank_metrics: largest group %d outside [1, %d]", max_group, kMaxMetricGroup);
  const size_t smem = 2 * sizeof(double) * static_cast<size_t>(max_group);
  static PerDeviceOnce attr_set;
  if (attr_set.need()) {
    RR_CUDA(cudaFuncSetAttribute(k_rank_metrics, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * sizeof(double) * kMaxMetricGroup));
    attr_set.mark();
  }
  k_rank_metrics<<<G, kLossThreads, smem, s>>>(scores, score_ld, targets, seg_off, max_group, ratio, out);
  RR_LAUNCH_CHECK("rank_metrics kernel");
  return RR_OK;
}

// ---------------------------------------------------------------------------------------
// Prediction: per-item ranking statistics over T score samples (MC dropout; T = 1 for one deterministic pass), one CTA per group.
// Ranks use the rule of k_rank_metrics, 1-based:  rank(i) = 1 + #{j : x_j > x_i} + #{j < i : x_j == x_i}.
// Sample t of the group is staged in shared memory (n floats: the comparisons and the max are exact on floats), the within-group
// softmax is shifted by the group maximum and taken in double.  The group's n = 8192 items cannot keep five double accumulators each
// on chip, so the items are taken in passes of kPredictItems * blockDim.x: in a pass every thread owns kPredictItems items and keeps
// their accumulators in registers across the whole T loop; a later pass streams the T samples again.  Sums are in double, the reductions
// are the fixed block_sum_d tree and nothing is atomic, so a repeated call is bit-identical.
// ---------------------------------------------------------------------------------------
constexpr int kPredictItems = 4;

__global__ void __launch_bounds__(kLossThreads) k_rank_predict(int T, const float* __restrict__ scores, long long sample_stride, int score_ld,
                                                               const int* __restrict__ seg, int max_group, float* __restrict__ out) {
  extern __shared__ float pred_sm[];             // x | mean, n entries each
  __shared__ double red[32];
  const int o = seg[blockIdx.x], n = seg[blockIdx.x + 1] - o;
  if (n <= 0) return;
  float* rows = out + static_cast<size_t>(o) * RR_PREDICT_COLS;
  if (n > max_group) {           // shared memory was sized for max_group: NaN rows, never an overrun
    for (int i = threadIdx.x; i < n * RR_PREDICT_COLS; i += blockDim.x) rows[i] = CUDART_NAN_F;
    return;
  }
  float* x = pred_sm;
  float* mean = pred_sm + n;
  const float* base = scores + static_cast<size_t>(o) * score_ld;
  const double dt = static_cast<double>(T);
  for (int p0 = 0; p0 < n; p0 += kPredictItems * blockDim.x) {
    double sum[kPredictItems], dev[kPredictItems], dev2[kPredictItems], prob[kPredictItems], rsum[kPredictItems];
    float x0[kPredictItems];
    int top1[kPredictItems];
#pragma unroll
    for (int k = 0; k < kPredictItems; ++k) {
      sum[k] = dev[k] = dev2[k] = prob[k] = rsum[k] = 0.0;
      x0[k] = 0.f;
      top1[k] = 0;
    }
    for (int t = 0; t < T; ++t) {
      const float* st = base + static_cast<size_t>(t) * sample_stride;
      float mx = -CUDART_INF_F;
      __syncthreads();                           // the previous sample's x[] has been read by everyone
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float v = st[static_cast<size_t>(i) * score_ld];
        x[i] = v;
        mx = fmaxf(mx, v);
      }
      mx = block_max(mx, reinterpret_cast<float*>(red));     // synchronises: x[] is complete
      const double dmx = static_cast<double>(mx);
      double z = 0.0;
      for (int i = threadIdx.x; i < n; i += blockDim.x) z += exp(static_cast<double>(x[i]) - dmx);
      z = block_sum_d(z, red);
      const double inv_z = 1.0 / z;
      float xi[kPredictItems];
      int cnt[kPredictItems];
#pragma unroll
      for (int k = 0; k < kPredictItems; ++k) {
        const int i = p0 + k * blockDim.x + threadIdx.x;
        xi[k] = i < n ? x[i] : 0.f;
        cnt[k] = 1;
      }
      for (int j = 0; j < n; ++j) {
        const float xj = x[j];
#pragma unroll
        for (int k = 0; k < kPredictItems; ++k) {
          const int i = p0 + k * blockDim.x + threadIdx.x;
          cnt[k] += (xj > xi[k]) || (xj == xi[k] && j < i);
        }
      }
#pragma unroll
      for (int k = 0; k < kPredictItems; ++k) {
        if (t == 0) x0[k] = xi[k];
        const double v = static_cast<double>(xi[k]), d = v - static_cast<double>(x0[k]);
        sum[k] += v;
        dev[k] += d;
        dev2[k] += d * d;
        prob[k] += exp(v - dmx) * inv_z;
        rsum[k] += static_cast<double>(cnt[k]);
        top1[k] += cnt[k] == 1;
      }
    }
#pragma unroll
    for (int k = 0; k < kPredictItems; ++k) {
      const int i = p0 + k * blockDim.x + threadIdx.x;
      if (i < n) {
        const double var = fmax((dev2[k] - dev[k] * dev[k] / dt) / dt, 0.0);    // about the first sample: no cancellation
        const float m = static_cast<float>(sum[k] / dt);
        float* r = rows + static_cast<size_t>(i) * RR_PREDICT_COLS;
        r[0] = m;
        r[1] = static_cast<float>(sqrt(var));
        r[3] = static_cast<float>(prob[k] / dt);
        r[4] = static_cast<float>(static_cast<double>(top1[k]) / dt);
        r[5] = static_cast<float>(rsum[k] / dt);
        mean[i] = m;
      }
    }
  }
  __syncthreads();
  // rank of the mean score: the fp32 value of column 0, so the rank is the stable order of the returned scores
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float mi = mean[i];
    int c = 1;
    for (int j = 0; j < n; ++j) c += (mean[j] > mi) || (mean[j] == mi && j < i);
    rows[static_cast<size_t>(i) * RR_PREDICT_COLS + 2] = static_cast<float>(c);
  }
}

int rank_predict(int N, int G, int T, const float* scores, long long sample_stride, int score_ld, const int* seg_off, int max_group, float* out,
                 cudaStream_t s) {
  ProfScope prof_scope(KC_LOSS, s);
  RR_REQUIRE(N > 0 && G > 0 && scores && seg_off && out, "rank_predict: NULL argument or empty input");
  RR_REQUIRE(T >= 1, "rank_predict: T must be >= 1 (got %d)", T);
  RR_REQUIRE(score_ld >= 1 && sample_stride >= 0, "rank_predict: score_ld must be >= 1 and sample_stride >= 0");
  RR_REQUIRE(max_group >= 1 && max_group <= kMaxGroup, "rank_predict: largest group %d outside [1, %d]", max_group, kMaxGroup);
  const size_t smem = 2 * sizeof(float) * static_cast<size_t>(max_group);
  static PerDeviceOnce attr_set;
  if (attr_set.need()) {
    RR_CUDA(cudaFuncSetAttribute(k_rank_predict, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * sizeof(float) * kMaxGroup));
    attr_set.mark();
  }
  k_rank_predict<<<G, kLossThreads, smem, s>>>(T, scores, sample_stride, score_ld, seg_off, max_group, out);
  RR_LAUNCH_CHECK("rank_predict kernel");
  return RR_OK;
}

}  // namespace rr
