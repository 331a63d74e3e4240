// fp32 SIMT GEMM family: the exact-fp32 implementation of the nn.Linear call sites
// (mpn.py:80,94,104,194,211,218; base_model.py:40-56) -- forward with fused
// bias/residual/ReLU/dropout epilogue and concat-free two-source K, dgrad, and split-K
// wgrad with fused bias gradient.  Operands are the padded, 16-byte-aligned layouts of
// rr_model.cu, so every global access is a float4.
//
// C(m,n) = sum_src sum_k A(m,k) * B(k,n)
//   A_KC : A(m,k) = A[m*lda + k]   else  A(m,k) = A[k*lda + m]
//   B_KC : B(k,n) = B[n*ldb + k]   else  B(k,n) = B[k*ldb + n]
#include "rr_common.cuh"

namespace rr {

constexpr int BM = 128, BN = 64, BK = 16, NT = 256;
constexpr int APAD = BM + 4, BPAD = BN + 4;

// EPI_SLAB: EPI_ATOMIC of deterministic mode, slab z STORES its tile to C + z * slab_stride and its bias partial to dbias + z * M
enum { EPI_FWD = 0, EPI_STORE = 1, EPI_ACCUM = 2, EPI_ATOMIC = 3, EPI_SLAB = 4 };

struct GemmSrc {
  const float* A;
  const float* B;
  int lda, ldb, K;
};

struct GemmArgs {
  GemmSrc src[2];
  int nsrc;
  int M, N;
  float* C;
  int ldc;
  // EPI_FWD
  const float* bias;
  const float* resid;
  int ldr;
  int relu;
  float p, inv_keep;
  uint64_t seed, stream_id;
  // EPI_ATOMIC (wgrad)
  float* dbias;
  int k_chunk;  // reduction rows per blockIdx.z
  long long slab_stride;  // EPI_SLAB
};

template <bool A_KC>
__device__ __forceinline__ void load_a(const GemmSrc& s, int M, int m0, int k0, int kend, int t, float4 (&r)[2]) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    if (A_KC) {
      const int row = m0 + (t >> 2) + i * 64, k = k0 + ((t & 3) << 2);
      r[i] = (row < M && k < kend) ? ld_f4(s.A + static_cast<size_t>(row) * s.lda + k) : f4_zero();
    } else {
      const int k = k0 + (t >> 5) + i * 8, m = m0 + ((t & 31) << 2);
      r[i] = (k < kend && m < M) ? ld_f4(s.A + static_cast<size_t>(k) * s.lda + m) : f4_zero();
    }
  }
}
template <bool A_KC>
__device__ __forceinline__ void store_a(float (*As)[APAD], int t, const float4 (&r)[2]) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    if (A_KC) {
      const int row = (t >> 2) + i * 64, k = (t & 3) << 2;
      As[k + 0][row] = r[i].x;
      As[k + 1][row] = r[i].y;
      As[k + 2][row] = r[i].z;
      As[k + 3][row] = r[i].w;
    } else {
      const int k = (t >> 5) + i * 8, m = (t & 31) << 2;
      *reinterpret_cast<float4*>(&As[k][m]) = r[i];
    }
  }
}
template <bool B_KC>
__device__ __forceinline__ float4 load_b(const GemmSrc& s, int N, int n0, int k0, int kend, int t) {
  if (B_KC) {
    const int n = n0 + (t >> 2), k = k0 + ((t & 3) << 2);
    return (n < N && k < kend) ? ld_f4(s.B + static_cast<size_t>(n) * s.ldb + k) : f4_zero();
  } else {
    const int k = k0 + (t >> 4), n = n0 + ((t & 15) << 2);
    return (k < kend && n < N) ? ld_f4(s.B + static_cast<size_t>(k) * s.ldb + n) : f4_zero();
  }
}
template <bool B_KC>
__device__ __forceinline__ void store_b(float (*Bs)[BPAD], int t, float4 r) {
  if (B_KC) {
    const int n = t >> 2, k = (t & 3) << 2;
    Bs[k + 0][n] = r.x;
    Bs[k + 1][n] = r.y;
    Bs[k + 2][n] = r.z;
    Bs[k + 3][n] = r.w;
  } else {
    const int k = t >> 4, n = (t & 15) << 2;
    *reinterpret_cast<float4*>(&Bs[k][n]) = r;
  }
}

template <bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__(NT, 2) k_gemm(GemmArgs g) {
  __shared__ __align__(16) float As[BK][APAD];
  __shared__ __align__(16) float Bs[BK][BPAD];
  const int t = threadIdx.x;
  const int ty = t >> 4, tx = t & 15;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bias_acc = 0.f;
  const bool do_bias = (EPI == EPI_ATOMIC || EPI == EPI_SLAB) && g.dbias != nullptr && blockIdx.y == 0;

  for (int s = 0; s < g.nsrc; ++s) {
    const GemmSrc src = g.src[s];
    int kbeg = 0, kend = src.K;
    if (EPI == EPI_ATOMIC || EPI == EPI_SLAB) {
      kbeg = blockIdx.z * g.k_chunk;
      kend = min(src.K, kbeg + g.k_chunk);
    }
    if (kbeg >= kend) continue;
    float4 ra[2], rb;
    load_a<A_KC>(src, g.M, m0, kbeg, kend, t, ra);
    rb = load_b<B_KC>(src, g.N, n0, kbeg, kend, t);
    for (int k0 = kbeg; k0 < kend; k0 += BK) {
      __syncthreads();
      store_a<A_KC>(As, t, ra);
      store_b<B_KC>(Bs, t, rb);
      __syncthreads();
      if (k0 + BK < kend) {
        load_a<A_KC>(src, g.M, m0, k0 + BK, kend, t, ra);
        rb = load_b<B_KC>(src, g.N, n0, k0 + BK, kend, t);
      }
      if (do_bias && t < BM) {
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) bias_acc += As[kk][t];
      }
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
        const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
      }
    }
  }

  const int n = n0 + tx * 4;
  if constexpr (EPI == EPI_SLAB) {
    if (do_bias && t < BM && m0 + t < g.M) g.dbias[static_cast<size_t>(blockIdx.z) * g.M + m0 + t] = bias_acc;
  } else {
    if (do_bias && t < BM && m0 + t < g.M) atomicAdd(g.dbias + m0 + t, bias_acc);
  }
  if (n >= g.N) return;
  float4 bv = f4_zero();
  if (EPI == EPI_FWD && g.bias) bv = ld_f4(g.bias + n);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + ty * 8 + i;
    if (m >= g.M) break;
    float4 v = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    float* cp = g.C + static_cast<size_t>(m) * g.ldc + n;
    if constexpr (EPI == EPI_SLAB) {
      st_f4(cp + blockIdx.z * g.slab_stride, v);
    } else if (EPI == EPI_FWD) {
      v = f4_add(v, bv);
      if (g.resid) v = f4_add(v, ld_f4(g.resid + static_cast<size_t>(m) * g.ldr + n));
      if (g.relu) v = f4_relu(v);
      if (g.p > 0.f) v = dropout4(v, g.p, g.inv_keep, g.seed, g.stream_id, (static_cast<uint64_t>(m) * g.ldc + n) >> 2);
      st_f4(cp, v);
    } else if (EPI == EPI_STORE) {
      st_f4(cp, v);
    } else if (EPI == EPI_ACCUM) {
      st_f4(cp, f4_add(v, *reinterpret_cast<const float4*>(cp)));
    } else {
      red_add_f4(cp, v);
    }
  }
}


int simt_fwd(int M, int n, const float* X1, int ldx1, const float* W1, int k1, const float* X2, int ldx2, const float* W2, int k2, const float* bias,
             const float* resid, int ldr, float* Y, int ldy, int flags, float p, uint64_t seed, uint64_t stream_id, cudaStream_t s) {
  ProfScope prof_scope(KC_GEMM_FWD, s);
  RR_REQUIRE(M >= 0 && n > 0 && (n & 3) == 0 && k1 > 0 && (k1 & 3) == 0 && (k2 & 3) == 0, "linear_fwd: M %d n %d k1 %d k2 %d (n, k multiples of 4)", M, n, k1, k2);
  RR_TRY(check_mat("X1", X1, ldx1));
  RR_TRY(check_mat("W1", W1, k1));
  RR_TRY(check_mat("Y", Y, ldy));
  if (X2) {
    RR_TRY(check_mat("X2", X2, ldx2));
    RR_TRY(check_mat("W2", W2, k2));
  }
  if (resid) RR_TRY(check_mat("residual", resid, ldr));
  if (bias) RR_REQUIRE(aligned16(bias), "bias must be 16-byte aligned");
  RR_REQUIRE(p >= 0.f && p < 1.f, "dropout p must be in [0,1)");
  if (M == 0) return RR_OK;
  GemmArgs g{};
  g.src[0] = {X1, W1, ldx1, k1, k1};
  g.nsrc = 1;
  if (X2 && k2 > 0) {
    g.src[1] = {X2, W2, ldx2, k2, k2};
    g.nsrc = 2;
  }
  g.M = M;
  g.N = n;
  g.C = Y;
  g.ldc = ldy;
  g.bias = bias;
  g.resid = resid;
  g.ldr = ldr;
  g.relu = flags & 1;
  g.p = (flags & 2) ? p : 0.f;
  g.inv_keep = g.p > 0.f ? 1.f / (1.f - g.p) : 1.f;
  g.seed = seed;
  g.stream_id = stream_id;
  dim3 grid((M + BM - 1) / BM, (n + BN - 1) / BN);
  k_gemm<true, true, EPI_FWD><<<grid, NT, 0, s>>>(g);
  RR_LAUNCH_CHECK("k_gemm<fwd>");
  return RR_OK;
}

int simt_dgrad(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx, int accumulate, cudaStream_t s) {
  ProfScope prof_scope(KC_GEMM_DGRAD, s);
  RR_REQUIRE(M >= 0 && n > 0 && k > 0 && (n & 3) == 0 && (k & 3) == 0, "linear_dgrad: M %d n %d k %d", M, n, k);
  RR_TRY(check_mat("dZ", dZ, lddz));
  RR_TRY(check_mat("W", W, ldw));
  RR_TRY(check_mat("dX", dX, lddx));
  if (M == 0) return RR_OK;
  GemmArgs g{};
  g.src[0] = {dZ, W, lddz, ldw, n};
  g.nsrc = 1;
  g.M = M;
  g.N = k;
  g.C = dX;
  g.ldc = lddx;
  dim3 grid((M + BM - 1) / BM, (k + BN - 1) / BN);
  if (accumulate) k_gemm<true, false, EPI_ACCUM><<<grid, NT, 0, s>>>(g);
  else k_gemm<true, false, EPI_STORE><<<grid, NT, 0, s>>>(g);
  RR_LAUNCH_CHECK("k_gemm<dgrad>");
  return RR_OK;
}

int simt_wgrad_splits(int M, int n, int k, int* chunk_out) {
  const int tiles = ((n + BM - 1) / BM) * ((k + BN - 1) / BN);
  int splits = (num_sms() * 2 + tiles - 1) / tiles;
  const int max_splits = (M + BK * 8 - 1) / (BK * 8);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  int chunk = (M + splits - 1) / splits;
  chunk = (chunk + BK - 1) / BK * BK;
  if (chunk_out) *chunk_out = chunk;
  return (M + chunk - 1) / chunk;
}

int simt_wgrad(int M, int n, int k, const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw, float* dbias, cudaStream_t s, float* slab,
               int* n_splits) {
  ProfScope prof_scope(KC_GEMM_WGRAD, s);
  GemmArgs g{};
  g.src[0] = {dZ, X, lddz, ldx, M};  // reduction runs over the M rows
  g.nsrc = 1;
  g.M = n;
  g.N = k;
  g.C = dW;
  g.ldc = lddw;
  g.dbias = dbias;
  int chunk = 0;
  const int splits = simt_wgrad_splits(M, n, k, &chunk);
  g.k_chunk = chunk;
  dim3 grid((n + BM - 1) / BM, (k + BN - 1) / BN, splits);
  if (slab) {
    g.C = slab;
    g.ldc = k;
    g.slab_stride = static_cast<long long>(n) * k;
    g.dbias = dbias ? slab + splits * g.slab_stride : nullptr;
    *n_splits = splits;
    k_gemm<false, false, EPI_SLAB><<<grid, NT, 0, s>>>(g);
  } else {
    k_gemm<false, false, EPI_ATOMIC><<<grid, NT, 0, s>>>(g);
  }
  RR_LAUNCH_CHECK("k_gemm<wgrad>");
  return RR_OK;
}

}  // namespace rr
