// Whole-model forward / backward of ReactionModel (models/base_model.py:150-171):
//   MPN(reactants), MPN(products)  ->  p - r  ->  MPNDiff over the product graph
//   -> scope-mean readout || add_features -> FFN -> head
// sequenced on one stream out of a caller-provided workspace.  Nothing is allocated here.
//
// Parameters arrive in the reference's state_dict layout and are re-packed once per call
// into zero-padded, 16-byte-aligned matrices; concatenated inputs of the reference
// ([f_atoms || a_message], [nei_message || nei_f_bonds], [diff || a_message]) are never
// materialised: their weight matrices are split column-wise and the GEMM accumulates two
// sources.  Gradients are produced in the padded layout and un-packed at the end.
#include "rr_common.cuh"

namespace rr {

static inline int pad16(int x) { return (x + 15) / 16 * 16; }
int padded(int w) { return pad16(w); }

constexpr int kMaxDepth = 16;

// ---- packed parameter layout (float offsets) ---------------------------------------------
// Every sub-module has its own padded width: hpe (encoder, and the difference d = p - r it produces), hpd (diff encoder), hpf (FFN hidden
// layers); the readout vector [mean(hid2) || add_features] is vp = pad16(hd + add_features) wide.
struct PackedLayout {
  int hpe, hpd, hpf, vp, F;
  size_t enc_Wi, enc_bi, enc_Wh, enc_bh, enc_Wo_a, enc_Wo_m, enc_bo;
  size_t dif_Wi, dif_bi, dif_Wh_m, dif_Wh_f, dif_bh, dif_Wo_d, dif_Wo_m, dif_bo;
  size_t ffn_W[RR_MAX_FFN], ffn_b[RR_MAX_FFN];
  int ffn_in[RR_MAX_FFN], ffn_out[RR_MAX_FFN];  // padded dims
  // transposed copies [in_pad, out_pad] of every weight that has a dgrad: K-major B operand of dX = dZ W on tcgen05
  size_t enc_Wh_T, enc_Wo_m_T, dif_Wi_T, dif_Wh_m_T, dif_Wo_d_T, dif_Wo_m_T, ffn_W_T[RR_MAX_FFN];
  size_t total;       // floats, transposed copies included
  size_t grad_total;  // floats of the gradient image (no transposed copies)
};

static PackedLayout make_packed(const rr_model_cfg_ex& c) {
  PackedLayout L{};
  L.hpe = pad16(c.base.hidden);
  L.hpd = pad16(c.diff_hidden);
  L.hpf = pad16(c.ffn_hidden);
  L.vp = pad16(c.diff_hidden + c.base.add_features);
  L.F = c.base.ffn_depth;
  size_t o = 0;
  auto take = [&](size_t n) {
    size_t r = o;
    o += (n + 63) / 64 * 64;
    return r;
  };
  const size_t he = L.hpe, hd = L.hpd;
  L.enc_Wi = take(he * RR_FB_LD); L.enc_bi = take(he);
  L.enc_Wh = take(he * he);       L.enc_bh = take(he);
  L.enc_Wo_a = take(he * RR_FA_LD); L.enc_Wo_m = take(he * he); L.enc_bo = take(he);
  L.dif_Wi = take(hd * he);       L.dif_bi = take(hd);
  L.dif_Wh_m = take(hd * hd);     L.dif_Wh_f = take(hd * RR_FB_LD); L.dif_bh = take(hd);
  L.dif_Wo_d = take(hd * he);     L.dif_Wo_m = take(hd * hd);       L.dif_bo = take(hd);
  for (int l = 0; l < L.F; ++l) {
    L.ffn_in[l] = (l == 0) ? L.vp : L.hpf;
    L.ffn_out[l] = (l == L.F - 1) ? RR_OUT_LD : L.hpf;
    L.ffn_W[l] = take(static_cast<size_t>(L.ffn_in[l]) * L.ffn_out[l]);
    L.ffn_b[l] = take(L.ffn_out[l]);
  }
  L.grad_total = o;
  L.enc_Wh_T = take(he * he);
  L.enc_Wo_m_T = take(he * he);
  L.dif_Wi_T = take(he * hd);
  L.dif_Wh_m_T = take(hd * hd);
  L.dif_Wo_d_T = take(he * hd);
  L.dif_Wo_m_T = take(hd * hd);
  for (int l = 0; l < L.F; ++l) L.ffn_W_T[l] = take(static_cast<size_t>(L.ffn_in[l]) * L.ffn_out[l]);
  L.total = o;
  return L;
}

struct PackEntry {
  float* ref;        // state_dict-layout tensor (source when packing, destination when un-packing)
  long long packed;  // float offset in the packed buffer
  int rows, cols, ref_ld, ref_col0, packed_ld;
  int transpose;     // packed[c][r] = ref[r][c]
};
constexpr int kMaxEntries = 48;
struct PackTable {
  PackEntry e[kMaxEntries];
  int n;
};

static PackTable make_table(const rr_model_cfg_ex& c, const PackedLayout& L, const rr_params& w, bool with_transposes) {
  PackTable T{};
  const int he = c.base.hidden, hd = c.diff_hidden, hf = c.ffn_hidden, hpe = L.hpe, hpd = L.hpd;
  auto add = [&](float* ref, size_t off, int rows, int cols, int ref_ld, int col0, int pld) {
    if (ref == nullptr) return;
    T.e[T.n++] = PackEntry{ref, static_cast<long long>(off), rows, cols, ref_ld, col0, pld, 0};
  };
  auto add_t = [&](float* ref, size_t off, int rows, int cols, int ref_ld, int col0, int pld) {
    if (ref == nullptr || !with_transposes) return;
    T.e[T.n++] = PackEntry{ref, static_cast<long long>(off), rows, cols, ref_ld, col0, pld, 1};
  };
  add(w.enc_Wi, L.enc_Wi, he, RR_FBOND_TOTAL, RR_FBOND_TOTAL, 0, RR_FB_LD);
  add(w.enc_bi, L.enc_bi, 1, he, he, 0, hpe);
  add(w.enc_Wh, L.enc_Wh, he, he, he, 0, hpe);
  add(w.enc_bh, L.enc_bh, 1, he, he, 0, hpe);
  add(w.enc_Wo, L.enc_Wo_a, he, RR_ATOM_FDIM, RR_ATOM_FDIM + he, 0, RR_FA_LD);
  add(w.enc_Wo, L.enc_Wo_m, he, he, RR_ATOM_FDIM + he, RR_ATOM_FDIM, hpe);
  add(w.enc_bo, L.enc_bo, 1, he, he, 0, hpe);
  add(w.dif_Wi, L.dif_Wi, hd, he, he, 0, hpe);
  add(w.dif_bi, L.dif_bi, 1, hd, hd, 0, hpd);
  add(w.dif_Wh, L.dif_Wh_m, hd, hd, hd + RR_FBOND_TOTAL, 0, hpd);
  add(w.dif_Wh, L.dif_Wh_f, hd, RR_FBOND_TOTAL, hd + RR_FBOND_TOTAL, hd, RR_FB_LD);
  add(w.dif_bh, L.dif_bh, 1, hd, hd, 0, hpd);
  add(w.dif_Wo, L.dif_Wo_d, hd, he, he + hd, 0, hpe);
  add(w.dif_Wo, L.dif_Wo_m, hd, hd, he + hd, he, hpd);
  add(w.dif_bo, L.dif_bo, 1, hd, hd, 0, hpd);
  for (int l = 0; l < L.F; ++l) {
    const int in = (l == 0) ? hd + c.base.add_features : hf;
    const int out = (l == L.F - 1) ? c.base.task_num : hf;
    add(w.ffn_W[l], L.ffn_W[l], out, in, in, 0, L.ffn_in[l]);
    add(w.ffn_b[l], L.ffn_b[l], 1, out, out, 0, L.ffn_out[l]);
    add_t(w.ffn_W[l], L.ffn_W_T[l], out, in, in, 0, L.ffn_out[l]);
  }
  add_t(w.enc_Wh, L.enc_Wh_T, he, he, he, 0, hpe);
  add_t(w.enc_Wo, L.enc_Wo_m_T, he, he, RR_ATOM_FDIM + he, RR_ATOM_FDIM, hpe);
  add_t(w.dif_Wi, L.dif_Wi_T, hd, he, he, 0, hpd);
  add_t(w.dif_Wh, L.dif_Wh_m_T, hd, hd, hd + RR_FBOND_TOTAL, 0, hpd);
  add_t(w.dif_Wo, L.dif_Wo_d_T, hd, he, he + hd, 0, hpd);
  add_t(w.dif_Wo, L.dif_Wo_m_T, hd, hd, he + hd, he, hpd);
  return T;
}

// direction 0: packed <- ref (pack);  1: ref <- packed (un-pack gradients)
// Packing also writes the TF32 split of every value (hi = nearest TF32, lo = v - hi) into the images hi_off / lo_off floats further on:
// the tcgen05 GEMMs then TMA-load both halves of the B operand instead of splitting the same weight tile once per row tile.
// The same values as bf16 pairs (hi = bf16(v), lo = bf16(v - hi)) go to two uint16 images (bhi / blo, same element offsets) for the
// backward GEMMs' 3 x bf16 split.
__device__ __forceinline__ uint16_t bf16_rn(float v) {
  uint16_t r;
  asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(r) : "f"(v));
  return r;
}
__global__ void k_pack(PackTable T, float* __restrict__ packed, int direction, long long hi_off, long long lo_off, uint16_t* __restrict__ bhi,
                       uint16_t* __restrict__ blo) {
  const PackEntry e = T.e[blockIdx.y];
  const long long n = static_cast<long long>(e.rows) * e.cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / e.cols), c = static_cast<int>(i - static_cast<long long>(r) * e.cols);
    float* pp = packed + e.packed + (e.transpose ? static_cast<long long>(c) * e.packed_ld + r : static_cast<long long>(r) * e.packed_ld + c);
    float* rp = e.ref + static_cast<long long>(r) * e.ref_ld + e.ref_col0 + c;
    if (direction == 0) {
      const float v = *rp;
      const float hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
      *pp = v;
      pp[hi_off] = hi;
      pp[lo_off] = v - hi;
      const uint16_t b1 = bf16_rn(v);
      bhi[pp - packed] = b1;
      blo[pp - packed] = bf16_rn(v - __uint_as_float(static_cast<uint32_t>(b1) << 16));
    } else {
      *rp = *pp;
    }
  }
}

// ---- head (base_model.py:59-108) -----------------------------------------------------------
__device__ __forceinline__ float softplus_t(float x) { return x > 20.f ? x : log1pf(expf(x)); }  // nn.Softplus(beta=1, threshold=20)
__global__ void k_head_fwd(int N, int task, int head, const float* __restrict__ z, float* __restrict__ out) {
  const int half = task >> 1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * task; i += gridDim.x * blockDim.x) {
    const int r = i / task, c = i - r * task;
    const float* zr = z + static_cast<size_t>(r) * RR_OUT_LD;
    float v;
    if (head == RR_HEAD_RAW) v = zr[c];
    else if (head == RR_HEAD_SOFTPLUS) v = softplus_t(zr[c]);
    else if (head == RR_HEAD_SOFTPLUS_P1) v = softplus_t(zr[c]) + 1.f;
    else if (head == RR_HEAD_NIG) {  // stack((mu, lambda, alpha, beta), dim=2).view(...): column c = 4 j + k reads quarter k, entry j
      const int j = c >> 2, k = c & 3, quarter = task >> 2;
      const float zc = zr[k * quarter + j];
      v = k == 0 ? zc : (k == 2 ? softplus_t(zc) + 1e-6f + 1.f : softplus_t(zc) + 1e-6f);
    } else {  // stack((first half, f(second half)), dim=2).view(...)  -> interleaved columns
      const int j = c >> 1;
      if ((c & 1) == 0) v = head == RR_HEAD_LOGNORM ? softplus_t(zr[j]) + 1e-6f : zr[j];
      else v = softplus_t(zr[half + j]) + (head == RR_HEAD_GAUSS_SOFTPLUS ? 0.f : 1e-6f);
    }
    out[i] = v;
  }
}
__global__ void k_head_bwd(int N, int task, int head, const float* __restrict__ z, const float* __restrict__ dout, float* __restrict__ dz) {
  const int half = task >> 1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * RR_OUT_LD; i += gridDim.x * blockDim.x) {
    const int r = i / RR_OUT_LD, c = i - r * RR_OUT_LD;
    float v = 0.f;
    if (c < task) {
      const float zc = z[i];
      const float sg = zc > 20.f ? 1.f : 1.f / (1.f + expf(-zc));
      const float* dr = dout + static_cast<size_t>(r) * task;
      if (head == RR_HEAD_RAW) v = dr[c];
      else if (head == RR_HEAD_SOFTPLUS || head == RR_HEAD_SOFTPLUS_P1) v = dr[c] * sg;
      else if (head == RR_HEAD_NIG) {
        const int quarter = task >> 2, k = c / quarter, j = c - k * quarter;
        v = dr[4 * j + k] * (k == 0 ? 1.f : sg);
      } else v = (c < half) ? dr[2 * c] * (head == RR_HEAD_LOGNORM ? sg : 1.f) : dr[2 * (c - half) + 1] * sg;
    }
    dz[i] = v;
  }
}

// ---- joint graph ------------------------------------------------------------------------------
// Index tables of the concatenation [reactant batch | product batch] in joint row space: the reactant part is copied, the product part
// is shifted by the reactant batch's row counts (valid slots only: an unused slot stays 0 and is never read, its multiplicity lives in
// rr_atom_meta).  Every segment keeps its own padding rows and max_num_bonds, so the joint launch computes exactly what two launches did.
__global__ void k_join_tables(rr_graph r, rr_graph p, rr_graph J) {
  const int A_r = r.n_atoms, B_r = r.n_bonds;
  int4* meta = reinterpret_cast<int4*>(const_cast<rr_atom_meta*>(J.a_meta));
  int* a2b = const_cast<int*>(J.a2b);
  int* a2r = const_cast<int*>(J.a2b_rev);
  int* a2a = const_cast<int*>(J.a2a);
  for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < J.n_atoms; a += gridDim.x * blockDim.x) {
    const bool second = a >= A_r;
    const rr_graph& g = second ? p : r;
    const int la = second ? a - A_r : a, ob = second ? B_r : 0, oa = second ? A_r : 0;
    int4 m = __ldg(reinterpret_cast<const int4*>(g.a_meta) + la);
    const int deg = m.x & 0xff;
    m.z += ob;
    m.w += oa;
    meta[a] = m;
    const size_t src = static_cast<size_t>(la) * g.wmax, dst = static_cast<size_t>(a) * J.wmax;
    for (int k = 0; k < J.wmax; ++k) {
      const bool v = k < deg;
      a2b[dst + k] = v ? __ldg(g.a2b + src + k) + ob : 0;
      a2r[dst + k] = v ? __ldg(g.a2b_rev + src + k) + ob : 0;
      a2a[dst + k] = v ? __ldg(g.a2a + src + k) + oa : 0;
    }
  }
  for (int sgm = blockIdx.x * blockDim.x + threadIdx.x; sgm < J.n_segments; sgm += gridDim.x * blockDim.x) {
    const bool second = sgm >= r.n_segments;
    const int ls = second ? sgm - r.n_segments : sgm;
    const_cast<int*>(J.pad_bonds)[sgm] = second ? __ldg(p.pad_bonds + ls) + B_r : __ldg(r.pad_bonds + ls);
    const_cast<int*>(J.pad_atoms)[sgm] = second ? __ldg(p.pad_atoms + ls) + A_r : __ldg(r.pad_atoms + ls);
  }
}

// ---- workspace layout -----------------------------------------------------------------------
struct EncBufs {
  float* inp;
  float* pre[kMaxDepth];
  float* m[kMaxDepth + 1];  // m[1..T]
  float* am;
  float* hid;
};
struct Workspace {
  PackedLayout L;
  float* packed;       // L.total floats, followed by its TF32 hi and lo images (img.tf32_hi, img.tf32_lo)
  WeightImages img;    // of packed; the bf16 images are L.total elements each
  float* dpacked;
  // The shared-weight encoder runs ONCE over the reactant and product batches together (mpn.py:61-108 is row-wise apart from the gathers,
  // and those stay inside a segment): every encoder buffer holds the reactant rows followed by the product rows.
  EncBufs enc[2];     // views: 0 = reactant rows, 1 = product rows of the joint buffers below
  EncBufs j;          // joint buffers [r rows | p rows]
  rr_graph J;         // the joint graph: index tables in joint row space (built by k_join_tables), features contiguous [r | p]
  bool copy_feats;    // r / p feature arrays are not adjacent in memory: copied into j_fa / j_fb once per forward
  float *j_fa, *j_fb;
  float *d, *inp2, *nf, *am2, *hid2, *vec, *zout;
  float* nm[kMaxDepth];
  float* m2[kMaxDepth + 1];
  float* x[RR_MAX_FFN];
  // backward scratch
  float *gB1, *gB2, *dinp, *gA1, *gA2, *gA3, *dD, *dI2, *dvec, *gN1, *gN2, *dzout;
  // deterministic mode only (last, so that every other offset is the same in both modes): the weight-gradient slabs and the padding-row
  // partials of the backward pass, one launch at a time
  float* det;
  long long det_bytes;
  size_t bytes;
};

static int carve(const rr_model_cfg_ex& cx, const rr_graph& r, const rr_graph& p, void* base, Workspace* W) {
  const rr_model_cfg& c = cx.base;
  RR_REQUIRE(c.hidden > 0 && c.hidden <= 4096, "hidden %d out of range", c.hidden);
  RR_REQUIRE(cx.diff_hidden > 0 && cx.diff_hidden <= 4096, "diff_hidden %d out of range", cx.diff_hidden);
  RR_REQUIRE(cx.ffn_hidden > 0 && cx.ffn_hidden <= 4096, "ffn_hidden %d out of range", cx.ffn_hidden);
  RR_REQUIRE(c.depth >= 1 && c.depth <= kMaxDepth && c.diff_depth >= 0 && c.diff_depth <= kMaxDepth, "depth %d / diff_depth %d out of range", c.depth, c.diff_depth);
  RR_REQUIRE(c.ffn_depth >= 1 && c.ffn_depth <= RR_MAX_FFN, "ffn_depth %d out of range", c.ffn_depth);
  RR_REQUIRE(c.task_num >= 1 && c.task_num <= RR_OUT_LD, "task_num %d out of range", c.task_num);
  RR_REQUIRE(c.add_features >= 0, "add_features < 0");
  RR_REQUIRE(c.r_atom_map != nullptr || (r.n_atoms == p.n_atoms && r.n_mols == p.n_mols),
             "reactant and product batches must have identical atom rows (p - r is atom-wise, base_model.py:168): %d vs %d", r.n_atoms, p.n_atoms);
  RR_REQUIRE(c.r_atom_map == nullptr || !(c.training && (c.dropout > 0.f || cx.diff_dropout > 0.f || cx.ffn_dropout > 0.f)),
             "r_atom_map (de-duplicated reactants) is exact only without dropout: pass NULL when training with dropout > 0");
  W->L = make_packed(cx);
  const size_t hpe = W->L.hpe, hpd = W->L.hpd, hpf = W->L.hpf, vp = W->L.vp;
  const size_t A = p.n_atoms, N = p.n_mols;
  const int T = c.depth - 1, Td = c.diff_depth - 1;
  const bool msg2 = c.diff_depth > 0;   // the diff encoder passes messages (mpn.py:199-216); at depth 0 it is W_i alone (mpn.py:220-221)
  char* cur = static_cast<char*>(base);
  size_t used = 0;
  auto take = [&](size_t floats) {
    float* ptr = base ? reinterpret_cast<float*>(cur + used) : nullptr;
    used += (floats * sizeof(float) + 255) / 256 * 256;
    return ptr;
  };
  W->packed = take(W->L.total);   // L.total is a multiple of 64 floats: the two TF32 images follow it without a gap
  W->img.base = W->packed;
  W->img.tf32_hi = take(W->L.total);
  W->img.tf32_lo = take(W->L.total);
  W->img.bf16_hi = reinterpret_cast<uint16_t*>(take((W->L.total + 1) / 2));
  W->img.bf16_lo = reinterpret_cast<uint16_t*>(take((W->L.total + 1) / 2));
  W->dpacked = take(W->L.grad_total);
  const size_t A_r = r.n_atoms, B_r = r.n_bonds, A_J = A_r + p.n_atoms, B_J = B_r + p.n_bonds;
  {
    EncBufs& e = W->j;
    e.inp = take(B_J * hpe);
    for (int t = 0; t < T; ++t) e.pre[t] = take(B_J * hpe);
    for (int t = 1; t <= T; ++t) e.m[t] = take(B_J * hpe);
    e.am = take(A_J * hpe);
    e.hid = take(A_J * hpe);
    auto part = [&](float* q, size_t rows) { return q ? q + rows * hpe : nullptr; };
    W->enc[0] = e;
    EncBufs& q = W->enc[1];
    q.inp = part(e.inp, B_r);
    for (int t = 0; t < T; ++t) q.pre[t] = part(e.pre[t], B_r);
    for (int t = 1; t <= T; ++t) q.m[t] = part(e.m[t], B_r);
    q.am = part(e.am, A_r);
    q.hid = part(e.hid, A_r);
  }
  {   // joint graph tables (int32) and, when the two batches' features are not adjacent in memory, a contiguous copy of them
    rr_graph& J = W->J;
    J = rr_graph{};
    J.n_atoms = static_cast<int>(A_J);
    J.n_bonds = static_cast<int>(B_J);
    J.n_mols = r.n_mols + p.n_mols;
    J.wmax = r.wmax > p.wmax ? r.wmax : p.wmax;
    J.n_segments = r.n_segments + p.n_segments;
    J.a_meta = reinterpret_cast<const rr_atom_meta*>(take(A_J * 4));
    J.a2b = reinterpret_cast<const int*>(take(A_J * J.wmax));
    J.a2b_rev = reinterpret_cast<const int*>(take(A_J * J.wmax));
    J.a2a = reinterpret_cast<const int*>(take(A_J * J.wmax));
    J.pad_bonds = reinterpret_cast<const int*>(take(J.n_segments));
    J.pad_atoms = reinterpret_cast<const int*>(take(J.n_segments));
    W->copy_feats = !(p.f_atoms == r.f_atoms + A_r * RR_FA_LD && p.f_bonds == r.f_bonds + B_r * RR_FB_LD);
    W->j_fa = W->copy_feats ? take(A_J * RR_FA_LD) : nullptr;
    W->j_fb = W->copy_feats ? take(B_J * RR_FB_LD) : nullptr;
    J.f_atoms = W->copy_feats ? W->j_fa : r.f_atoms;
    J.f_bonds = W->copy_feats ? W->j_fb : r.f_bonds;
  }
  W->d = take(A * hpe);
  W->inp2 = msg2 ? take(A * hpd) : nullptr;
  W->nf = msg2 ? take(A * RR_FB_LD) : nullptr;
  for (int t = 0; t < Td; ++t) W->nm[t] = take(A * hpd);
  for (int t = 1; t <= Td; ++t) W->m2[t] = take(A * hpd);
  W->am2 = msg2 ? take(A * hpd) : nullptr;
  W->hid2 = take(A * hpd);
  W->vec = take(N * vp);
  for (int l = 0; l + 1 < c.ffn_depth; ++l) W->x[l] = take(N * hpf);
  W->zout = take(N * RR_OUT_LD);
  W->gB1 = take(B_J * hpe);
  W->gB2 = take(B_J * hpe);
  W->dinp = take(B_J * hpe);
  // gA1 / gA2: encoder atom gradients over the joint rows, and before that the diff encoder's over the product rows
  const size_t gA = A_J * hpe > A * hpd ? A_J * hpe : A * hpd;
  W->gA1 = take(gA);
  W->gA2 = take(gA);
  W->gA3 = msg2 ? take(A * hpd) : nullptr;
  W->dD = take(A * hpe);
  W->dI2 = msg2 ? take(A * hpd) : nullptr;
  W->dvec = take(N * vp);
  W->gN1 = take(N * hpf);
  W->gN2 = take(N * hpf);
  W->dzout = take(N * RR_OUT_LD);
  W->det = nullptr;
  W->det_bytes = 0;
  if (deterministic()) {
    const int A_J_ = static_cast<int>(A_J), B_J_ = static_cast<int>(B_J), A_ = static_cast<int>(A), N_ = static_cast<int>(N);
    const int he = static_cast<int>(hpe), hd = static_cast<int>(hpd);
    long long need = 0;
    auto at_least = [&](long long b) { need = b > need ? b : need; };
    at_least(wgrad_det_bytes(B_J_, he, he));              // encoder W_h
    at_least(wgrad_det_bytes(B_J_, he, RR_FB_LD));        // encoder W_i
    at_least(wgrad_det_bytes(A_J_, he, he));              // encoder W_o (message part)
    at_least(wgrad_det_bytes(A_J_, he, RR_FA_LD));        // encoder W_o (atom features)
    at_least(wgrad_det_bytes(A_, hd, he));                // diff encoder W_i, W_o (d part)
    at_least(wgrad_det_bytes(A_, hd, hd));                // diff encoder W_h, W_o (message parts)
    at_least(wgrad_det_bytes(A_, hd, RR_FB_LD));          // diff encoder W_h (bond features)
    for (int l = 0; l < c.ffn_depth; ++l) at_least(wgrad_det_bytes(N_, W->L.ffn_out[l], W->L.ffn_in[l]));
    at_least(bias_grad_bytes(B_J_, he));                  // a bias that trains under a frozen weight (linear_bias_grad)
    at_least(bias_grad_bytes(A_J_, he));
    at_least(bias_grad_bytes(A_, hd));
    at_least(bias_grad_bytes(N_, static_cast<int>(hpf) > RR_OUT_LD ? static_cast<int>(hpf) : RR_OUT_LD));
    at_least(pad_parts_bytes(A_J_, r.n_segments + p.n_segments, he));   // gathers over the joint graph
    at_least(pad_parts_bytes(A_, p.n_segments, hd));                    // and over the product graph
    W->det = take(static_cast<size_t>((need + 3) / 4));
    W->det_bytes = (need + 3) / 4 * 4;
  }
  W->bytes = used;
  return RR_OK;
}

// byte offset of a named forward buffer inside the workspace (tests compare per-layer activations with the oracle)
long long model_buffer_offset(const rr_model_cfg_ex* cx, const rr_graph* r, const rr_graph* p, const char* name) {
  const rr_model_cfg* c = &cx->base;
  Workspace W;
  char* base = reinterpret_cast<char*>(static_cast<uintptr_t>(4096));
  if (carve(*cx, *r, *p, base, &W) != RR_OK) return -1;
  auto off = [&](const float* ptr) -> long long {
    if (ptr == nullptr) {
      fail(RR_ERR_INVALID, "buffer %s does not exist at diff_depth %d", name, c->diff_depth);
      return -1;
    }
    return static_cast<long long>(reinterpret_cast<const char*>(ptr) - base);
  };
  char buf[64];
  for (int k = 0; k < 2; ++k) {
    snprintf(buf, sizeof(buf), "enc%d.inp", k);
    if (!strcmp(name, buf)) return off(W.enc[k].inp);
    snprintf(buf, sizeof(buf), "enc%d.am", k);
    if (!strcmp(name, buf)) return off(W.enc[k].am);
    snprintf(buf, sizeof(buf), "enc%d.hid", k);
    if (!strcmp(name, buf)) return off(W.enc[k].hid);
    for (int t = 0; t < c->depth - 1; ++t) {
      snprintf(buf, sizeof(buf), "enc%d.pre%d", k, t);
      if (!strcmp(name, buf)) return off(W.enc[k].pre[t]);
      snprintf(buf, sizeof(buf), "enc%d.m%d", k, t + 1);
      if (!strcmp(name, buf)) return off(W.enc[k].m[t + 1]);
    }
  }
  for (int t = 0; t < c->diff_depth - 1; ++t) {
    snprintf(buf, sizeof(buf), "nm%d", t);
    if (!strcmp(name, buf)) return off(W.nm[t]);
    snprintf(buf, sizeof(buf), "m2_%d", t + 1);
    if (!strcmp(name, buf)) return off(W.m2[t + 1]);
  }
  if (!strcmp(name, "d")) return off(W.d);
  if (!strcmp(name, "inp2")) return off(W.inp2);
  if (!strcmp(name, "nf")) return off(W.nf);
  if (!strcmp(name, "am2")) return off(W.am2);
  if (!strcmp(name, "hid2")) return off(W.hid2);
  if (!strcmp(name, "vec")) return off(W.vec);
  if (!strcmp(name, "zout")) return off(W.zout);
  for (int l = 0; l + 1 < c->ffn_depth; ++l) {
    snprintf(buf, sizeof(buf), "x%d", l);
    if (!strcmp(name, buf)) return off(W.x[l]);
  }
  fail(RR_ERR_INVALID, "unknown buffer name %s", name);
  return -1;
}

long long model_workspace_bytes(const rr_model_cfg_ex* c, const rr_graph* r, const rr_graph* p) {
  Workspace W;
  if (carve(*c, *r, *p, nullptr, &W) != RR_OK) return -1;
  return static_cast<long long>(W.bytes);
}

static int check_model_args(const rr_model_cfg_ex* cx, const rr_params* w, const rr_graph* r, const rr_graph* p, void* ws, long long ws_bytes,
                            Workspace* W) {
  RR_REQUIRE(cx && w && r && p && ws, "model: NULL argument");
  const rr_model_cfg* c = &cx->base;
  RR_REQUIRE(aligned16(ws), "workspace must be 16-byte aligned");
  RR_TRY(carve(*cx, *r, *p, ws, W));
  if (static_cast<long long>(W->bytes) > ws_bytes) return fail(RR_ERR_WORKSPACE, "workspace %lld bytes < required %zu", ws_bytes, W->bytes);
  RR_REQUIRE(w->enc_Wi && w->enc_Wo && w->enc_bo && w->dif_Wi, "model: missing parameter pointer");
  RR_REQUIRE(c->depth == 1 || w->enc_Wh, "model: encoder.W_h missing for depth > 1");
  RR_REQUIRE(c->diff_depth <= 1 || w->dif_Wh, "model: diff_encoder.W_h missing for diff_depth > 1");
  RR_REQUIRE(c->diff_depth == 0 || (w->dif_Wo && w->dif_bo), "model: diff_encoder.W_o missing for diff_depth > 0");
  for (int l = 0; l < c->ffn_depth; ++l) RR_REQUIRE(w->ffn_W[l], "model: ffn weight %d missing", l);
  RR_REQUIRE(c->dropout >= 0.f && c->dropout < 1.f, "dropout must be in [0,1)");
  RR_REQUIRE(cx->diff_dropout >= 0.f && cx->diff_dropout < 1.f, "diff_dropout must be in [0,1)");
  RR_REQUIRE(cx->ffn_dropout >= 0.f && cx->ffn_dropout < 1.f, "ffn_dropout must be in [0,1)");
  RR_REQUIRE(r->f_bonds && r->f_atoms && p->f_bonds && p->f_atoms, "model: graph features missing");
  RR_REQUIRE(c->head >= RR_HEAD_RAW && c->head <= RR_HEAD_NIG, "unknown head %d", c->head);
  if (c->head == RR_HEAD_NIG) RR_REQUIRE((c->task_num & 3) == 0, "the NIG head needs task_num %% 4 == 0");
  else if (c->head != RR_HEAD_RAW && c->head != RR_HEAD_SOFTPLUS && c->head != RR_HEAD_SOFTPLUS_P1)
    RR_REQUIRE((c->task_num & 1) == 0, "two-parameter heads need an even task_num");
  return RR_OK;
}

static int pack_params(const rr_model_cfg_ex& c, const Workspace& W, const rr_params& w, cudaStream_t s) {
  RR_CUDA(cudaMemsetAsync(W.packed, 0, 3 * W.L.total * sizeof(float), s));   // the weights and their TF32 images
  RR_CUDA(cudaMemsetAsync(W.img.bf16_hi, 0, W.L.total * sizeof(uint16_t), s));
  RR_CUDA(cudaMemsetAsync(W.img.bf16_lo, 0, W.L.total * sizeof(uint16_t), s));
  PackTable T = make_table(c, W.L, w, true);
  k_pack<<<dim3(32, T.n), 256, 0, s>>>(T, W.packed, 0, W.img.tf32_hi - W.packed, W.img.tf32_lo - W.packed, W.img.bf16_hi, W.img.bf16_lo);
  RR_LAUNCH_CHECK("k_pack");
  return RR_OK;
}

// Fill the joint graph of this call's workspace: write the index tables; the features are copied only when the two batches
// do not already sit next to each other in memory (DeviceGraph.assemble_pair lays them out adjacent, so the product path copies nothing).
static int build_joint(const Workspace& W, const rr_graph& r, const rr_graph& p, cudaStream_t s) {
  ProfScope prof_scope(KC_MISC, s);
  const int n = W.J.n_atoms;
  int blocks = (n + 255) / 256;
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  if (blocks < 1) blocks = 1;
  k_join_tables<<<blocks, 256, 0, s>>>(r, p, W.J);
  RR_LAUNCH_CHECK("k_join_tables");
  if (W.copy_feats) {
    RR_CUDA(cudaMemcpyAsync(W.j_fa, r.f_atoms, static_cast<size_t>(r.n_atoms) * RR_FA_LD * 4, cudaMemcpyDeviceToDevice, s));
    RR_CUDA(cudaMemcpyAsync(W.j_fa + static_cast<size_t>(r.n_atoms) * RR_FA_LD, p.f_atoms, static_cast<size_t>(p.n_atoms) * RR_FA_LD * 4, cudaMemcpyDeviceToDevice, s));
    RR_CUDA(cudaMemcpyAsync(W.j_fb, r.f_bonds, static_cast<size_t>(r.n_bonds) * RR_FB_LD * 4, cudaMemcpyDeviceToDevice, s));
    RR_CUDA(cudaMemcpyAsync(W.j_fb + static_cast<size_t>(r.n_bonds) * RR_FB_LD, p.f_bonds, static_cast<size_t>(p.n_bonds) * RR_FB_LD * 4, cudaMemcpyDeviceToDevice, s));
  }
  return RR_OK;
}

// Dropout: each sub-module's sites use its own p (encoder: m^t, hid; diff encoder: m2^t, hid2; FFN: vec, x[l]).  Philox stream ids, which
// tests regenerate the masks from: sid starts at 1 and every lin() call takes the next one, with or without dropout, in launch order --
// encoder W_i, W_h x (depth - 1), W_o; diff encoder W_i, W_h x (diff_depth - 1), W_o; then the readout (vec); then the FFN layers.  At
// diff_depth 0 the diff encoder is W_i alone, and its id is the one that carries hid2's ReLU and dropout.
int model_forward(const rr_model_cfg_ex* cx, const rr_params* w, const rr_graph* r, const rr_graph* p, const float* addf, float* scores,
                  void* ws, long long ws_bytes, cudaStream_t s) {
  Workspace W;
  RR_TRY(check_model_args(cx, w, r, p, ws, ws_bytes, &W));
  const rr_model_cfg* c = &cx->base;
  RR_REQUIRE(scores != nullptr, "scores is NULL");
  RR_REQUIRE(c->add_features == 0 || addf != nullptr, "add_features is NULL but add_features_dim = %d", c->add_features);
  const PackedLayout& L = W.L;
  const int hpe = L.hpe, hpd = L.hpd, vp = L.vp;
  const int T = c->depth - 1, Td = c->diff_depth - 1;
  const float pe = c->training ? c->dropout : 0.f, pd = c->training ? cx->diff_dropout : 0.f, pf = c->training ? cx->ffn_dropout : 0.f;
  const int act_e = 1 | (pe > 0.f ? 2 : 0), act_d = 1 | (pd > 0.f ? 2 : 0), act_f = 1 | (pf > 0.f ? 2 : 0);
  const float* P = W.packed;
  uint64_t sid = 1;
  RR_TRY(pack_params(*cx, W, *w, s));

  // Y = act(X1 W1^T + X2 W2^T + bias + resid) with dropout p; resid has Y's row stride; pad_rows: the segment padding rows of Y (see linear_fwd)
  auto lin = [&](const int* pad_rows, int n_pad, int M, int n, const float* X1, int ldx1, size_t W1, int k1, const float* X2, int ldx2, size_t W2, int k2,
                 size_t bias, const float* resid, float* Y, int ldy, int flags, float pdrop) -> int {
    return linear_fwd(M, n, X1, ldx1, P + W1, k1, X2, ldx2, X2 ? P + W2 : nullptr, k2, P + bias, resid, ldy, Y, ldy, flags, pdrop, c->seed, sid++, s,
                      &W.img, pad_rows, n_pad);
  };
  RR_TRY(build_joint(W, *r, *p, s));
  {  // mpn.py:61-108, once over [reactant rows | product rows]: the weights are shared (base_model.py:155-156)
    const rr_graph* g = &W.J;
    EncBufs& e = W.j;
    // f_bonds[pad] = 0: the padding rows of W_i's output are the bias exactly, on any GEMM path
    RR_TRY(lin(nullptr, 0, g->n_bonds, hpe, g->f_bonds, RR_FB_LD, L.enc_Wi, RR_FB_LD, nullptr, 0, 0, 0, L.enc_bi, nullptr, e.inp, hpe, 0, pe));
    const float* src = e.inp;
    int relu_src = 1;
    for (int t = 0; t < T; ++t) {
      RR_TRY(bond_message_fwd(g, src, e.pre[t], hpe, relu_src, s));
      RR_TRY(lin(g->pad_bonds, g->n_segments, g->n_bonds, hpe, e.pre[t], hpe, L.enc_Wh, hpe, nullptr, 0, 0, 0, L.enc_bh, e.inp, e.m[t + 1], hpe, act_e, pe));
      src = e.m[t + 1];
      relu_src = 0;
    }
    RR_TRY(neighbor_sum_fwd(g, 0, src, e.am, hpe, relu_src, s));
    RR_TRY(lin(g->pad_atoms, g->n_segments, g->n_atoms, hpe, g->f_atoms, RR_FA_LD, L.enc_Wo_a, RR_FA_LD, e.am, hpe, L.enc_Wo_m, hpe, L.enc_bo, nullptr, e.hid,
               hpe, act_e, pe));
  }
  const int A = p->n_atoms;
  if (c->r_atom_map) RR_TRY(sub_gather(A, hpe, W.enc[1].hid, W.enc[0].hid, c->r_atom_map, W.d, s));
  else RR_TRY(sub(static_cast<long long>(A) * hpe, W.enc[1].hid, W.enc[0].hid, W.d, s));  // base_model.py:168

  // mpn.py:170-240 over the product graph
  if (c->diff_depth == 0) {  // mpn.py:220-221: atom_hiddens = dropout(relu(W_i(diff)))
    RR_TRY(lin(p->pad_atoms, p->n_segments, A, hpd, W.d, hpe, L.dif_Wi, hpe, nullptr, 0, 0, 0, L.dif_bi, nullptr, W.hid2, hpd, act_d, pd));
  } else {
    RR_TRY(lin(p->pad_atoms, p->n_segments, A, hpd, W.d, hpe, L.dif_Wi, hpe, nullptr, 0, 0, 0, L.dif_bi, nullptr, W.inp2, hpd, 0, pd));
    if (Td > 0) RR_TRY(neighbor_sum_fwd(p, 0, p->f_bonds, W.nf, RR_FB_LD, 0, s));
    const float* src = W.inp2;
    int relu_src = 1;
    for (int t = 0; t < Td; ++t) {
      RR_TRY(neighbor_sum_fwd(p, 1, src, W.nm[t], hpd, relu_src, s));
      RR_TRY(lin(p->pad_atoms, p->n_segments, A, hpd, W.nm[t], hpd, L.dif_Wh_m, hpd, W.nf, RR_FB_LD, L.dif_Wh_f, RR_FB_LD, L.dif_bh, W.inp2, W.m2[t + 1],
                 hpd, act_d, pd));
      src = W.m2[t + 1];
      relu_src = 0;
    }
    RR_TRY(neighbor_sum_fwd(p, 1, src, W.am2, hpd, relu_src, s));
    RR_TRY(lin(p->pad_atoms, p->n_segments, A, hpd, W.d, hpe, L.dif_Wo_d, hpe, W.am2, hpd, L.dif_Wo_m, hpd, L.dif_bo, nullptr, W.hid2, hpd, act_d, pd));
  }
  RR_TRY(readout_fwd(p, W.hid2, hpd, cx->diff_hidden, addf, c->add_features, W.vec, vp, pf, c->seed, sid++, s));

  // base_model.py:40-60
  const int N = p->n_mols;
  const float* x = W.vec;
  int ldx = vp;
  for (int l = 0; l < c->ffn_depth; ++l) {
    const bool last = (l == c->ffn_depth - 1);
    float* y = last ? W.zout : W.x[l];
    RR_TRY(lin(nullptr, 0, N, L.ffn_out[l], x, ldx, L.ffn_W[l], L.ffn_in[l], nullptr, 0, 0, 0, L.ffn_b[l], nullptr, y, L.ffn_out[l], last ? 0 : act_f, pf));
    x = y;
    ldx = L.ffn_out[l];
  }
  {
    const int n = N * c->task_num;
    k_head_fwd<<<(n + 255) / 256, 256, 0, s>>>(N, c->task_num, c->head, W.zout, scores);
    RR_LAUNCH_CHECK("k_head_fwd");
  }
  return RR_OK;
}

// Only the gradients the caller asks for are computed: a NULL pointer in `grads` means that tensor is neither computed nor written
// (frozen).  Layers in graph order from the input up: encoder W_i < W_h < W_o < diff encoder W_i < W_h < W_o < FFN 0 .. F-1.  A layer's
// weight gradient runs when its weight is requested (its bias fused in), its bias gradient alone (linear_bias_grad) when only the bias
// is; the dgrad chain runs through a layer only while some layer below it trains.  With every pointer set this is the full backward,
// launch for launch.
int model_backward(const rr_model_cfg_ex* cx, const rr_params* w, const rr_graph* r, const rr_graph* p, const float* dscores, rr_params* grads,
                   void* ws, long long ws_bytes, cudaStream_t s) {
  Workspace W;
  RR_TRY(check_model_args(cx, w, r, p, ws, ws_bytes, &W));
  const rr_model_cfg* c = &cx->base;
  RR_REQUIRE(dscores && grads, "backward: NULL argument");
  enum { E_I, E_H, E_O, D_I, D_H, D_O, F0 };
  const rr_params& gp = *grads;
  const int nlev = F0 + c->ffn_depth;
  bool wreq[F0 + RR_MAX_FFN] = {gp.enc_Wi != nullptr, gp.enc_Wh != nullptr, gp.enc_Wo != nullptr, gp.dif_Wi != nullptr, gp.dif_Wh != nullptr,
                                gp.dif_Wo != nullptr};
  bool breq[F0 + RR_MAX_FFN] = {gp.enc_bi != nullptr, gp.enc_bh != nullptr, gp.enc_bo != nullptr, gp.dif_bi != nullptr, gp.dif_bh != nullptr,
                                gp.dif_bo != nullptr};
  for (int l = 0; l < c->ffn_depth; ++l) {
    wreq[F0 + l] = gp.ffn_W[l] != nullptr;
    breq[F0 + l] = gp.ffn_b[l] != nullptr;
  }
  bool below[F0 + RR_MAX_FFN + 1];   // below[lv]: some layer under lv trains
  below[0] = false;
  for (int lv = 0; lv < nlev; ++lv) below[lv + 1] = below[lv] || wreq[lv] || breq[lv];
  if (!below[nlev]) return RR_OK;
  if (deterministic() && c->r_atom_map && below[D_I])
    return fail(RR_ERR_UNSUPPORTED, "deterministic mode: the backward pass of de-duplicated reactants (r_atom_map) sums rows with atomics");
  const PackedLayout& L = W.L;
  const int hpe = L.hpe, hpd = L.hpd, hpf = L.hpf, vp = L.vp;
  const int T = c->depth - 1, Td = c->diff_depth - 1;
  const float pe = c->training ? c->dropout : 0.f, pd = c->training ? cx->diff_dropout : 0.f, pf = c->training ? cx->ffn_dropout : 0.f;
  const float keep_e = pe > 0.f ? 1.f / (1.f - pe) : 1.f, keep_d = pd > 0.f ? 1.f / (1.f - pd) : 1.f, keep_f = pf > 0.f ? 1.f / (1.f - pf) : 1.f;
  const float* P = W.packed;  // still holds this step's packed weights
  float* G = W.dpacked;
  RR_CUDA(cudaMemsetAsync(G, 0, L.grad_total * sizeof(float), s));
  const int N = p->n_mols, A = p->n_atoms;
  // the bias gradient of layer lv when its weight is frozen (otherwise the weight gradient computes it, or it is not wanted)
  auto bias_only = [&](int lv, int M, int n, const float* dZ, int lddz, size_t db) -> int {
    return (!wreq[lv] && breq[lv]) ? linear_bias_grad(M, n, dZ, lddz, G + db, s, W.det, W.det_bytes) : RR_OK;
  };

  auto chain = [&]() -> int {
    {
      const int n = N * RR_OUT_LD;
      k_head_bwd<<<(n + 255) / 256, 256, 0, s>>>(N, c->task_num, c->head, W.zout, dscores, W.dzout);
      RR_LAUNCH_CHECK("k_head_bwd");
    }
    // FFN
    {
      const float* g = W.dzout;
      int ldg = RR_OUT_LD;
      float* scratch[2] = {W.gN1, W.gN2};
      for (int l = c->ffn_depth - 1; l >= 0; --l) {
        const float* x = (l == 0) ? W.vec : W.x[l - 1];
        if (wreq[F0 + l])
          RR_TRY(linear_wgrad(N, L.ffn_out[l], L.ffn_in[l], g, ldg, x, L.ffn_in[l], G + L.ffn_W[l], L.ffn_in[l], G + L.ffn_b[l], s, W.det, W.det_bytes));
        RR_TRY(bias_only(F0 + l, N, L.ffn_out[l], g, ldg, L.ffn_b[l]));
        if (!below[F0 + l]) return RR_OK;
        if (l > 0) {
          float* dx = scratch[l & 1];
          RR_TRY(linear_dgrad(N, L.ffn_out[l], L.ffn_in[l], g, ldg, P + L.ffn_W[l], L.ffn_in[l], P + L.ffn_W_T[l], L.ffn_out[l], dx, hpf, 0, W.img, s));
          RR_TRY(relu_bwd(N, hpf, dx, W.x[l - 1], keep_f, 0, dx, nullptr, 0, s));
          g = dx;
          ldg = hpf;
        } else {
          RR_TRY(linear_dgrad(N, L.ffn_out[l], L.ffn_in[l], g, ldg, P + L.ffn_W[l], L.ffn_in[l], P + L.ffn_W_T[l], L.ffn_out[l], W.dvec, vp, 0, W.img, s));
        }
      }
    }
    // readout: the gradient of the diff encoder's last layer (W_o, or W_i at diff_depth 0) through hid2's ReLU / dropout mask
    RR_TRY(readout_bwd(p, W.dvec, vp, W.vec, W.hid2, W.gA1, hpd, pf, pd, s));
    const float* dWi = W.gA1;   // gradient of W_i's output
    if (c->diff_depth > 0) {
      if (wreq[D_O]) {
        RR_TRY(linear_wgrad(A, hpd, hpe, W.gA1, hpd, W.d, hpe, G + L.dif_Wo_d, hpe, G + L.dif_bo, s, W.det, W.det_bytes));
        RR_TRY(linear_wgrad(A, hpd, hpd, W.gA1, hpd, W.am2, hpd, G + L.dif_Wo_m, hpd, nullptr, s, W.det, W.det_bytes));
      }
      RR_TRY(bias_only(D_O, A, hpd, W.gA1, hpd, L.dif_bo));
      if (!below[D_O]) return RR_OK;
      if (below[D_I]) RR_TRY(linear_dgrad(A, hpd, hpe, W.gA1, hpd, P + L.dif_Wo_d, hpe, P + L.dif_Wo_d_T, hpd, W.dD, hpe, 0, W.img, s));  // only the encoder reads dD
      RR_TRY(linear_dgrad(A, hpd, hpd, W.gA1, hpd, P + L.dif_Wo_m, hpd, P + L.dif_Wo_m_T, hpd, W.gA2, hpd, 0, W.img, s));
      // Every gather backward is followed by exactly one ReLU (+ dropout) backward: the mask of the message it produced the gradient of.
      // Both run as one kernel (rr_mp_pipe.cu): t_next >= 1 -> mask of m2^{t_next}, result kept (gA1) and summed into dI2;
      // t_next == 0 -> mask [inp2 > 0] of m2^0 = relu(inp2), only the sum into dI2 is wanted.
      auto diff_nbr_bwd = [&](int t_next) {
        if (t_next >= 1)
          return neighbor_sum_bwd_act(p, 1, W.gA2, W.gA1, hpd, W.m2[t_next], keep_d, 0, W.dI2, t_next == Td ? 1 : 2, 0, s, W.det, W.det_bytes);
        return neighbor_sum_bwd_act(p, 1, W.gA2, W.gA3, hpd, W.inp2, 1.f, 1, W.dI2, Td == 0 ? 1 : 2, 1, s, W.det, W.det_bytes);
      };
      RR_TRY(diff_nbr_bwd(Td));
      for (int t = Td; t >= 1; --t) {
        if (wreq[D_H]) {
          RR_TRY(linear_wgrad(A, hpd, hpd, W.gA1, hpd, W.nm[t - 1], hpd, G + L.dif_Wh_m, hpd, G + L.dif_bh, s, W.det, W.det_bytes));
          RR_TRY(linear_wgrad(A, hpd, RR_FB_LD, W.gA1, hpd, W.nf, RR_FB_LD, G + L.dif_Wh_f, RR_FB_LD, nullptr, s, W.det, W.det_bytes));
        }
        RR_TRY(bias_only(D_H, A, hpd, W.gA1, hpd, L.dif_bh));
        if (t == 1 && !below[D_H]) return RR_OK;   // what follows feeds W_i and the encoder only
        RR_TRY(linear_dgrad(A, hpd, hpd, W.gA1, hpd, P + L.dif_Wh_m, hpd, P + L.dif_Wh_m_T, hpd, W.gA2, hpd, 0, W.img, s));
        RR_TRY(diff_nbr_bwd(t - 1));
      }
      dWi = W.dI2;
    }
    if (wreq[D_I]) RR_TRY(linear_wgrad(A, hpd, hpe, dWi, hpd, W.d, hpe, G + L.dif_Wi, hpe, G + L.dif_bi, s, W.det, W.det_bytes));
    RR_TRY(bias_only(D_I, A, hpd, dWi, hpd, L.dif_bi));
    if (!below[D_I]) return RR_OK;
    // accumulates onto W_o's share of dD; at diff_depth 0 it is the only share
    RR_TRY(linear_dgrad(A, hpd, hpe, dWi, hpd, P + L.dif_Wi, hpe, P + L.dif_Wi_T, hpd, W.dD, hpe, c->diff_depth > 0 ? 1 : 0, W.img, s));

    // shared encoder, once over [reactant rows | product rows]: d(hid_p) = +dD, d(hid_r) = -dD (base_model.py:168), each through the
    // ReLU / dropout mask of its own rows; the weight gradients of both halves come out of one launch per layer (base_model.py:155-156)
    // (the joint graph's tables, and its feature copy if one was needed, are in the workspace since the forward)
    const rr_graph* g = &W.J;
    EncBufs& e = W.j;
    const int A_r = r->n_atoms, A_J = g->n_atoms, B_J = g->n_bonds;
    float* gA1_p = W.gA1 + static_cast<size_t>(A_r) * hpe;
    RR_TRY(relu_bwd(A, hpe, W.dD, W.enc[1].hid, keep_e, 0, gA1_p, nullptr, 0, s));
    if (c->r_atom_map) {   // shared reactant rows: sum the gradient over the copies first (gA2 is free until the dgrad below)
      RR_CUDA(cudaMemsetAsync(W.gA2, 0, static_cast<size_t>(A_r) * hpe * sizeof(float), s));
      RR_TRY(scatter_add_rows(A, hpe, W.dD, c->r_atom_map, W.gA2, s));
      RR_TRY(relu_bwd(A_r, hpe, W.gA2, W.enc[0].hid, -keep_e, 0, W.gA1, nullptr, 0, s));
    } else {
      RR_TRY(relu_bwd(A_r, hpe, W.dD, W.enc[0].hid, -keep_e, 0, W.gA1, nullptr, 0, s));
    }
    if (wreq[E_O]) {
      RR_TRY(linear_wgrad(A_J, hpe, RR_FA_LD, W.gA1, hpe, g->f_atoms, RR_FA_LD, G + L.enc_Wo_a, RR_FA_LD, G + L.enc_bo, s, W.det, W.det_bytes));
      RR_TRY(linear_wgrad(A_J, hpe, hpe, W.gA1, hpe, e.am, hpe, G + L.enc_Wo_m, hpe, nullptr, s, W.det, W.det_bytes));
    }
    RR_TRY(bias_only(E_O, A_J, hpe, W.gA1, hpe, L.enc_bo));
    if (!below[E_O]) return RR_OK;
    RR_TRY(linear_dgrad(A_J, hpe, hpe, W.gA1, hpe, P + L.enc_Wo_m, hpe, P + L.enc_Wo_m_T, hpe, W.gA2, hpe, 0, W.img, s));
    if (T >= 1) RR_TRY(neighbor_sum_bwd_act(g, 0, W.gA2, W.gB1, hpe, e.m[T], keep_e, 0, W.dinp, 1, 0, s, W.det, W.det_bytes));
    else RR_TRY(neighbor_sum_bwd_act(g, 0, W.gA2, W.gB1, hpe, e.inp, 1.f, 1, W.dinp, 1, 1, s, W.det, W.det_bytes));
    for (int t = T; t >= 1; --t) {
      if (wreq[E_H]) RR_TRY(linear_wgrad(B_J, hpe, hpe, W.gB1, hpe, e.pre[t - 1], hpe, G + L.enc_Wh, hpe, G + L.enc_bh, s, W.det, W.det_bytes));
      RR_TRY(bias_only(E_H, B_J, hpe, W.gB1, hpe, L.enc_bh));
      if (t == 1 && !below[E_H]) return RR_OK;   // what follows feeds W_i only
      RR_TRY(linear_dgrad(B_J, hpe, hpe, W.gB1, hpe, P + L.enc_Wh, hpe, P + L.enc_Wh_T, hpe, W.gB2, hpe, 0, W.img, s));
      if (t - 1 >= 1) RR_TRY(bond_message_bwd_act(g, W.gB2, W.gB1, hpe, e.m[t - 1], keep_e, 0, W.dinp, 2, 0, s, W.det, W.det_bytes));
      else RR_TRY(bond_message_bwd_act(g, W.gB2, W.gB1, hpe, e.inp, 1.f, 1, W.dinp, 2, 1, s, W.det, W.det_bytes));
    }
    if (wreq[E_I]) RR_TRY(linear_wgrad(B_J, hpe, RR_FB_LD, W.dinp, hpe, g->f_bonds, RR_FB_LD, G + L.enc_Wi, RR_FB_LD, G + L.enc_bi, s, W.det, W.det_bytes));
    return bias_only(E_I, B_J, hpe, W.dinp, hpe, L.enc_bi);
  };
  RR_TRY(chain());

  PackTable Tb = make_table(*cx, L, *grads, false);
  k_pack<<<dim3(32, Tb.n), 256, 0, s>>>(Tb, G, 1, 0, 0, nullptr, nullptr);
  RR_LAUNCH_CHECK("k_pack(grads)");
  return RR_OK;
}

}  // namespace rr
