// Message-passing gather-sum kernels (models/mpn.py of the reference), HBM-bound.
//
// Work decomposition: one thread per (atom, 16-byte column chunk).  A block holds
// `apb` atoms x `cpr` chunks (cpr = ld/4), so every lane does useful work even when the
// row width (e.g. 304 floats = 76 chunks) is not a multiple of the warp size, and a
// thread's chunk index stays fixed across its grid-stride iterations -- which lets the
// padding-row gradient be accumulated in registers and flushed with a few atomics.
//
// Every real bond row is read once and written once per pass (the algorithmic minimum,
// SURVEY.md §8d): for atom a with incoming bonds b_k, the outgoing bonds are exactly
// rev(b_k), so   pre[rev(b_k)] = (sum_j m[b_j] + pad_count*m[pad]) - m[b_k]
// is produced from registers without materialising a_message or the [A, W, h] gather
// (mpn.py:89-92).  The padding row is gathered with its multiplicity instead of once per
// padded slot (featurization.py:281-286).
#include <stdlib.h>

#include "rr_common.cuh"

namespace rr {

constexpr int kFast = 4;  // neighbours kept in registers; larger in-degrees take the reload path

// One atom's gather task.  Everything in it is loaded WITHOUT waiting for the in-degree (the index rows are read
// unconditionally up to kFast), and the task of the thread's NEXT atom is prefetched while the current rows are in
// flight: the dependent chain meta -> indices -> rows collapses to one DRAM round trip per atom in steady state.
struct Task {
  int deg, pad_count, pad_bond, pad_atom;
  bool is_pad;
  int idx[kFast];
  int rev[kFast];
};

template <bool WITH_REV>
__device__ __forceinline__ void load_task(Task& t, const rr_graph& g, const int* __restrict__ table, int a) {
  const int4 m = __ldg(reinterpret_cast<const int4*>(g.a_meta) + a);
  const int* ib = table + static_cast<size_t>(a) * g.wmax;
  const int* rb = g.a2b_rev + static_cast<size_t>(a) * g.wmax;
  if (g.wmax == 4) {
    const int4 i4 = __ldg(reinterpret_cast<const int4*>(ib));
    t.idx[0] = i4.x; t.idx[1] = i4.y; t.idx[2] = i4.z; t.idx[3] = i4.w;
    if (WITH_REV) {
      const int4 r4 = __ldg(reinterpret_cast<const int4*>(rb));
      t.rev[0] = r4.x; t.rev[1] = r4.y; t.rev[2] = r4.z; t.rev[3] = r4.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < kFast; ++k) {
      t.idx[k] = (k < g.wmax) ? __ldg(ib + k) : 0;
      if (WITH_REV) t.rev[k] = (k < g.wmax) ? __ldg(rb + k) : 0;
    }
  }
  t.deg = m.x & 0xff;
  t.is_pad = (m.x >> 8) & 1;
  t.pad_count = m.y;
  t.pad_bond = m.z;
  t.pad_atom = m.w;
}

__device__ __forceinline__ float4 ld_row(const float* base, int row, int ld, int c4, bool relu) {
  float4 v = ld_f4(base + static_cast<size_t>(row) * ld + c4);
  return relu ? f4_relu(v) : v;
}

// block = apb atoms x cpr chunks; grid-stride over atoms with a one-task prefetch
#define RR_ATOM_SETUP()                                                            \
  const int cpr = ld >> 2;                                                         \
  const int slot = threadIdx.x / cpr;                                              \
  const int c4 = (threadIdx.x - slot * cpr) << 2;                                  \
  const int apb = blockDim.x / cpr;                                                \
  if (slot >= apb) return;                                                         \
  const int stride = gridDim.x * apb;                                              \
  int a = blockIdx.x * apb + slot;                                                 \
  if (a >= g.n_atoms) return

// ---------------------------------------------------------------------------------------
// forward: pre = bond_message(m)                                         mpn.py:89-92
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512, 2) k_bond_fwd(rr_graph g, const float* __restrict__ m, float* __restrict__ pre, int ld, int relu) {
  RR_ATOM_SETUP();
  Task nx;
  load_task<true>(nx, g, g.a2b, a);
  for (; a < g.n_atoms; a += stride) {
    const Task t = nx;
    if (a + stride < g.n_atoms) load_task<true>(nx, g, g.a2b, a + stride);
    float4 acc = f4_zero();
    if (t.pad_count > 0) acc = f4_scale(static_cast<float>(t.pad_count), ld_row(m, t.pad_bond, ld, c4, relu));
    float4 v[kFast];
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) v[k] = ld_row(m, t.idx[k], ld, c4, relu);
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) acc = f4_add(acc, v[k]);
    const int* ib = g.a2b + static_cast<size_t>(a) * g.wmax;
    const int* rb = g.a2b_rev + static_cast<size_t>(a) * g.wmax;
    for (int k = kFast; k < t.deg; ++k) acc = f4_add(acc, ld_row(m, __ldg(ib + k), ld, c4, relu));
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) st_f4(pre + static_cast<size_t>(t.rev[k]) * ld + c4, f4_sub(acc, v[k]));
    for (int k = kFast; k < t.deg; ++k)
      st_f4(pre + static_cast<size_t>(__ldg(rb + k)) * ld + c4, f4_sub(acc, ld_row(m, __ldg(ib + k), ld, c4, relu)));
    if (t.is_pad)  // the padding bond: b2a = pad atom, b2revb = itself (featurization.py:262-264)
      st_f4(pre + static_cast<size_t>(t.pad_bond) * ld + c4, f4_sub(acc, ld_row(m, t.pad_bond, ld, c4, relu)));
  }
}

// ---------------------------------------------------------------------------------------
// backward: dm from dpre.  dm[b_k] = S_a - dpre[rev(b_k)],  S_a = sum_k dpre[rev(b_k)]
// padding row: dm[pad] += sum_a pad_count_a * S_a - dpre[pad]   (row pre-zeroed by k_zero_rows)
// DET = true (deterministic mode): the padding-row partials go to pp, and pad_rows_sum() adds them (rr_common.cuh: PadParts)
// ---------------------------------------------------------------------------------------
template <bool DET>
__global__ void __launch_bounds__(512, 2) k_bond_bwd(rr_graph g, const float* __restrict__ dpre, float* __restrict__ dm, int ld, PadParts pp) {
  RR_ATOM_SETUP();
  float4 pad_acc = f4_zero();
  int pad_row = -1;
  int pad_j = 0;
  const long long unit = static_cast<long long>(blockIdx.x) * apb + slot;
  Task nx;
  load_task<true>(nx, g, g.a2b, a);
  for (; a < g.n_atoms; a += stride) {
    const Task t = nx;
    if (a + stride < g.n_atoms) load_task<true>(nx, g, g.a2b, a + stride);
    if (t.pad_bond != pad_row) {
      if constexpr (DET) {
        if (pad_row >= 0) pad_part_store(pp, unit, pad_j, pad_row, ld, c4, pad_acc);
      } else {
        if (pad_row >= 0) red_add_f4(dm + static_cast<size_t>(pad_row) * ld + c4, pad_acc);
      }
      pad_acc = f4_zero();
      pad_row = t.pad_bond;
    }
    float4 S = f4_zero();
    float4 self = f4_zero();
    if (t.is_pad) {
      self = ld_row(dpre, t.pad_bond, ld, c4, false);
      S = self;
    }
    float4 v[kFast];
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) v[k] = ld_row(dpre, t.rev[k], ld, c4, false);
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) S = f4_add(S, v[k]);
    const int* ib = g.a2b + static_cast<size_t>(a) * g.wmax;
    const int* rb = g.a2b_rev + static_cast<size_t>(a) * g.wmax;
    for (int k = kFast; k < t.deg; ++k) S = f4_add(S, ld_row(dpre, __ldg(rb + k), ld, c4, false));
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) st_f4(dm + static_cast<size_t>(t.idx[k]) * ld + c4, f4_sub(S, v[k]));
    for (int k = kFast; k < t.deg; ++k)
      st_f4(dm + static_cast<size_t>(__ldg(ib + k)) * ld + c4, f4_sub(S, ld_row(dpre, __ldg(rb + k), ld, c4, false)));
    pad_acc = f4_fma(static_cast<float>(t.pad_count), S, pad_acc);
    pad_acc = f4_sub(pad_acc, self);
  }
  if constexpr (DET) {
    if (pad_row >= 0) pad_part_store(pp, unit, pad_j, pad_row, ld, c4, pad_acc);
  } else {
    if (pad_row >= 0) red_add_f4(dm + static_cast<size_t>(pad_row) * ld + c4, pad_acc);
  }
}

// ---------------------------------------------------------------------------------------
// neighbour sum: out[a] = pad_count*src[pad] + sum_k src[idx[a,k]]       mpn.py:100-102,201-206,215
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512, 2) k_nbr_sum_fwd(rr_graph g, int which, const float* __restrict__ src, float* __restrict__ out, int ld, int relu) {
  const int* table = which ? g.a2a : g.a2b;
  RR_ATOM_SETUP();
  Task nx;
  load_task<false>(nx, g, table, a);
  for (; a < g.n_atoms; a += stride) {
    const Task t = nx;
    if (a + stride < g.n_atoms) load_task<false>(nx, g, table, a + stride);
    float4 acc = f4_zero();
    if (t.pad_count > 0) acc = f4_scale(static_cast<float>(t.pad_count), ld_row(src, which ? t.pad_atom : t.pad_bond, ld, c4, relu));
    float4 v[kFast];
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) v[k] = ld_row(src, t.idx[k], ld, c4, relu);
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) acc = f4_add(acc, v[k]);
    const int* ib = table + static_cast<size_t>(a) * g.wmax;
    for (int k = kFast; k < t.deg; ++k) acc = f4_add(acc, ld_row(src, __ldg(ib + k), ld, c4, relu));
    st_f4(out + static_cast<size_t>(a) * ld + c4, acc);
  }
}

// backward over bond rows (which = 0): dsrc[b_k] = dout[a]; dsrc[pad] += pad_count * dout[a]
template <bool DET>
__global__ void __launch_bounds__(512, 2) k_nbr_sum_bwd_bond(rr_graph g, const float* __restrict__ dout, float* __restrict__ dsrc, int ld, PadParts pp) {
  RR_ATOM_SETUP();
  float4 pad_acc = f4_zero();
  int pad_row = -1;
  int pad_j = 0;
  const long long unit = static_cast<long long>(blockIdx.x) * apb + slot;
  Task nx;
  load_task<false>(nx, g, g.a2b, a);
  float4 vn = ld_row(dout, a, ld, c4, false);
  for (; a < g.n_atoms; a += stride) {
    const Task t = nx;
    const float4 v = vn;
    if (a + stride < g.n_atoms) {
      load_task<false>(nx, g, g.a2b, a + stride);
      vn = ld_row(dout, a + stride, ld, c4, false);
    }
    if (t.pad_bond != pad_row) {
      if constexpr (DET) {
        if (pad_row >= 0) pad_part_store(pp, unit, pad_j, pad_row, ld, c4, pad_acc);
      } else {
        if (pad_row >= 0) red_add_f4(dsrc + static_cast<size_t>(pad_row) * ld + c4, pad_acc);
      }
      pad_acc = f4_zero();
      pad_row = t.pad_bond;
    }
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) st_f4(dsrc + static_cast<size_t>(t.idx[k]) * ld + c4, v);
    const int* ib = g.a2b + static_cast<size_t>(a) * g.wmax;
    for (int k = kFast; k < t.deg; ++k) st_f4(dsrc + static_cast<size_t>(__ldg(ib + k)) * ld + c4, v);
    pad_acc = f4_fma(static_cast<float>(t.pad_count), v, pad_acc);
  }
  if constexpr (DET) {
    if (pad_row >= 0) pad_part_store(pp, unit, pad_j, pad_row, ld, c4, pad_acc);
  } else {
    if (pad_row >= 0) red_add_f4(dsrc + static_cast<size_t>(pad_row) * ld + c4, pad_acc);
  }
}

// backward over atom rows (which = 1): the neighbour relation is symmetric, so
// dsrc[a] = sum_k dout[a2a[a,k]] (real neighbours only); dsrc[pad_atom] += pad_count_a * dout[a]
template <bool DET>
__global__ void __launch_bounds__(512, 2) k_nbr_sum_bwd_atom(rr_graph g, const float* __restrict__ dout, float* __restrict__ dsrc, int ld, PadParts pp) {
  RR_ATOM_SETUP();
  float4 pad_acc = f4_zero();
  int pad_row = -1;
  int pad_j = 0;
  const long long unit = static_cast<long long>(blockIdx.x) * apb + slot;
  Task nx;
  load_task<false>(nx, g, g.a2a, a);
  for (; a < g.n_atoms; a += stride) {
    const Task t = nx;
    if (a + stride < g.n_atoms) load_task<false>(nx, g, g.a2a, a + stride);
    if (t.pad_atom != pad_row) {
      if constexpr (DET) {
        if (pad_row >= 0) pad_part_store(pp, unit, pad_j, pad_row, ld, c4, pad_acc);
      } else {
        if (pad_row >= 0) red_add_f4(dsrc + static_cast<size_t>(pad_row) * ld + c4, pad_acc);
      }
      pad_acc = f4_zero();
      pad_row = t.pad_atom;
    }
    float4 self = f4_zero();
    if (t.pad_count > 0) self = ld_row(dout, a, ld, c4, false);
    float4 v[kFast];
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) v[k] = ld_row(dout, t.idx[k], ld, c4, false);
    float4 acc = f4_zero();
#pragma unroll
    for (int k = 0; k < kFast; ++k)
      if (k < t.deg) acc = f4_add(acc, v[k]);
    const int* ib = g.a2a + static_cast<size_t>(a) * g.wmax;
    for (int k = kFast; k < t.deg; ++k) acc = f4_add(acc, ld_row(dout, __ldg(ib + k), ld, c4, false));
    if (!t.is_pad) st_f4(dsrc + static_cast<size_t>(a) * ld + c4, acc);
    pad_acc = f4_fma(static_cast<float>(t.pad_count), self, pad_acc);
  }
  if constexpr (DET) {
    if (pad_row >= 0) pad_part_store(pp, unit, pad_j, pad_row, ld, c4, pad_acc);
  } else {
    if (pad_row >= 0) red_add_f4(dsrc + static_cast<size_t>(pad_row) * ld + c4, pad_acc);
  }
}

__global__ void k_zero_rows(float* __restrict__ base, const int* __restrict__ rows, int n_rows, int ld) {
  const int r = blockIdx.x;
  if (r >= n_rows) return;
  float* p = base + static_cast<size_t>(__ldg(rows + r)) * ld;
  for (int c = threadIdx.x * 4; c < ld; c += blockDim.x * 4) st_f4(p + c, f4_zero());
}

// ---------------------------------------------------------------------------------------
// readout                                                                mpn.py:224-238
// ---------------------------------------------------------------------------------------
__global__ void k_readout_fwd(rr_graph g, const float* __restrict__ hid, int hp, int hidden, const float* __restrict__ addf, int n_add,
                              float* __restrict__ vec, int vp, float p, uint64_t seed, uint64_t stream_id) {
  const int cpr = vp >> 2;
  const long long total = static_cast<long long>(g.n_mols) * cpr;
  const float inv_keep = p > 0.f ? 1.f / (1.f - p) : 1.f;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(t / cpr);
    const int c4 = static_cast<int>(t - static_cast<long long>(i) * cpr) << 2;
    const int start = __ldg(g.mol_start + i), size = __ldg(g.mol_size + i);
    float4 acc = f4_zero();
    if (c4 < hp)
      for (int a = start; a < start + size; ++a) acc = f4_add(acc, ld_f4(hid + static_cast<size_t>(a) * hp + c4));
    if (size > 0) acc = f4_scale(1.f / static_cast<float>(size), acc);  // size == 0 -> cached_zero_vector (mpn.py:225-226)
    float e[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = c4 + j;
      if (col >= hidden) e[j] = (col < hidden + n_add) ? __ldg(addf + static_cast<size_t>(i) * n_add + (col - hidden)) : 0.f;
    }
    float4 o = make_float4(e[0], e[1], e[2], e[3]);
    if (p > 0.f) o = dropout4(o, p, inv_keep, seed, stream_id, static_cast<uint64_t>(t));
    st_f4(vec + static_cast<size_t>(i) * vp + c4, o);
  }
}

// dz[a] = dvec[mol]/size * [vec != 0]*keep_vec * [hid[a] != 0]*keep_hid  (relu + both dropouts: the FFN's on vec, the diff encoder's on hid)
__global__ void k_readout_bwd(rr_graph g, const float* __restrict__ dvec, int vp, const float* __restrict__ vec, const float* __restrict__ hid,
                              float* __restrict__ dz, int hp, float keep_vec, float keep_hid) {
  const int cpr = hp >> 2;
  const long long total = static_cast<long long>(g.n_mols) * cpr;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(t / cpr);
    const int c4 = static_cast<int>(t - static_cast<long long>(i) * cpr) << 2;
    const int start = __ldg(g.mol_start + i), size = __ldg(g.mol_size + i);
    if (size <= 0) continue;
    float4 d = f4_zero();
    if (c4 < vp) {
      d = ld_f4(dvec + static_cast<size_t>(i) * vp + c4);
      if (keep_vec != 1.f) {  // the FFN's first dropout acted on vec
        const float4 y = ld_f4(vec + static_cast<size_t>(i) * vp + c4);
        d.x = y.x != 0.f ? d.x * keep_vec : 0.f;
        d.y = y.y != 0.f ? d.y * keep_vec : 0.f;
        d.z = y.z != 0.f ? d.z * keep_vec : 0.f;
        d.w = y.w != 0.f ? d.w * keep_vec : 0.f;
      }
    }
    const float s = keep_hid / static_cast<float>(size);
    d = f4_scale(s, d);
    for (int a = start; a < start + size; ++a) {
      const float4 h = ld_f4(hid + static_cast<size_t>(a) * hp + c4);
      float4 o;
      o.x = h.x != 0.f ? d.x : 0.f;
      o.y = h.y != 0.f ? d.y : 0.f;
      o.z = h.z != 0.f ? d.z : 0.f;
      o.w = h.w != 0.f ? d.w : 0.f;
      st_f4(dz + static_cast<size_t>(a) * hp + c4, o);
    }
  }
}

// ---------------------------------------------------------------------------------------
// elementwise
// ---------------------------------------------------------------------------------------
__global__ void k_relu_bwd(long long n4, const float* __restrict__ dy, const float* __restrict__ y, float scale, int preact,
                           float* __restrict__ dz, float* __restrict__ acc, int acc_mode) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 g = ld_f4_stream(dy + i * 4);
    const float4 v = ld_f4_stream(y + i * 4);
    float4 o;
    if (preact) {
      o.x = v.x > 0.f ? g.x * scale : 0.f;
      o.y = v.y > 0.f ? g.y * scale : 0.f;
      o.z = v.z > 0.f ? g.z * scale : 0.f;
      o.w = v.w > 0.f ? g.w * scale : 0.f;
    } else {
      o.x = v.x != 0.f ? g.x * scale : 0.f;
      o.y = v.y != 0.f ? g.y * scale : 0.f;
      o.z = v.z != 0.f ? g.z * scale : 0.f;
      o.w = v.w != 0.f ? g.w * scale : 0.f;
    }
    if (dz) st_f4(dz + i * 4, o);
    if (acc_mode == 1) st_f4(acc + i * 4, o);
    else if (acc_mode == 2) st_f4(acc + i * 4, f4_add(ld_f4_stream(acc + i * 4), o));
  }
}

__global__ void k_sub(long long n4, const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * blockDim.x)
    st_f4(out + i * 4, f4_sub(ld_f4_stream(a + i * 4), ld_f4_stream(b + i * 4)));
}

// d[a] = hid_p[a] - hid_r[map[a]]: base_model.py:168 with de-duplicated reactants (rr_model_cfg.r_atom_map)
__global__ void k_sub_gather(long long rows, int cpr, const float* __restrict__ a, const float* __restrict__ b, const int* __restrict__ map,
                             float* __restrict__ out) {
  const long long n4 = rows * cpr;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cpr;
    const int c = static_cast<int>(i - r * cpr);
    const long long rb = __ldg(map + r);
    st_f4(out + i * 4, f4_sub(ld_f4_stream(a + i * 4), ld_f4(b + (rb * cpr + c) * 4)));
  }
}
// dst[map[a]] += src[a]: the gradient of a shared reactant row is the sum over its copies (dst zeroed by the caller)
__global__ void k_scatter_add_rows(long long rows, int cpr, const float* __restrict__ src, const int* __restrict__ map, float* __restrict__ dst) {
  const long long n4 = rows * cpr;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cpr;
    const int c = static_cast<int>(i - r * cpr);
    const float4 v = ld_f4_stream(src + i * 4);
    float* d = dst + (static_cast<long long>(__ldg(map + r)) * cpr + c) * 4;
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(d), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
  }
}

// ---------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------
static int check_graph(const rr_graph* g, int ld) {
  RR_REQUIRE(g != nullptr, "graph is NULL");
  RR_REQUIRE(g->n_atoms > 0 && g->n_bonds > 0 && g->wmax > 0, "graph sizes must be positive (atoms %d bonds %d wmax %d)", g->n_atoms, g->n_bonds, g->wmax);
  RR_REQUIRE(ld > 0 && (ld & 3) == 0 && ld <= 2048, "row stride %d must be a multiple of 4 and <= 2048", ld);
  RR_REQUIRE(g->a_meta && g->a2b && g->a2b_rev && g->a2a, "graph index arrays are NULL");
  RR_REQUIRE(aligned16(g->a_meta), "a_meta must be 16-byte aligned");
  return RR_OK;
}

static void atom_launch_dims(int n_atoms, int ld, dim3* grid, dim3* block) {
  const int cpr = ld >> 2;
  int apb = 256 / cpr;
  if (apb < 1) apb = 1;
  int threads = apb * cpr;
  const int blocks_needed = (n_atoms + apb - 1) / apb;
  int per_sm = 2048 / ((threads + 31) / 32 * 32);
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;   // ~64 registers per thread: 4 resident blocks of ~256 threads, each thread walks several atoms
  int g = num_sms() * per_sm;
  if (g > blocks_needed) g = blocks_needed;
  if (g < 1) g = 1;
  *grid = dim3(g);
  *block = dim3(threads);
}

// second-generation kernels (rr_mp_pipe.cu); RR_MP_V1=1 selects the first generation, which the tests use as the pipeline's reference
enum { PIPE_BOND_FWD = 0, PIPE_BOND_BWD = 1, PIPE_NBR_FWD = 2, PIPE_NBR_BWD_BOND = 3, PIPE_NBR_BWD_ATOM = 4 };
static bool use_pipe() { return switches().mp_v1 != 1; }

int bond_message_fwd(const rr_graph* g, const float* m, float* pre, int hp, int relu_src, cudaStream_t s) {
  ProfScope prof_scope(KC_BOND_FWD, s);
  RR_TRY(check_graph(g, hp));
  RR_REQUIRE(m && pre && aligned16(m) && aligned16(pre), "m/pre must be non-NULL and 16-byte aligned");
  if (use_pipe()) {
    const int st = rowpipe_launch(PIPE_BOND_FWD, g, 0, m, pre, hp, relu_src, nullptr, 1.f, 0, nullptr, 0, 0, s);
    if (st != RR_ERR_UNSUPPORTED) return st;
  }
  dim3 grid, block;
  atom_launch_dims(g->n_atoms, hp, &grid, &block);
  k_bond_fwd<<<grid, block, 0, s>>>(*g, m, pre, hp, relu_src);
  RR_LAUNCH_CHECK("k_bond_fwd");
  return RR_OK;
}

static int zero_rows(float* base, const int* rows, int n, int ld, cudaStream_t s) {
  if (n <= 0) return RR_OK;
  k_zero_rows<<<n, 128, 0, s>>>(base, rows, n, ld);
  RR_LAUNCH_CHECK("k_zero_rows");
  return RR_OK;
}

static int check_act(const float* y, float* acc, int acc_mode, int skip_out) {
  RR_REQUIRE(y != nullptr && aligned16(y), "fused relu backward: y must be non-NULL and 16-byte aligned");
  RR_REQUIRE(acc_mode >= 0 && acc_mode <= 2 && (acc_mode == 0 || (acc && aligned16(acc))), "fused relu backward: acc_mode %d needs an aligned acc", acc_mode);
  RR_REQUIRE(!skip_out || acc_mode != 0, "fused relu backward: skip_out without acc discards the result");
  return RR_OK;
}

// dm = bond_message_bwd(dpre), then (y != NULL) the ReLU / dropout backward that follows it in the model:
// dz = dm * mask(y) * scale written to dm (unless skip_out) and stored / added into acc
// Deterministic mode: scratch for the padding-row partials (the caller's `det` when given, else transient)
static int det_pad_scratch(DetScratch* ds, const rr_graph* g, int ld, void* det, long long det_bytes, long long* bytes, cudaStream_t s) {
  const long long need = pad_parts_bytes(g->n_atoms, g->n_segments, ld);
  RR_TRY(det_scratch(ds, det, det_bytes, need, s));
  *bytes = det ? det_bytes : need;
  return RR_OK;
}
// first generation, deterministic: the partials of the launch's units (blocks x atoms per block, see atom_launch_dims)
static int v1_pad_parts(const DetScratch& ds, long long bytes, const rr_graph* g, int ld, dim3 grid, PadParts* pp, cudaStream_t s) {
  const int apb = 256 / (ld >> 2) > 0 ? 256 / (ld >> 2) : 1;
  const long long units = static_cast<long long>(grid.x) * apb;
  return pad_parts_setup(ds.p, bytes, units, (g->n_atoms + units - 1) / units, g->n_segments, ld, pp, s);
}

int bond_message_bwd_act(const rr_graph* g, const float* dpre, float* dm, int hp, const float* y, float scale, int preact, float* acc, int acc_mode,
                         int skip_out, cudaStream_t s, void* det, long long det_bytes) {
  RR_TRY(check_graph(g, hp));
  RR_REQUIRE(dpre && dm && aligned16(dpre) && aligned16(dm), "dpre/dm must be non-NULL and 16-byte aligned");
  RR_REQUIRE(g->pad_bonds && g->n_segments > 0, "graph needs pad_bonds/n_segments");
  if (y) RR_TRY(check_act(y, acc, acc_mode, skip_out));
  {
    ProfScope prof_scope(KC_BOND_BWD, s);
    DetScratch ds;
    long long ds_bytes = 0;
    PadParts pp{};
    const bool in_det = deterministic();
    if (in_det) RR_TRY(det_pad_scratch(&ds, g, hp, det, det_bytes, &ds_bytes, s));
    RR_TRY(zero_rows(dm, g->pad_bonds, g->n_segments, hp, s));
    int st = RR_ERR_UNSUPPORTED;
    if (use_pipe()) st = rowpipe_launch(PIPE_BOND_BWD, g, 0, dpre, dm, hp, 0, y, scale, preact, acc, acc_mode, skip_out, s, ds.p, ds_bytes, &pp);
    if (st == RR_OK) {
      if (in_det) RR_TRY(pad_rows_sum(dm, g->pad_bonds, g->n_segments, hp, pp, s));
      return y ? pad_rows_act(dm, g->pad_bonds, g->n_segments, hp, y, scale, preact, acc, acc_mode, skip_out, s) : RR_OK;
    }
    if (st != RR_ERR_UNSUPPORTED) return st;
    dim3 grid, block;
    atom_launch_dims(g->n_atoms, hp, &grid, &block);
    if (in_det) {
      RR_TRY(v1_pad_parts(ds, ds_bytes, g, hp, grid, &pp, s));
      k_bond_bwd<true><<<grid, block, 0, s>>>(*g, dpre, dm, hp, pp);
      RR_LAUNCH_CHECK("k_bond_bwd");
      RR_TRY(pad_rows_sum(dm, g->pad_bonds, g->n_segments, hp, pp, s));
    } else {
      k_bond_bwd<false><<<grid, block, 0, s>>>(*g, dpre, dm, hp, pp);
      RR_LAUNCH_CHECK("k_bond_bwd");
    }
  }
  return y ? relu_bwd(g->n_bonds, hp, dm, y, scale, preact, skip_out ? nullptr : dm, acc, acc_mode, s) : RR_OK;
}

int bond_message_bwd(const rr_graph* g, const float* dpre, float* dm, int hp, cudaStream_t s) {
  return bond_message_bwd_act(g, dpre, dm, hp, nullptr, 1.f, 0, nullptr, 0, 0, s);
}

int neighbor_sum_fwd(const rr_graph* g, int which, const float* src, float* out, int ld, int relu_src, cudaStream_t s) {
  ProfScope prof_scope(KC_NBR_FWD, s);
  RR_TRY(check_graph(g, ld));
  RR_REQUIRE(src && out && aligned16(src) && aligned16(out), "src/out must be non-NULL and 16-byte aligned");
  if (use_pipe()) {
    const int st = rowpipe_launch(PIPE_NBR_FWD, g, which, src, out, ld, relu_src, nullptr, 1.f, 0, nullptr, 0, 0, s);
    if (st != RR_ERR_UNSUPPORTED) return st;
  }
  dim3 grid, block;
  atom_launch_dims(g->n_atoms, ld, &grid, &block);
  k_nbr_sum_fwd<<<grid, block, 0, s>>>(*g, which, src, out, ld, relu_src);
  RR_LAUNCH_CHECK("k_nbr_sum_fwd");
  return RR_OK;
}

int neighbor_sum_bwd_act(const rr_graph* g, int which, const float* dout, float* dsrc, int ld, const float* y, float scale, int preact, float* acc,
                         int acc_mode, int skip_out, cudaStream_t s, void* det, long long det_bytes) {
  RR_TRY(check_graph(g, ld));
  RR_REQUIRE(dout && dsrc && aligned16(dout) && aligned16(dsrc), "dout/dsrc must be non-NULL and 16-byte aligned");
  RR_REQUIRE(g->pad_bonds && g->pad_atoms && g->n_segments > 0, "graph needs pad rows/n_segments");
  if (y) RR_TRY(check_act(y, acc, acc_mode, skip_out));
  const int* pads = which == 0 ? g->pad_bonds : g->pad_atoms;
  {
    ProfScope prof_scope(KC_NBR_BWD, s);
    DetScratch ds;
    long long ds_bytes = 0;
    PadParts pp{};
    const bool in_det = deterministic();
    if (in_det) RR_TRY(det_pad_scratch(&ds, g, ld, det, det_bytes, &ds_bytes, s));
    RR_TRY(zero_rows(dsrc, pads, g->n_segments, ld, s));
    int st = RR_ERR_UNSUPPORTED;
    if (use_pipe())
      st = rowpipe_launch(which == 0 ? PIPE_NBR_BWD_BOND : PIPE_NBR_BWD_ATOM, g, which, dout, dsrc, ld, 0, y, scale, preact, acc, acc_mode, skip_out, s, ds.p,
                          ds_bytes, &pp);
    if (st == RR_OK) {
      if (in_det) RR_TRY(pad_rows_sum(dsrc, pads, g->n_segments, ld, pp, s));
      return y ? pad_rows_act(dsrc, pads, g->n_segments, ld, y, scale, preact, acc, acc_mode, skip_out, s) : RR_OK;
    }
    if (st != RR_ERR_UNSUPPORTED) return st;
    dim3 grid, block;
    atom_launch_dims(g->n_atoms, ld, &grid, &block);
    if (in_det) RR_TRY(v1_pad_parts(ds, ds_bytes, g, ld, grid, &pp, s));
    if (which == 0) {
      if (in_det) k_nbr_sum_bwd_bond<true><<<grid, block, 0, s>>>(*g, dout, dsrc, ld, pp);
      else k_nbr_sum_bwd_bond<false><<<grid, block, 0, s>>>(*g, dout, dsrc, ld, pp);
      RR_LAUNCH_CHECK("k_nbr_sum_bwd_bond");
    } else {
      if (in_det) k_nbr_sum_bwd_atom<true><<<grid, block, 0, s>>>(*g, dout, dsrc, ld, pp);
      else k_nbr_sum_bwd_atom<false><<<grid, block, 0, s>>>(*g, dout, dsrc, ld, pp);
      RR_LAUNCH_CHECK("k_nbr_sum_bwd_atom");
    }
    if (in_det) RR_TRY(pad_rows_sum(dsrc, pads, g->n_segments, ld, pp, s));
  }
  return y ? relu_bwd(which == 0 ? g->n_bonds : g->n_atoms, ld, dsrc, y, scale, preact, skip_out ? nullptr : dsrc, acc, acc_mode, s) : RR_OK;
}

int neighbor_sum_bwd(const rr_graph* g, int which, const float* dout, float* dsrc, int ld, cudaStream_t s) {
  return neighbor_sum_bwd_act(g, which, dout, dsrc, ld, nullptr, 1.f, 0, nullptr, 0, 0, s);
}

int readout_fwd(const rr_graph* g, const float* hid, int hp, int hidden, const float* addf, int n_add, float* vec, int vp, float p,
                uint64_t seed, uint64_t stream_id, cudaStream_t s) {
  ProfScope prof_scope(KC_READOUT, s);
  RR_REQUIRE(g && g->n_mols > 0 && g->mol_start && g->mol_size, "graph has no molecule scope");
  RR_REQUIRE((hp & 3) == 0 && (vp & 3) == 0 && vp >= hidden + n_add && hidden <= hp, "readout widths hp %d vp %d hidden %d n_add %d", hp, vp, hidden, n_add);
  RR_REQUIRE(n_add == 0 || addf != nullptr, "add_features is NULL");
  RR_REQUIRE(p >= 0.f && p < 1.f, "dropout p must be in [0,1)");
  const long long total = static_cast<long long>(g->n_mols) * (vp >> 2);
  int blocks = static_cast<int>((total + 255) / 256);
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  k_readout_fwd<<<blocks, 256, 0, s>>>(*g, hid, hp, hidden, addf, n_add, vec, vp, p, seed, stream_id);
  RR_LAUNCH_CHECK("k_readout_fwd");
  return RR_OK;
}

int readout_bwd(const rr_graph* g, const float* dvec, int vp, const float* vec, const float* hid, float* dz, int hp, float p_vec, float p_hid,
                cudaStream_t s) {
  ProfScope prof_scope(KC_READOUT, s);
  RR_REQUIRE(g && g->n_mols > 0 && g->mol_start && g->mol_size && g->pad_atoms, "graph has no molecule scope");
  RR_REQUIRE((hp & 3) == 0 && (vp & 3) == 0 && vp >= hp, "readout_bwd needs vp >= hp (vp %d hp %d)", vp, hp);
  RR_TRY(zero_rows(dz, g->pad_atoms, g->n_segments, hp, s));
  const long long total = static_cast<long long>(g->n_mols) * (hp >> 2);
  int blocks = static_cast<int>((total + 255) / 256);
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  k_readout_bwd<<<blocks, 256, 0, s>>>(*g, dvec, vp, vec, hid, dz, hp, p_vec > 0.f ? 1.f / (1.f - p_vec) : 1.f,
                                       p_hid > 0.f ? 1.f / (1.f - p_hid) : 1.f);
  RR_LAUNCH_CHECK("k_readout_bwd");
  return RR_OK;
}

int relu_bwd(long long rows, int ld, const float* dy, const float* y, float scale, int preact, float* dz, float* acc, int acc_mode, cudaStream_t s) {
  ProfScope prof_scope(KC_ELEMENTWISE, s);
  RR_REQUIRE((ld & 3) == 0 && rows >= 0, "relu_bwd: ld %d must be a multiple of 4", ld);
  RR_REQUIRE(dy && y && (dz || acc_mode), "relu_bwd: NULL argument");
  RR_REQUIRE(acc_mode == 0 || acc != nullptr, "relu_bwd: acc is NULL");
  const long long n4 = rows * ld / 4;
  if (n4 == 0) return RR_OK;
  long long blocks = (n4 + 255) / 256;
  if (blocks > num_sms() * 16) blocks = num_sms() * 16;
  k_relu_bwd<<<static_cast<int>(blocks), 256, 0, s>>>(n4, dy, y, scale, preact, dz, acc, acc_mode);
  RR_LAUNCH_CHECK("k_relu_bwd");
  return RR_OK;
}

int sub_gather(long long rows, int ld, const float* a, const float* b, const int* map, float* out, cudaStream_t s) {
  ProfScope prof_scope(KC_ELEMENTWISE, s);
  RR_REQUIRE((ld & 3) == 0 && a && b && map && out && rows >= 0, "sub_gather: bad argument (ld %d)", ld);
  const long long n4 = rows * (ld >> 2);
  if (n4 == 0) return RR_OK;
  long long blocks = (n4 + 255) / 256;
  if (blocks > num_sms() * 16) blocks = num_sms() * 16;
  k_sub_gather<<<static_cast<int>(blocks), 256, 0, s>>>(rows, ld >> 2, a, b, map, out);
  RR_LAUNCH_CHECK("k_sub_gather");
  return RR_OK;
}

int scatter_add_rows(long long rows, int ld, const float* src, const int* map, float* dst, cudaStream_t s) {
  ProfScope prof_scope(KC_ELEMENTWISE, s);
  RR_REQUIRE((ld & 3) == 0 && src && map && dst && rows >= 0, "scatter_add_rows: bad argument (ld %d)", ld);
  const long long n4 = rows * (ld >> 2);
  if (n4 == 0) return RR_OK;
  long long blocks = (n4 + 255) / 256;
  if (blocks > num_sms() * 16) blocks = num_sms() * 16;
  k_scatter_add_rows<<<static_cast<int>(blocks), 256, 0, s>>>(rows, ld >> 2, src, map, dst);
  RR_LAUNCH_CHECK("k_scatter_add_rows");
  return RR_OK;
}

int sub(long long n, const float* a, const float* b, float* out, cudaStream_t s) {
  ProfScope prof_scope(KC_ELEMENTWISE, s);
  RR_REQUIRE((n & 3) == 0 && a && b && out, "sub: n %lld must be a multiple of 4", n);
  const long long n4 = n / 4;
  if (n4 == 0) return RR_OK;
  long long blocks = (n4 + 255) / 256;
  if (blocks > num_sms() * 16) blocks = num_sms() * 16;
  k_sub<<<static_cast<int>(blocks), 256, 0, s>>>(n4, a, b, out);
  RR_LAUNCH_CHECK("k_sub");
  return RR_OK;
}

}  // namespace rr
