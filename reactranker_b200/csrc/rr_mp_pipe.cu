// Message-passing gather kernels, second generation: rows travel global -> shared memory as 1-D TMA bulk copies
// (cp.async.bulk + mbarrier complete_tx) issued by a producer warp that runs several stages ahead of the consumer
// warps, so the bytes in flight are bounded by shared memory (~190 KB per SM) instead of by the registers of the threads
// that will eventually consume them.  The first-generation kernels (rr_mp.cu: one thread per (atom, 16-byte chunk), rows
// loaded into registers) kept ~30 KB in flight per SM and stopped at 2.3-3.3 TB/s.
//
// One stage = `apb` consecutive atoms (as many as 256 consumer threads cover at ld/4 chunks per row).  For every atom
// the producer lane that owns it reads the atom's record (rr_atom_meta) and index rows, stores them as the stage's task
// list, and issues one bulk copy per needed row:
//   neighbour sources (up to 3): src_j[table_j[a, k]], k < min(deg, 4)          (rows of m / dpre / y / acc ...)
//   own-row sources   (up to 3): src_j[a]                                       (one copy for the stage's contiguous atoms)
// Consumers wait on the stage's "full" barrier, combine the rows out of shared memory and write their results straight to
// global memory (coalesced 16 bytes per lane), then release the stage.  The ops:
//   BOND_FWD      pre[rev(b_k)] = (sum_j m[b_j] + pad_count m[pad]) - m[b_k]                   mpn.py:89-92
//   BOND_BWD      dm[b_k] = S_a - dpre[rev(b_k)],  S_a = sum_k dpre[rev(b_k)]                   (autograd of the above)
//   NBR_FWD       out[a] = pad_count src[pad] + sum_k src[idx[a,k]]                            mpn.py:100-102, 201-206, 215
//   NBR_BWD_BOND  dsrc[b_k] = dout[a]                                                          (a2b table)
//   NBR_BWD_ATOM  dsrc[a] = sum_k dout[a2a[a,k]]                                               (symmetric relation)
// The backward ops optionally carry the ReLU / inverted-dropout backward that always follows them in the model
// (rr_relu_bwd: dz = d * [y != 0] * scale, acc (+)= dz) so that the raw gradient never makes a round trip through HBM;
// the segment padding rows, which are reduced with atomics, get that epilogue from a tiny follow-up kernel.  In deterministic mode the
// backward ops store the padding-row partials instead (k_rowpipe<.., DET = true>) and k_pad_rows_sum adds them in a fixed order first.
#include <stdlib.h>

#include "rr_common.cuh"

namespace rr {
namespace pipe {

constexpr int kFast = 4;          // neighbours staged per atom; larger in-degrees read the rest straight from global memory (fewer
                                  // staged rows and a deeper ring measured slower: profiles/r02_mp_kstage.md)
constexpr int MAX_CONSUMERS = 512; // consumer threads: 16 warps when at least four such stages fit, else 8
constexpr int PRODUCERS = 4;      // producer warps: one warp issuing every stage was the bottleneck (a single warp retires ~1 instruction per 4-5
                                  // cycles and a stage costs it several hundred); the warps take the rounds in turn

constexpr int MAX_STAGES = 16;
constexpr int SMEM_BUDGET = 200 * 1024;

enum Op { BOND_FWD = 0, BOND_BWD = 1, NBR_FWD = 2, NBR_BWD_BOND = 3, NBR_BWD_ATOM = 4 };

// A stage's task list: 48 bytes per atom in shared memory, three 16-byte words
//   q0 = { deg | is_pad << 8 | valid << 9, pad_count, pad_row, atom }   q1 = idx[0..3]   q2 = rev[0..3]
// pad_row is the segment's padding row in the row space the op reduces into.
struct Task {
  int deg, flags, pad_count, pad_row;
  int idx[kFast];
  int rev[kFast];
  int atom, valid;
};
constexpr int TASK_BYTES = 48;

struct Args {
  rr_graph g;
  int op, ld, relu_src, which;
  const float* src;
  float* out;
  // fused ReLU-backward epilogue (y == NULL: none)
  const float* y;
  float scale;
  int preact;
  float* acc;
  int acc_mode;     // 0 none, 1 acc = dz, 2 acc += dz
  int skip_out;     // do not write dz for ordinary rows (only acc is wanted)
  int acc_red;      // acc += dz as a fire-and-forget vector reduction (red.global.add.v4.f32) instead of staging the accumulator rows:
                    // a third fewer bytes per stage, so twice the atoms (and 16 consumer warps) fit the ring
  int apb, stages, n_stage_total;
  int kstage;       // neighbour rows staged per atom (<= kFast); neighbours beyond it are read straight from global memory by the consumer
  int producers, round_stages, consumer_warps;   // active producer warps, stages per producer round
  int n_nbr, n_own; // row sources per neighbour / per atom
  int stage_bytes, row_bytes;
  PadParts pp;      // DET kernels: padding-row partials, unit = blockIdx.x * apb + slot
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "PIPE_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra PIPE_DONE;\n\t"
      "bra PIPE_WAIT;\n\t"
      "PIPE_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
               "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ float4 lds4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float4 mask_scale(float4 d, float4 y, float scale, int preact) {
  float4 o;
  if (preact) {
    o.x = y.x > 0.f ? d.x * scale : 0.f;
    o.y = y.y > 0.f ? d.y * scale : 0.f;
    o.z = y.z > 0.f ? d.z * scale : 0.f;
    o.w = y.w > 0.f ? d.w * scale : 0.f;
  } else {
    o.x = y.x != 0.f ? d.x * scale : 0.f;
    o.y = y.y != 0.f ? d.y * scale : 0.f;
    o.z = y.z != 0.f ? d.z * scale : 0.f;
    o.w = y.w != 0.f ? d.w * scale : 0.f;
  }
  return o;
}

template <int OP>
__device__ __forceinline__ const float* nbr_source(const Args& a, int j) {
  switch (OP) {
    case BOND_BWD: return j == 0 ? a.src : (j == 1 ? a.y : a.acc);
    case NBR_BWD_BOND: return j == 0 ? a.y : a.acc;
    default: return a.src;
  }
}
template <int OP>
__device__ __forceinline__ const float* own_source(const Args& a, int j) {
  if (OP == NBR_BWD_BOND) return a.src;
  return j == 0 ? a.src : (j == 1 ? a.y : a.acc);             // NBR_BWD_ATOM: dout[a], y[a], acc[a]
}

// DET = true (deterministic mode, backward ops): a padding-row partial is stored to A.pp instead of added into the row with atomics.
template <int OP, bool FUSED, bool DET>
__global__ void __launch_bounds__(MAX_CONSUMERS + 32 * PRODUCERS, 1) k_rowpipe(const __grid_constant__ Args A) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~static_cast<uintptr_t>(127));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + MAX_STAGES;
  uint8_t* stage0 = smem + 256;
  const rr_graph& g = A.g;
  const int S = A.stages, apb = A.apb, ld = A.ld;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Every CTA takes ONE contiguous run of stages (not a round-robin): with many segments in a launch (RankNet windows, evaluation
  // batches) a CTA then meets one or two segments, and the atomics into a segment's padding row come from a handful of CTAs instead of all.
  const int per = A.n_stage_total / gridDim.x, rem = A.n_stage_total - per * gridDim.x;
  const int first_stage = blockIdx.x * per + min(static_cast<int>(blockIdx.x), rem);
  const int my_stages = per + (static_cast<int>(blockIdx.x) < rem ? 1 : 0);
  const int nbr_rows_per_atom = A.kstage * A.n_nbr;
  // stage layout: tasks [apb] | neighbour rows [apb][kFast][n_nbr] | own rows [n_own][apb]
  const int task_bytes = apb * TASK_BYTES;
  const int own_off = task_bytes + apb * nbr_rows_per_atom * A.row_bytes;

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, A.consumer_warps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_launch_dependents();
  pdl_wait();               // see rr_common.cuh: nothing above reads or writes global memory

  if (warp >= A.consumer_warps) {
    // ------------------------------------------------ producer ------------------------------------------------
    // The producer works in ROUNDS of R = 32 / apb stages: lane l owns atom (l % apb) of the round's stage (l / apb), so one round of index
    // loads (issued a whole round ahead) feeds R stages and their latency is paid once per R stages, hidden behind the previous round.
    const int R = A.round_stages, NP = A.producers;    // NP * R <= S: no producer ever starts a stage two laps of the ring ahead
    const int my_r = lane / apb, my_slot = lane - my_r * apb;
    const bool atom_tab = (OP == NBR_BWD_ATOM) || (OP == NBR_FWD && A.which);
    constexpr bool need_rev = (OP == BOND_FWD || OP == BOND_BWD);
    auto load = [&](int it_base, Task& t) {
      const int my_it = it_base + my_r;
      const long long sidx = first_stage + my_it;
      const long long a = sidx * apb + my_slot;
      t.valid = (my_r < R && my_it < my_stages && a < g.n_atoms) ? 1 : 0;
      t.atom = static_cast<int>(a);
      t.deg = 0;
      if (!t.valid) return;
      const int4 m = __ldg(reinterpret_cast<const int4*>(g.a_meta) + a);
      t.deg = m.x & 0xff;
      t.flags = (m.x >> 8) & 1;
      t.pad_count = m.y;
      t.pad_row = atom_tab ? m.w : m.z;
      const int* tb = (atom_tab ? g.a2a : g.a2b) + static_cast<size_t>(a) * g.wmax;
      const int* rb = g.a2b_rev + static_cast<size_t>(a) * g.wmax;
      if (g.wmax == 4) {
        const int4 i4 = __ldg(reinterpret_cast<const int4*>(tb));
        t.idx[0] = i4.x; t.idx[1] = i4.y; t.idx[2] = i4.z; t.idx[3] = i4.w;
        if (need_rev) {
          const int4 r4 = __ldg(reinterpret_cast<const int4*>(rb));
          t.rev[0] = r4.x; t.rev[1] = r4.y; t.rev[2] = r4.z; t.rev[3] = r4.w;
        }
      } else {
#pragma unroll
        for (int k = 0; k < kFast; ++k) {
          t.idx[k] = (k < g.wmax) ? __ldg(tb + k) : 0;
          t.rev[k] = (k < g.wmax && need_rev) ? __ldg(rb + k) : 0;
        }
      }
    };
    const int pw = warp - A.consumer_warps;          // this producer warp takes rounds pw, pw + NP, ...
    if (pw >= NP) return;
    Task nx;
    load(pw * R, nx);
    for (int it_base = pw * R; it_base < my_stages; it_base += NP * R) {
      const Task t = nx;
      load(it_base + NP * R, nx);
      const int nfetch = t.valid ? min(t.deg, A.kstage) : 0;
      for (int rr = 0; rr < R; ++rr) {
        const int it = it_base + rr;
        if (it >= my_stages) break;
        const int sidx = first_stage + it;
        const int st = it % S;
        const uint32_t ph = (it / S) & 1;
        if (lane == 0) mbar_wait(empty + st, ph ^ 1);
        __syncwarp();
        uint8_t* base = stage0 + static_cast<size_t>(st) * A.stage_bytes;
        const bool mine = (my_r == rr);
        if (mine) {
          const uint32_t tp = smem_u32(base) + my_slot * TASK_BYTES;
          const int w0 = t.valid ? (t.deg | (t.flags << 8) | (1 << 9)) : 0;
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(tp), "r"(w0), "r"(t.pad_count), "r"(t.pad_row), "r"(t.atom) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(tp + 16), "r"(t.idx[0]), "r"(t.idx[1]), "r"(t.idx[2]), "r"(t.idx[3]) : "memory");
          if (need_rev)
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(tp + 32), "r"(t.rev[0]), "r"(t.rev[1]), "r"(t.rev[2]), "r"(t.rev[3]) : "memory");
        }
        const int first_atom = static_cast<int>(sidx) * apb;
        const int n_valid = min(apb, g.n_atoms - first_atom);
        uint32_t bytes = mine ? static_cast<uint32_t>(nfetch * A.n_nbr) * A.row_bytes : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) bytes += __shfl_xor_sync(0xffffffffu, bytes, o);
        bytes += static_cast<uint32_t>(A.n_own * n_valid) * A.row_bytes;
        if (lane == 0) mbar_expect_tx(full + st, bytes);
        __syncwarp();
        if (mine && t.valid) {
          const uint32_t rows = smem_u32(base + task_bytes) + static_cast<uint32_t>(my_slot * nbr_rows_per_atom) * A.row_bytes;
          for (int j = 0; j < A.n_nbr; ++j) {
            const float* sp = nbr_source<OP>(A, j);
            const bool use_rev = (OP == BOND_BWD && j == 0);
            for (int k = 0; k < nfetch; ++k) {
              const int row = use_rev ? t.rev[k] : t.idx[k];
              bulk_g2s(rows + static_cast<uint32_t>(k * A.n_nbr + j) * A.row_bytes, sp + static_cast<size_t>(row) * ld, A.row_bytes, full + st);
            }
          }
        }
        if (lane < A.n_own)
          bulk_g2s(smem_u32(base + own_off) + static_cast<uint32_t>(lane * apb) * A.row_bytes, own_source<OP>(A, lane) + static_cast<size_t>(first_atom) * ld,
                   static_cast<uint32_t>(n_valid) * A.row_bytes, full + st);
      }
    }
  } else {
    // ------------------------------------------------ consumers -----------------------------------------------
    // The per-stage instruction count of these 8 warps is what bounds the kernel once the rows arrive in time, so everything that does not
    // depend on the stage is hoisted and the op is a template parameter.
    const int cpr = ld >> 2;
    const int slot = threadIdx.x / cpr;
    const int c4 = (threadIdx.x - slot * cpr) << 2;
    const bool active = slot < apb;
    constexpr bool REDUCES = (OP == BOND_BWD || OP == NBR_BWD_BOND || OP == NBR_BWD_ATOM);
    float4 pad_acc = f4_zero();
    int pad_row = -1;
    int pad_j = 0;                    // DET: padding rows this unit has met
    const long long unit = static_cast<long long>(blockIdx.x) * apb + slot;
    float4 padv_c = f4_zero();        // this thread's chunk of the segment's padding row of src: constant while the segment lasts
    int padv_row = -1;
    const float* src_c = A.src + c4;
    float* out_c = A.out + c4;
    const float* y_c = A.y + c4;
    float* acc_c = A.acc + c4;
    const uint32_t nbr_stride = static_cast<uint32_t>(A.n_nbr) * A.row_bytes;           // between neighbours k of one source
    const uint32_t task_off = slot * TASK_BYTES;
    const uint32_t rows_off = task_bytes + static_cast<uint32_t>(slot * nbr_rows_per_atom) * A.row_bytes + c4 * 4;
    const uint32_t own_off_t = own_off + static_cast<uint32_t>(slot) * A.row_bytes + c4 * 4;
    const uint32_t own_stride = static_cast<uint32_t>(apb) * A.row_bytes;
    const uint32_t stage0_u = smem_u32(stage0);
    auto pad_value = [&](int row) {
      if (row != padv_row) {
        padv_c = ld_f4(src_c + static_cast<size_t>(row) * ld);
        if (A.relu_src) padv_c = f4_relu(padv_c);
        padv_row = row;
      }
      return padv_c;
    };
    auto epilogue = [&](float4 d, float4 yv, float4 av, size_t off) {     // fused rr_relu_bwd on one 16-byte chunk
      const float4 o = mask_scale(d, yv, A.scale, A.preact);
      if (!A.skip_out) st_f4(out_c + off, o);
      if (A.acc_mode == 1) st_f4(acc_c + off, o);
      else if (A.acc_mode == 2) {
        if (A.acc_red) asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(acc_c + off), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w) : "memory");
        else st_f4(acc_c + off, f4_add(av, o));
      }
    };
    int st = 0;
    uint32_t ph = 0;
    for (int it = 0; it < my_stages; ++it) {
      mbar_wait(full + st, ph);
      const uint32_t base = stage0_u + static_cast<uint32_t>(st) * A.stage_bytes;
      int4 q0 = make_int4(0, 0, 0, 0);
      if (active) asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(q0.x), "=r"(q0.y), "=r"(q0.z), "=r"(q0.w) : "r"(base + task_off));
      if (q0.x & (1 << 9)) {
        const int deg = q0.x & 0xff, is_pad = (q0.x >> 8) & 1, pad_count = q0.y, prow = q0.z, a = q0.w;
        const int nf = min(deg, A.kstage);
        const uint32_t rows = base + rows_off;
        auto nbr = [&](int k, int j) { return lds4(rows + k * nbr_stride + j * A.row_bytes); };
        int4 q1 = make_int4(0, 0, 0, 0);     // rows this op writes: rev (BOND_FWD) or idx (BOND_BWD, NBR_BWD_BOND)
        if (OP == BOND_FWD) asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(q1.x), "=r"(q1.y), "=r"(q1.z), "=r"(q1.w) : "r"(base + task_off + 32));
        if (OP == BOND_BWD || OP == NBR_BWD_BOND)
          asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(q1.x), "=r"(q1.y), "=r"(q1.z), "=r"(q1.w) : "r"(base + task_off + 16));
        const int wrow[kFast] = {q1.x, q1.y, q1.z, q1.w};
        if (REDUCES && prow != pad_row) {
          if constexpr (DET) {
            if (pad_row >= 0) pad_part_store(A.pp, unit, pad_j, pad_row, ld, c4, pad_acc);
          } else {
            if (pad_row >= 0) red_add_f4(out_c + static_cast<size_t>(pad_row) * ld, pad_acc);
          }
          pad_acc = f4_zero();
          pad_row = prow;
        }
        if (OP == BOND_FWD) {
          float4 acc = f4_zero(), padv = f4_zero();
          if (pad_count > 0 || is_pad) {
            padv = pad_value(prow);
            acc = f4_scale(static_cast<float>(pad_count), padv);
          }
          float4 v[kFast];
#pragma unroll
          for (int k = 0; k < kFast; ++k)
            if (k < nf) {
              v[k] = nbr(k, 0);
              if (A.relu_src) v[k] = f4_relu(v[k]);
              acc = f4_add(acc, v[k]);
            }
          if (deg > A.kstage) {
            const int* ib = g.a2b + static_cast<size_t>(a) * g.wmax;
            for (int k = A.kstage; k < deg; ++k) {
              const float4 x = ld_f4(src_c + static_cast<size_t>(__ldg(ib + k)) * ld);
              acc = f4_add(acc, A.relu_src ? f4_relu(x) : x);
            }
          }
#pragma unroll
          for (int k = 0; k < kFast; ++k)
            if (k < nf) st_f4(out_c + static_cast<size_t>(wrow[k]) * ld, f4_sub(acc, v[k]));
          if (deg > A.kstage) {
            const int* ib = g.a2b + static_cast<size_t>(a) * g.wmax;
            const int* rb = g.a2b_rev + static_cast<size_t>(a) * g.wmax;
            for (int k = A.kstage; k < deg; ++k) {
              const float4 x = ld_f4(src_c + static_cast<size_t>(__ldg(ib + k)) * ld);
              st_f4(out_c + static_cast<size_t>(__ldg(rb + k)) * ld, f4_sub(acc, A.relu_src ? f4_relu(x) : x));
            }
          }
          if (is_pad) st_f4(out_c + static_cast<size_t>(prow) * ld, f4_sub(acc, padv));   // the padding bond: b2revb = itself
        } else if (OP == BOND_BWD) {
          float4 S4 = f4_zero(), self = f4_zero();
          if (is_pad) {
            self = ld_f4(src_c + static_cast<size_t>(prow) * ld);
            S4 = self;
          }
          float4 v[kFast];
#pragma unroll
          for (int k = 0; k < kFast; ++k)
            if (k < nf) {
              v[k] = nbr(k, 0);
              S4 = f4_add(S4, v[k]);
            }
          if (deg > A.kstage) {
            const int* rb = g.a2b_rev + static_cast<size_t>(a) * g.wmax;
            for (int k = A.kstage; k < deg; ++k) S4 = f4_add(S4, ld_f4(src_c + static_cast<size_t>(__ldg(rb + k)) * ld));
          }
#pragma unroll
          for (int k = 0; k < kFast; ++k)
            if (k < nf) {
              const size_t off = static_cast<size_t>(wrow[k]) * ld;
              const float4 d = f4_sub(S4, v[k]);
              if (FUSED) epilogue(d, nbr(k, 1), (A.acc_mode == 2 && !A.acc_red) ? nbr(k, 2) : f4_zero(), off);
              else st_f4(out_c + off, d);
            }
          if (deg > A.kstage) {
            const int* ib = g.a2b + static_cast<size_t>(a) * g.wmax;
            const int* rb = g.a2b_rev + static_cast<size_t>(a) * g.wmax;
            for (int k = A.kstage; k < deg; ++k) {
              const size_t off = static_cast<size_t>(__ldg(ib + k)) * ld;
              const float4 d = f4_sub(S4, ld_f4(src_c + static_cast<size_t>(__ldg(rb + k)) * ld));
              if (FUSED) epilogue(d, ld_f4(y_c + off), (A.acc_mode == 2 && !A.acc_red) ? ld_f4(acc_c + off) : f4_zero(), off);
              else st_f4(out_c + off, d);
            }
          }
          pad_acc = f4_fma(static_cast<float>(pad_count), S4, pad_acc);
          pad_acc = f4_sub(pad_acc, self);
        } else if (OP == NBR_FWD) {
          float4 acc = f4_zero();
          if (pad_count > 0) acc = f4_scale(static_cast<float>(pad_count), pad_value(prow));
#pragma unroll
          for (int k = 0; k < kFast; ++k)
            if (k < nf) {
              const float4 x = nbr(k, 0);
              acc = f4_add(acc, A.relu_src ? f4_relu(x) : x);
            }
          if (deg > A.kstage) {
            const int* tb = (A.which ? g.a2a : g.a2b) + static_cast<size_t>(a) * g.wmax;
            for (int k = A.kstage; k < deg; ++k) {
              const float4 x = ld_f4(src_c + static_cast<size_t>(__ldg(tb + k)) * ld);
              acc = f4_add(acc, A.relu_src ? f4_relu(x) : x);
            }
          }
          st_f4(out_c + static_cast<size_t>(a) * ld, acc);
        } else if (OP == NBR_BWD_BOND) {
          const float4 d = lds4(base + own_off_t);
#pragma unroll
          for (int k = 0; k < kFast; ++k)
            if (k < nf) {
              const size_t off = static_cast<size_t>(wrow[k]) * ld;
              if (FUSED) epilogue(d, nbr(k, 0), (A.acc_mode == 2 && !A.acc_red) ? nbr(k, 1) : f4_zero(), off);
              else st_f4(out_c + off, d);
            }
          if (deg > A.kstage) {
            const int* ib = g.a2b + static_cast<size_t>(a) * g.wmax;
            for (int k = A.kstage; k < deg; ++k) {
              const size_t off = static_cast<size_t>(__ldg(ib + k)) * ld;
              if (FUSED) epilogue(d, ld_f4(y_c + off), (A.acc_mode == 2 && !A.acc_red) ? ld_f4(acc_c + off) : f4_zero(), off);
              else st_f4(out_c + off, d);
            }
          }
          pad_acc = f4_fma(static_cast<float>(pad_count), d, pad_acc);
        } else {  // NBR_BWD_ATOM
          float4 acc = f4_zero();
#pragma unroll
          for (int k = 0; k < kFast; ++k)
            if (k < nf) acc = f4_add(acc, nbr(k, 0));
          if (deg > A.kstage) {
            const int* ab = g.a2a + static_cast<size_t>(a) * g.wmax;
            for (int k = A.kstage; k < deg; ++k) acc = f4_add(acc, ld_f4(src_c + static_cast<size_t>(__ldg(ab + k)) * ld));
          }
          if (!is_pad) {
            const size_t off = static_cast<size_t>(a) * ld;
            if (FUSED) epilogue(acc, lds4(base + own_off_t + own_stride), (A.acc_mode == 2 && !A.acc_red) ? lds4(base + own_off_t + 2 * own_stride) : f4_zero(), off);
            else st_f4(out_c + off, acc);
          }
          pad_acc = f4_fma(static_cast<float>(pad_count), lds4(base + own_off_t), pad_acc);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty + st);
      if (++st == S) {
        st = 0;
        ph ^= 1;
      }
    }
    if constexpr (DET) {
      if (REDUCES && active && pad_row >= 0) pad_part_store(A.pp, unit, pad_j, pad_row, ld, c4, pad_acc);
    } else {
      if (REDUCES && active && pad_row >= 0) red_add_f4(out_c + static_cast<size_t>(pad_row) * ld, pad_acc);
    }
  }
}

// The padding rows collect their gradient with atomics, so their fused ReLU-backward runs afterwards: one block per row.
__global__ void k_pad_rows_act(float* __restrict__ out, const int* __restrict__ rows, int n_rows, int ld, const float* __restrict__ y, float scale, int preact,
                               float* __restrict__ acc, int acc_mode, int skip_out) {
  const int r = blockIdx.x;
  if (r >= n_rows) return;
  const size_t base = static_cast<size_t>(__ldg(rows + r)) * ld;
  for (int c = threadIdx.x * 4; c < ld; c += blockDim.x * 4) {
    const float4 o = mask_scale(*reinterpret_cast<const float4*>(out + base + c), ld_f4(y + base + c), scale, preact);
    if (!skip_out) st_f4(out + base + c, o);
    if (acc_mode == 1) st_f4(acc + base + c, o);
    else if (acc_mode == 2) st_f4(acc + base + c, f4_add(*reinterpret_cast<const float4*>(acc + base + c), o));
  }
}

// Deterministic mode: out[rows[r]] = the entries tagged rows[r].  One block per row: threadIdx.x walks the row's 16-byte chunks, and each
// of the blockDim.y slices adds a fixed contiguous run of entries in entry order (four loads in flight; an entry of another row adds an
// exact 0); the slices' sums are then added in slice order.  The partition depends only on the entry count and the row width.
__global__ void k_pad_rows_sum(float* __restrict__ out, const int* __restrict__ rows, int ld, const float* __restrict__ parts,
                               const int* __restrict__ tags, long long entries) {
  extern __shared__ float4 slice_sum[];
  const int row = __ldg(rows + blockIdx.x);
  const int c = threadIdx.x * 4;
  const long long per = (entries + blockDim.y - 1) / blockDim.y;
  const long long e_beg = per * threadIdx.y, e_end = min(entries, e_beg + per);
  float4 acc = f4_zero();
  if (c < ld) {
    long long e = e_beg;
    for (; e + 4 <= e_end; e += 4) {
      float4 v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = __ldg(tags + e + q) == row ? ld_f4(parts + (e + q) * ld + c) : f4_zero();
#pragma unroll
      for (int q = 0; q < 4; ++q) acc = f4_add(acc, v[q]);
    }
    for (; e < e_end; ++e)
      if (__ldg(tags + e) == row) acc = f4_add(acc, ld_f4(parts + e * ld + c));
  }
  slice_sum[threadIdx.y * blockDim.x + threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < ld) {
    for (int y = 1; y < static_cast<int>(blockDim.y); ++y) acc = f4_add(acc, slice_sum[y * blockDim.x + threadIdx.x]);
    st_f4(out + static_cast<size_t>(row) * ld + c, acc);
  }
}

}  // namespace pipe

long long pad_parts_bytes(int n_atoms, int n_segments, int ld) {
  const long long cpr = ld >> 2;
  const long long v1_units = static_cast<long long>(num_sms()) * 4 * (cpr < 256 ? 256 / cpr : 1);
  const long long pipe_units = static_cast<long long>(num_sms()) * 32;
  const long long U = v1_units > pipe_units ? v1_units : pipe_units;
  long long entries = U * n_segments;
  if (entries > n_atoms + 2 * U) entries = n_atoms + 2 * U;   // a unit meets at most as many padding rows as it has atoms
  return entries * (static_cast<long long>(ld) * 4 + 4) + 64;
}

int pad_parts_setup(void* scratch, long long bytes, long long units, long long atoms_per_unit, int n_segments, int ld, PadParts* pp, cudaStream_t s) {
  // Segments are concatenated (rr_graph), so a unit walking its atoms upwards meets each padding row in one run: at most
  // min(n_segments, its atoms) of them.
  long long jcap = atoms_per_unit < n_segments ? atoms_per_unit : n_segments;
  if (jcap < 1) jcap = 1;
  const long long entries = units * jcap;
  const long long need = entries * (static_cast<long long>(ld) * 4 + 4);
  if (scratch == nullptr || need > bytes) return fail(RR_ERR_WORKSPACE, "deterministic padding rows: scratch of %lld bytes < %lld", bytes, need);
  pp->parts = static_cast<float*>(scratch);
  pp->tags = reinterpret_cast<int*>(static_cast<char*>(scratch) + entries * ld * 4);
  pp->jcap = static_cast<int>(jcap);
  pp->entries = entries;
  RR_CUDA(cudaMemsetAsync(pp->tags, 0xFF, static_cast<size_t>(entries) * sizeof(int), s));
  return RR_OK;
}

int pad_rows_sum(float* out, const int* rows, int n_rows, int ld, const PadParts& pp, cudaStream_t s) {
  if (n_rows <= 0) return RR_OK;
  const int tx = ((ld >> 2) + 31) / 32 * 32, ty = 1024 / tx;
  pipe::k_pad_rows_sum<<<n_rows, dim3(tx, ty), static_cast<size_t>(tx) * ty * sizeof(float4), s>>>(out, rows, ld, pp.parts, pp.tags, pp.entries);
  RR_LAUNCH_CHECK("k_pad_rows_sum");
  return RR_OK;
}

// Host side: returns RR_ERR_UNSUPPORTED (without launching) when the shape does not suit the pipeline, so callers can use the first-generation kernel.
int rowpipe_launch(int op, const rr_graph* g, int which, const float* src, float* out, int ld, int relu_src, const float* y, float scale, int preact,
                   float* acc, int acc_mode, int skip_out, cudaStream_t s, void* det, long long det_bytes, PadParts* pp) {
  using namespace pipe;
  Args A{};
  A.g = *g;
  A.op = op;
  A.ld = ld;
  A.relu_src = relu_src;
  A.which = which;
  A.src = src;
  A.out = out;
  A.y = y;
  A.scale = scale;
  A.preact = preact;
  A.acc = acc;
  A.acc_mode = y ? acc_mode : 0;
  A.skip_out = y ? skip_out : 0;
  const int cpr = ld >> 2;
  if (cpr < 1 || cpr > 256 || (ld & 3)) return RR_ERR_UNSUPPORTED;
  A.row_bytes = ld * 4;
  const bool fused = y != nullptr;
  A.kstage = kFast;   // a kernel argument, not a constant: compiled with a constant kFast the bond-row backward ran 2 % slower (B200, 1000 W)
  // measured (scripts/bench_mp.py): the bond-row backward gains 30 % (273 -> 190 us) from reducing into acc, the atom-row backward, whose
  // accumulator rows are one contiguous bulk copy per stage, loses 13 %: every acc element is added to exactly once, so both are deterministic
  A.acc_red = (op == BOND_BWD);
  const bool stage_acc = fused && A.acc_mode == 2 && !A.acc_red;
  switch (op) {
    case BOND_FWD: A.n_nbr = 1; A.n_own = 0; break;
    case BOND_BWD: A.n_nbr = fused ? (stage_acc ? 3 : 2) : 1; A.n_own = 0; break;
    case NBR_FWD: A.n_nbr = 1; A.n_own = 0; break;
    case NBR_BWD_BOND: A.n_nbr = fused ? (stage_acc ? 2 : 1) : 0; A.n_own = 1; break;
    default: A.n_nbr = 1; A.n_own = fused ? (stage_acc ? 3 : 2) : 1; break;
  }
  for (int consumers = MAX_CONSUMERS; consumers >= 256; consumers -= 256) {
    A.consumer_warps = consumers / 32;
    A.apb = consumers / cpr;
    if (A.apb > 32) A.apb = 32;
    A.stage_bytes = A.apb * TASK_BYTES + A.apb * (A.kstage * A.n_nbr + A.n_own) * A.row_bytes;
    A.stage_bytes = (A.stage_bytes + 127) / 128 * 128;
    A.stages = SMEM_BUDGET / A.stage_bytes;
    if (A.stages > MAX_STAGES) A.stages = MAX_STAGES;
    if (A.stages >= 4) break;
  }
  if (A.stages < 2) return RR_ERR_UNSUPPORTED;
  A.n_stage_total = (g->n_atoms + A.apb - 1) / A.apb;
  A.producers = A.stages < PRODUCERS ? A.stages : PRODUCERS;
  A.round_stages = 32 / A.apb;
  if (A.round_stages > A.stages / A.producers) A.round_stages = A.stages / A.producers;
  if (A.round_stages < 1) A.round_stages = 1;
  int grid = num_sms();
  if (grid > A.n_stage_total) grid = A.n_stage_total;
  const size_t smem = 128 + 256 + static_cast<size_t>(A.stages) * A.stage_bytes;
  const bool det_op = det != nullptr && (op == BOND_BWD || op == NBR_BWD_BOND || op == NBR_BWD_ATOM);
  if (det_op) {
    RR_TRY(pad_parts_setup(det, det_bytes, static_cast<long long>(grid) * A.apb, (A.n_stage_total + grid - 1) / grid, g->n_segments, ld, &A.pp, s));
    *pp = A.pp;
  }
#define RR_PIPE_LAUNCH1(OPV, F, D)                                                                                          \
  do {                                                                                                                      \
    static PerDeviceOnce attr_set;                                                                                           \
    if (attr_set.need()) {                                                                                                        \
      RR_CUDA(cudaFuncSetAttribute(k_rowpipe<OPV, F, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BUDGET + 1024));   \
      attr_set.mark();                                                                                                      \
    }                                                                                                                       \
    RR_CUDA(launch_pdl(k_rowpipe<OPV, F, D>, dim3(grid), dim3(A.consumer_warps * 32 + 32 * PRODUCERS), smem, s, A));                                                                    \
  } while (0)
#define RR_PIPE_LAUNCH(OPV, F)                      \
  do {                                              \
    if (det_op) RR_PIPE_LAUNCH1(OPV, F, true);      \
    else RR_PIPE_LAUNCH1(OPV, F, false);            \
  } while (0)
  switch (op) {
    case BOND_FWD: RR_PIPE_LAUNCH1(BOND_FWD, false, false); break;
    case BOND_BWD: if (fused) RR_PIPE_LAUNCH(BOND_BWD, true); else RR_PIPE_LAUNCH(BOND_BWD, false); break;
    case NBR_FWD: RR_PIPE_LAUNCH1(NBR_FWD, false, false); break;
    case NBR_BWD_BOND: if (fused) RR_PIPE_LAUNCH(NBR_BWD_BOND, true); else RR_PIPE_LAUNCH(NBR_BWD_BOND, false); break;
    case NBR_BWD_ATOM: if (fused) RR_PIPE_LAUNCH(NBR_BWD_ATOM, true); else RR_PIPE_LAUNCH(NBR_BWD_ATOM, false); break;
    default: return fail(RR_ERR_INVALID, "rowpipe: unknown op %d", op);
  }
#undef RR_PIPE_LAUNCH
#undef RR_PIPE_LAUNCH1
  RR_LAUNCH_CHECK("k_rowpipe");
  return RR_OK;
}

int pad_rows_act(float* out, const int* rows, int n_rows, int ld, const float* y, float scale, int preact, float* acc, int acc_mode, int skip_out,
                 cudaStream_t s) {
  if (n_rows <= 0) return RR_OK;
  pipe::k_pad_rows_act<<<n_rows, 128, 0, s>>>(out, rows, n_rows, ld, y, scale, preact, acc, acc_mode, skip_out);
  RR_LAUNCH_CHECK("k_pad_rows_act");
  return RR_OK;
}

}  // namespace rr
