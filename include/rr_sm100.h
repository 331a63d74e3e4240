/* librr_sm100 -- C ABI of the B200-native ReactRanker training hot path.
 *
 * The reference (IannLiu/ReactRanker) has no FFI/plugin layer: the path is Python that
 * launches stock ATen kernels (SURVEY.md §2b).  This header is therefore the NEW drop-in
 * boundary (SURVEY.md §8b); each entry point cites the reference call site it replaces
 * (paths relative to the reference root, package reactranker/).  INTEGRATION.md shows the
 * ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every pointer is a DEVICE pointer borrowed for the duration of the call unless its
 *     name starts with h_ ; the library allocates nothing persistent.
 *   - every function returns 0 on success or a negative rr_status; rr_last_error() gives
 *     the message (thread-local).  Work is enqueued on `stream` (a cudaStream_t passed as
 *     void*); asynchronous CUDA faults surface at the caller's next synchronisation.
 *   - activations are fp32 row-major [rows, ld] with ld a multiple of 4 (16-byte rows);
 *     the padded hidden width hp = rr_padded(hidden) has its columns [hidden, hp) zero.
 *   - graph indices are int32.  A launch may concatenate several reference batches
 *     ("segments", e.g. one per RankNet group); each keeps its own padding rows and its
 *     own max_num_bonds through rr_atom_meta, which reproduces the reference's
 *     "a2b right-padded with 0 => row 0 is gathered" semantics (featurization.py:281-286,
 *     SURVEY.md §0 trap 1) without materialising the padded slots.
 */
#ifndef RR_SM100_H
#define RR_SM100_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RR_ABI_VERSION 3
#define RR_ATOM_FDIM 61   /* features/featurization.py:63 */
#define RR_BOND_FDIM 22   /* features/featurization.py:64 */
#define RR_FBOND_TOTAL 83 /* models/base_model.py:129     */
#define RR_FA_LD 64       /* padded row stride of f_atoms on the device */
#define RR_FB_LD 88       /* padded row stride of f_bonds on the device */
#define RR_MAX_FFN 4
#define RR_OUT_LD 16      /* padded width of the last FFN layer's output */

typedef enum {
  RR_OK = 0,
  RR_ERR_INVALID = -1,     /* bad shape / alignment / argument            */
  RR_ERR_CUDA = -2,        /* a CUDA runtime call failed                  */
  RR_ERR_ARCH = -3,        /* device is not sm_100                        */
  RR_ERR_UNSUPPORTED = -4, /* legal in the reference, not built here yet  */
  RR_ERR_WORKSPACE = -5    /* workspace too small                         */
} rr_status;

/* per-atom record (16 bytes, one vector load) */
typedef struct {
  int32_t deg_flags; /* bits 0..7 in-degree, bit 8: this row is a segment's padding atom */
  int32_t pad_count; /* max_num_bonds(segment) - in-degree: multiplicity of the pad row  */
  int32_t pad_bond;  /* row of the segment's padding bond  (0 in a single batch)         */
  int32_t pad_atom;  /* row of the segment's padding atom  (0 in a single batch)         */
} rr_atom_meta;

/* One batched graph = BatchMolGraph.get_components() + get_a2a() (featurization.py:292-329)
 * in device layout. */
typedef struct {
  int32_t n_atoms;    /* rows incl. padding atoms  (BatchMolGraph.n_atoms)              */
  int32_t n_bonds;    /* rows incl. padding bonds  (BatchMolGraph.n_bonds)              */
  int32_t n_mols;     /* len(a_scope)                                                   */
  int32_t wmax;       /* row stride of a2b/a2b_rev/a2a = max in-degree over the launch  */
  int32_t n_segments; /* reference batches concatenated in this launch                  */
  const float* f_atoms;        /* [n_atoms, RR_FA_LD]   cols >= 61 zero                 */
  const float* f_bonds;        /* [n_bonds, RR_FB_LD]   cols >= 83 zero                 */
  const rr_atom_meta* a_meta;  /* [n_atoms]                                             */
  const int32_t* a2b;          /* [n_atoms, wmax] incoming bond rows, first deg valid   */
  const int32_t* a2b_rev;      /* [n_atoms, wmax] b2revb[a2b]                           */
  const int32_t* a2a;          /* [n_atoms, wmax] b2a[a2b]  (get_a2a)                   */
  const int32_t* mol_start;    /* [n_mols] a_scope starts                               */
  const int32_t* mol_size;     /* [n_mols] a_scope sizes                                */
  const int32_t* pad_bonds;    /* [n_segments] padding bond rows                        */
  const int32_t* pad_atoms;    /* [n_segments] padding atom rows                        */
} rr_graph;

/* Device-resident molecule store: the MolGraph cache of Parsing_features (load_reactions.py:540-586) kept in HBM.
 * Molecule i owns atoms [atom_off[i], atom_off[i]+n_atoms[i]) and bonds [bond_off[i], ...) of the concatenated arrays;
 * indices inside a molecule are local (MolGraph numbering, featurization.py:135-210, b2revb = b xor 1). */
typedef struct {
  const float* f_atoms;      /* [sum A, RR_FA_LD]                                   */
  const float* f_bonds;      /* [sum B, RR_FB_LD]                                   */
  const int32_t* n_atoms;    /* [n_molecules]                                       */
  const int32_t* n_bonds;    /* [n_molecules]                                       */
  const int64_t* atom_off;   /* [n_molecules]                                       */
  const int64_t* bond_off;   /* [n_molecules]                                       */
  const int32_t* deg;        /* [sum A] in-degree                                   */
  const int32_t* a2b_start;  /* [sum A] start of the atom's list in a2b_flat, local */
  const int32_t* a2b_flat;   /* [sum B] incoming bonds per atom, local bond ids     */
  const int32_t* b2a;        /* [sum B] source atom of each bond, local             */
} rr_mol_store;

typedef enum {
  RR_HEAD_RAW = 0,
  RR_HEAD_EVIDENTIAL_RANKING = 1, /* base_model.py:91-98   (score, softplus + 1e-6) interleaved      */
  RR_HEAD_GAUSS_SOFTPLUS = 2,     /* base_model.py:71-82   (mu, softplus)                            */
  RR_HEAD_SOFTPLUS = 3,           /* base_model.py:99-100                                            */
  RR_HEAD_LOGNORM = 4,            /* base_model.py:83-90   (softplus + 1e-6, softplus + 1e-6)        */
  RR_HEAD_SOFTPLUS_P1 = 5,        /* base_model.py:101-104 softplus + 1                              */
  RR_HEAD_NIG = 6                 /* base_model.py:61-70   (mu, sp + 1e-6, sp + 1 + 1e-6, sp + 1e-6), task_num % 4 == 0 */
} rr_head;

/* build_model(...) (models/base_model.py:235-297): one hidden size and one dropout for every sub-module.  rr_model_cfg_ex below gives
 * the diff encoder and the FFN their own. */
typedef struct {
  int32_t hidden;       /* hidden_size (1..4096)                          */
  int32_t depth;        /* mpnn_depth       (1..16)                       */
  int32_t diff_depth;   /* mpnn_diff_depth  (0..16; 0: no message passing, mpn.py:220-221) */
  int32_t ffn_depth;    /* ffn_depth        (1..RR_MAX_FFN)               */
  int32_t task_num;     /* width of the last layer (<= RR_OUT_LD)         */
  int32_t add_features; /* add_features_dim                               */
  int32_t head;         /* rr_head                                        */
  int32_t training;     /* nn.Module.training: dropout active             */
  float dropout;        /* p of every nn.Dropout                          */
  uint64_t seed;        /* Philox seed of this step's dropout masks       */
  /* Optional reactant de-duplication (ABI 2).  The reference repeats the reactant MolGraph once per candidate
   * (load_reactions.py:574-576); without dropout every copy gets the same encoding.  With r_atom_map != NULL the reactant graph holds
   * each distinct reactant ONCE (per segment) and r_atom_map[a] (device, int32, [p.n_atoms]) names the row of the reactant encoder's
   * output that product atom row a subtracts (base_model.py:168), padding rows included.  Exact in eval mode and at dropout 0 (the
   * gradient of the shared rows is the sum over the copies); with dropout > 0 the copies would share their masks, so callers leave
   * it NULL there.  NULL: one reactant row per product row. */
  const int32_t* r_atom_map;
} rr_model_cfg;

/* ReactionModel(mpnn_hidden_size, mpnn_diff_hidden_size, ffn_hidden_size, mpnn_dropout, mpnn_diff_dropout, ffn_dropout, ...)
 * (models/base_model.py:111-148): per-sub-module widths and dropouts.  base.hidden and base.dropout are the encoder's (MPN).  Every field is
 * required: widths in 1..4096, dropouts in [0, 1).  The diff encoder reads the encoder's width (W_i [diff_hidden, hidden]) and the FFN's
 * first layer diff_hidden + add_features.  Dropout sites: the encoder's messages and atom hiddens take base.dropout, the diff encoder's
 * diff_dropout, the readout vector and the FFN's hidden layers ffn_dropout.  r_atom_map is refused while training if any of the three
 * is > 0. */
typedef struct {
  rr_model_cfg base;
  int32_t diff_hidden;  /* mpnn_diff_hidden_size */
  int32_t ffn_hidden;   /* ffn_hidden_size       */
  float diff_dropout;   /* mpnn_diff_dropout     */
  float ffn_dropout;    /* ffn_dropout           */
} rr_model_cfg_ex;

/* Parameters in the reference's state_dict layout (row-major [out, in], SURVEY.md §5); he / hd / hf: the encoder's, diff encoder's
 * and FFN's hidden size (all = hidden with rr_model_cfg).  NULL bias = use_bias False.  encoder.W_h is needed for depth > 1,
 * diff_encoder.W_h for diff_depth > 1, diff_encoder.W_o for diff_depth > 0.  The same struct with writable pointers receives the
 * gradients (overwritten, not accumulated).  In that role a NULL pointer means "not needed": the tensor's gradient is neither computed
 * nor written (a frozen parameter).  A split weight is one tensor (encoder.W_o, diff_encoder.W_h, diff_encoder.W_o). */
typedef struct {
  float* enc_Wi; float* enc_bi;   /* encoder.W_i   [he, 83]        mpn.py:50  */
  float* enc_Wh; float* enc_bh;   /* encoder.W_h   [he, he]        mpn.py:57  */
  float* enc_Wo; float* enc_bo;   /* encoder.W_o   [he, 61+he]     mpn.py:59  */
  float* dif_Wi; float* dif_bi;   /* diff_encoder.W_i [hd, he]     mpn.py:161 */
  float* dif_Wh; float* dif_bh;   /* diff_encoder.W_h [hd, hd+83]  mpn.py:165 */
  float* dif_Wo; float* dif_bo;   /* diff_encoder.W_o [hd, he+hd]  mpn.py:168 */
  float* ffn_W[RR_MAX_FFN];       /* ffn.ffn.{1,4,7,..}: (hd+add) -> hf -> ... -> task_num  base_model.py:40-56 */
  float* ffn_b[RR_MAX_FFN];
} rr_params;

/* ---- library ------------------------------------------------------------------------ */
int rr_version(void);
const char* rr_last_error(void);
/* fails with RR_ERR_ARCH unless `device` is compute capability 10.x */
int rr_device_check(int device);
/* padded hidden width used by every activation buffer */
int rr_padded(int width);

/* ---- batch assembly on the device (replaces the host BatchMolGraph build + the per-step feature upload) ---------- */
/* Writes every array of `out` (whose sizes and device buffers the caller provides) for the molecules mol_ids[0..n_mols)
 * placed at atom rows a_start[i] / bond rows b_start[i]; mol_W / mol_pad_bond / mol_pad_atom give each molecule's
 * segment (max_num_bonds and padding rows), seg_* list the segments' padding rows.  Result == the host-packed graph. */
int rr_graph_assemble(const rr_mol_store* store, int n_mols, const int32_t* mol_ids, const int32_t* a_start, const int32_t* b_start,
                      const int32_t* mol_W, const int32_t* mol_pad_bond, const int32_t* mol_pad_atom, int n_segments,
                      const int32_t* seg_pad_atom, const int32_t* seg_pad_bond, const int32_t* seg_W, const rr_graph* out, void* stream);

/* Host side of the same step (HOST pointers only, no device work): the control block rr_graph_assemble reads, for the molecules
 * h_ids[0..n_mols) (store ids, segments back to back, h_seg_lens molecules each), laid out exactly as the reference lays out one
 * BatchMolGraph per segment (featurization.py:246-290): one padding row, then the molecules' rows; max_num_bonds = max(1, largest
 * in-degree) unless h_W_override[s] (>= that) is given -- data-parallel shards pass the global batch's value.
 *   h_ctl  int32[6 n_mols + 3 n_segments]: [ids | a_start | b_start | W | pad_bond | pad_atom] per molecule, [a0 | b0 | W] per segment;
 *          pass its device copy to rr_graph_assemble as (ctl, ctl + n, ctl + 2n, ..., ctl + 6n, ctl + 6n + S, ctl + 6n + 2S)
 *   h_dims int64[5]: n_atoms, n_bonds, n_mols, wmax, n_segments of the graph;   h_seg_* int64[n_segments], optional (NULL): rows / W per segment
 * Replaces the host arithmetic of load_reactions.py:549-578 + featurization.py:246-290 (SURVEY.md 8b: rr_batch_build). */
int rr_batch_build(int n_mols, const int32_t* h_ids, int n_store, const int32_t* h_store_n_atoms, const int32_t* h_store_n_bonds,
                   const int32_t* h_store_max_degree, int n_segments, const int64_t* h_seg_lens, const int64_t* h_W_override,
                   int32_t* h_ctl, int64_t* h_dims, int64_t* h_seg_atoms, int64_t* h_seg_bonds, int64_t* h_seg_W);

/* ---- message passing (models/mpn.py) -------------------------------------------------- */
/* mpn.py:89-92   pre[b] = (sum_k m[a2b[b2a[b],k]]) - m[b2revb[b]]   for every bond row.
 * relu_src != 0 applies relu() to m on load (m0 = relu(input), mpn.py:81). */
int rr_bond_message_fwd(const rr_graph* g, const float* m, float* pre, int hp, int relu_src, void* stream);
/* backward of the above: dm from dpre (gather-only; padding rows reduced with atomics) */
int rr_bond_message_bwd(const rr_graph* g, const float* dpre, float* dm, int hp, void* stream);
/* mpn.py:100-102 / 201 / 215: out[a] = sum_k src[idx[a,k]] incl. padding multiplicity.
 * which: 0 = a2b over bond rows (pad row = pad_bond), 1 = a2a over atom rows (pad_atom). */
int rr_neighbor_sum_fwd(const rr_graph* g, int which, const float* src, float* out, int ld, int relu_src, void* stream);
/* backward of which=0: dsrc[b] = dout[atom b points into]; of which=1: symmetric gather */
int rr_neighbor_sum_bwd(const rr_graph* g, int which, const float* dout, float* dsrc, int ld, void* stream);
/* The two backward gathers fused with the ReLU / inverted-dropout backward that follows them in MPN / MPNDiff (autograd of
 * mpn.py:81,95-97,208-213): dz = gather_bwd(...) * [y != 0] * scale  (y_is_preact: [y > 0]), written to dm / dsrc unless skip_out,
 * and acc = dz (acc_mode 1) or acc += dz (acc_mode 2).  y == NULL: the plain gather backward. */
int rr_bond_message_bwd_act(const rr_graph* g, const float* dpre, float* dm, int hp, const float* y, float scale, int y_is_preact,
                            float* acc, int acc_mode, int skip_out, void* stream);
int rr_neighbor_sum_bwd_act(const rr_graph* g, int which, const float* dout, float* dsrc, int ld, const float* y, float scale,
                            int y_is_preact, float* acc, int acc_mode, int skip_out, void* stream);
/* mpn.py:224-238: vec[i] = mean(hid[a_scope[i]])[:hidden] || add_features[i] (zero padded to vp),
 * then the FFN's first dropout (base_model.py:40).  hid is [n_atoms, hp], vec is [n_mols, vp]. */
int rr_readout_fwd(const rr_graph* g, const float* hid, int hp, int hidden, const float* add_features, int n_add,
                   float* vec, int vp, float dropout, uint64_t seed, uint64_t stream_id, void* stream);
/* backward, fused with the relu/dropout mask of hid: dz[a] = dvec[mol(a)]/size * [hid!=0]*scale (the same dropout p on vec and hid) */
int rr_readout_bwd(const rr_graph* g, const float* dvec, int vp, const float* vec, const float* hid, float* dz,
                   int hp, float dropout, void* stream);

/* ---- dense layers (nn.Linear call sites of mpn.py / base_model.py) -------------------- */
/* Y[M,n] = act(X1 W1^T + X2 W2^T + bias + residual), W* row-major [n_pad, k*] zero padded.
 * flags: bit0 relu, bit1 dropout(p, seed, stream_id) after relu. X2/W2/bias/residual may be NULL. */
int rr_linear_fwd(int M, int n, const float* X1, int ldx1, const float* W1, int k1,
                  const float* X2, int ldx2, const float* W2, int k2, const float* bias,
                  const float* residual, int ldr, float* Y, int ldy, int flags, float dropout,
                  uint64_t seed, uint64_t stream_id, void* stream);
/* Which GEMM implementation the dense layers use.  TC = the tcgen05 tensor cores (TMA-fed, accumulating in TMEM) where the shape suits
 * them, the exact-fp32 SIMT kernels otherwise:
 *   mode | forward | dgrad of rr_model_backward | wgrad           | padding rows of rr_model_forward
 *    0   | SIMT    | SIMT                       | SIMT            | as computed
 *    1   | TC      | TC                         | TC for M >= 256 | recomputed in exact arithmetic, also where a shape fell back to SIMT
 *    2   | TC      | SIMT                       | SIMT            | recomputed, as in mode 1
 *    3   | SIMT    | TC                         | SIMT            | as computed
 * rr_linear_dgrad is SIMT in every mode, rr_linear_dgrad_tc TC in every mode.  A TC GEMM splits its fp32 operands into 3 x TF32 products
 * (fp32-class accuracy, ~1e-6 relative) or 3 x bf16 products, as the two switches below select.  Process-wide. */
int rr_set_gemm_mode(int mode);
int rr_get_gemm_mode(void);
/* Operand split of the BACKWARD tensor-core GEMMs (dgrad and wgrad; gradients never decide a ReLU mask): 1 (default) = 3 x bf16 products
 * (x = bf16(x) + bf16(x - bf16(x)): 16 significand bits per operand, fp32 accumulation, ~5e-6 relative, half the tensor-pipe time),
 * 0 = the forward's 3 x tf32 split.  Process-wide; the Python package sets it from RR_BWD_BF16 when it loads the library. */
int rr_set_backward_bf16(int on);
int rr_get_backward_bf16(void);
/* Operand split of the FORWARD tensor-core GEMMs of rr_model_forward: 0 (default) = 3 x tf32, 1 = the backward's 3 x bf16 split (same
 * kernel, half the tensor-pipe time and operand bytes; 16 instead of 21 significand bits per operand).  rr_linear_fwd always takes 3 x tf32.
 * Process-wide; the Python package sets it from RR_FWD_BF16 when it loads the library. */
int rr_set_forward_bf16(int on);
int rr_get_forward_bf16(void);
/* Deterministic mode (torch.use_deterministic_algorithms of the Python package): 1 = every kernel rr_model_backward and
 * rr_loss_fwdbwd(_ex) launch produces the same bits on every run for identical inputs, in every GEMM mode, backward split and gather
 * generation.  The sums the default path forms with atomics (weight-gradient row slabs, segment padding rows, loss parts) are written as
 * partials with plain stores and added in a fixed order instead.  The guarantee holds on one GPU model with one build of this library:
 * the weight gradient's slab count follows the SM count, so a part with a different SM count may round differently.
 * Scratch: rr_model_workspace_bytes includes it when the switch is on (rr_model_backward fails with RR_ERR_WORKSPACE, writing nothing,
 * if the workspace was sized without it); entry points without a workspace take it from the stream-ordered allocator (cudaMallocAsync /
 * cudaFreeAsync on `stream`) in this mode only.  rr_model_backward with rr_model_cfg.r_atom_map returns RR_ERR_UNSUPPORTED in this mode
 * when an encoder gradient is requested (the sum over shared reactant rows lives in the encoder's backward only).
 * on must be 0 (default) or 1, else RR_ERR_INVALID.  Process-wide. */
int rr_set_deterministic(int on);
int rr_get_deterministic(void);
/* dX[M,k] (+)= dZ[M,n] W[n,k]   (accumulate != 0 adds) */
int rr_linear_dgrad(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw,
                    float* dX, int lddx, int accumulate, void* stream);
/* The same dX (+)= dZ W on the tcgen05 tensor cores, in the operand split rr_set_backward_bf16 selects (the kernel rr_model_backward uses:
 * autograd of every nn.Linear of mpn.py / base_model.py).  The model keeps transposed, pre-split images of its weights; a direct caller
 * provides `scratch` (device, 16-byte aligned, >= rr_linear_dgrad_tc_scratch_bytes(n, k)) for them.  Needs k % 16 == 0 and n % 4 == 0
 * (RR_ERR_UNSUPPORTED otherwise). */
int64_t rr_linear_dgrad_tc_scratch_bytes(int n, int k);
int rr_linear_dgrad_tc(int M, int n, int k, const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx,
                       int accumulate, void* scratch, int64_t scratch_bytes, void* stream);
/* dW[n,k] += dZ^T X ; dbias[n] += colsum(dZ) when dbias != NULL.  Caller zeroes dW/dbias. */
int rr_linear_wgrad(int M, int n, int k, const float* dZ, int lddz, const float* X, int ldx,
                    float* dW, int lddw, float* dbias, void* stream);
/* dz = dy * [y != 0] * scale (relu + inverted-dropout backward); acc (+)= dz when acc != NULL:
 * acc_mode 0 none, 1 acc = dz, 2 acc += dz.  y_is_preact: mask is [y > 0]. */
int rr_relu_bwd(int64_t rows, int ld, const float* dy, const float* y, float scale, int y_is_preact,
                float* dz, float* acc, int acc_mode, void* stream);
/* out = a - b  (models/base_model.py:168) */
int rr_sub(int64_t n, const float* a, const float* b, float* out, void* stream);

/* ---- LTR losses (train/loss.py, train/train_pairwise.py) ------------------------------- */
/* All take scores [N] (or [N,2]), targets [N], seg_off [G+1] (prefix sums of `scope`) and
 * return the loss in loss[0] and dL/dscore in dscore, normalised exactly like the reference. */
typedef enum {
  RR_LOSS_LISTMLE = 0,    /* MLEloss            loss.py:64-99   (+LogCumsumExp 9-61)      */
  RR_LOSS_LISTNET = 1,    /* ListnetLoss        loss.py:317-352                            */
  RR_LOSS_EVIDENTIAL = 2, /* evidential_ranking loss.py:477-556 (scores [N,2])             */
  RR_LOSS_RANKNET = 3,    /* sum_session        train_pairwise.py:98-122,141-147           */
  RR_LOSS_GAUSS = 4,      /* GaussDisLoss       loss.py:144-162 (scores [N,2])             */
  RR_LOSS_MSE = 5,        /* nn.MSELoss         train_listwise.py:166-167                  */
  RR_LOSS_EXPMSE = 6,     /* mean((e^t - e^s)^2) train_listwise.py:276-281 ('regression_exploss') */
  RR_LOSS_LISTMLE_DIS = 7,/* MLEDisLoss        loss.py:102-141 (scores [N,2] = mean, variance; norm = groups) */
  RR_LOSS_LISTNET_DIS = 8,/* Listnet_For_Gauss loss.py:233-272 (scores [N,2]; norm = groups, items averaged per group) */
  RR_LOSS_LISTNET_UQ = 9, /* Listnet_with_uq   loss.py:355-399 (positive scores; `sigma` carries the annealing coefficient) */
  RR_LOSS_RANKNET_ACC = 10,/* RankNet 'accelerate_grad' train_pairwise.py:123-137: same cost, dscore = the row sums only (half of autograd's) */
  RR_LOSS_LOGNORM = 11,   /* Lognorm           loss.py:165-184 (scores [N,2] = m, v, both positive; norm = N) */
  RR_LOSS_DIRICHLET_UQ = 12,/* Dirichlet_uq    loss.py:440-474 (1-D positive concentrations; `sigma` = annealing coefficient; norm = groups) */
  RR_LOSS_NIG = 13,       /* evidential_loss_new loss.py:402-437 as called at train_listwise.py:229-260: scores [N,4] = mu, v, alpha, beta
                             against EVERY target of the batch (the [N,1] x [N] broadcast); norm = N*N; `sigma` = lam; no seg_off */
  RR_LOSS_LAMBDARANK = 14,/* LambdaRank: RankNet over each group's pairs t_i > t_j (each once), weighted by |dNDCG| of swapping them; norm = groups */
  RR_LOSS_LAMBDARANK_TOP = 15 /* the same with the NDCG cut at K = max(1, round_half_even(n / 4)), the validation's NDCG@25% */
} rr_loss_kind;
/* norm: the divisor the reference applies (G, N or the window's ordered-pair count); sigma: RankNet, LambdaRank */
int rr_loss_fwdbwd(int kind, int N, int G, const float* scores, const float* targets, const int32_t* seg_off,
                   float norm, float sigma, float* loss, float* dscore, void* stream);
/* The same with the size of the largest group given (the caller has `scope` on the host): ListMLE, RankNet and LambdaRank keep a group in shared
 * memory and size it for max_group, up to rr_loss_max_group() = 8192 candidates.  rr_loss_fwdbwd assumes groups of at most 2048; a
 * group larger than the capacity yields NaN in loss and dscore, never a shared-memory overrun. */
int rr_loss_fwdbwd_ex(int kind, int N, int G, const float* scores, const float* targets, const int32_t* seg_off, int max_group,
                      float norm, float sigma, float* loss, float* dscore, void* stream);
/* largest group the segmented kernels accept */
int rr_loss_max_group(void);

/* Per-group ranking metrics of the validation pass, replacing the host loops of eval.py:475-555 (ranking_metrics) and 76-177
   (evaluate_top_scores): scores stay on the device, RR_METRIC_COLS doubles per group come back.
     scores  [N * score_ld] fp32, the ranking score of item i at scores[i * score_ld] (score_ld = task_num picks column 0 of a [N, task] output)
     targets [N] fp64 (the DataFrame column as is, so ties and order are the reference's), seg_off [G + 1], max_group <= 8192
     ratio   the top fraction (0.25 everywhere in the reference): K = max(1, round-half-even(n * ratio)), Python's round()
   out [G, 8]: 0 predicted top-1 == true top-1 | 1 |pred top-K n true top-K| / K | 2 predicted top-1 in true top-K | 3 true top-1 in predicted
   top-K | 4 NDCG@1 | 5 NDCG@2 as eval.py:544 computes it | 6 NDCG@K | 7 NDCG@all.  Stable descending order (ties keep the earlier item).
   An empty group yields zeros; a group larger than max_group yields NaN in all eight columns. */
#define RR_METRIC_COLS 8
int rr_rank_metrics(int N, int G, const float* scores, int score_ld, const double* targets, const int32_t* seg_off, int max_group,
                    double ratio, double* out, void* stream);

/* Per-item ranking statistics of a prediction pass (reactranker_b200/predict.py) over T samples of the scores: T = 1 for one eval-mode
   forward, T > 1 for MC dropout (one train-mode forward per sample).  No targets: one CTA per group, nothing but the table comes back.
     scores  fp32, item i of sample t at scores[t * sample_stride + i * score_ld] (score_ld = task_num picks column 0 of [N, task] outputs)
     seg_off [G + 1], max_group <= rr_loss_max_group() = 8192, T >= 1
   out [N, RR_PREDICT_COLS] fp32, one row per item:
     0 mean of the score over the samples | 1 its standard deviation, population form (ddof 0; 0 when T = 1) | 2 1-based rank of column 0
     within the group | 3 mean over samples of the within-group softmax (ListNet / Plackett-Luce probability of ranking first) | 4 fraction
     of samples in which the item ranks first | 5 mean over samples of the item's rank.
   Ranks are the stable descending order of k_rank_metrics (rank(i) = 1 + #{j : x_j > x_i} + #{j < i : x_j == x_i}); column 2 ranks the
   fp32 value of column 0, so it is the stable order of the returned means.  The softmax is shifted by the group maximum and every sum is
   taken in double without atomics: a repeated call is bit-identical.  An empty group writes nothing; a group larger than max_group gets
   NaN in all of its rows. */
#define RR_PREDICT_COLS 6
int rr_rank_predict(int N, int G, int T, const float* scores, int64_t sample_stride, int score_ld, const int32_t* seg_off, int max_group,
                    float* out, void* stream);

/* ---- whole model (models/base_model.py:150-171) ---------------------------------------- */
/* bytes of workspace rr_model_forward/backward need for these sizes */
int64_t rr_model_workspace_bytes(const rr_model_cfg* cfg, const rr_graph* r, const rr_graph* p);
/* Byte offset, inside the workspace, of a forward activation saved for backward -- for per-layer parity tests.
 * Names: enc{0,1}.inp, enc{0,1}.pre<t>, enc{0,1}.m<t+1>, enc{0,1}.am, enc{0,1}.hid (0 = reactants, 1 = products),
 * d, inp2, nf, nm<t>, m2_<t+1>, am2, hid2, vec, x<l>, zout.  -1 on error, and for inp2 / nf / am2 at diff_depth 0, where they do not exist. */
int64_t rr_model_buffer_offset(const rr_model_cfg* cfg, const rr_graph* r, const rr_graph* p, const char* name);
/* scores: [n_mols] if task_num==1 else [n_mols, task_num].  ws must stay untouched until the
 * matching rr_model_backward has run. */
int rr_model_forward(const rr_model_cfg* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p,
                     const float* add_features, float* scores, void* ws, int64_t ws_bytes, void* stream);
/* dscores has the shape of scores; grads receives d/d(parameter) in state_dict layout.  Only the non-NULL gradients of grads are
 * computed (see rr_params): layers in graph order are encoder W_i < W_h < W_o < diff encoder W_i < W_h < W_o < FFN 0 .. F-1, and the
 * backward runs through a layer only while some tensor below it is requested; nothing below the lowest requested tensor is launched.
 * A weight gradient is launched only when the weight is requested; a requested bias under a NULL weight gets its own column-sum
 * kernel (bit-identical run to run in both modes).  All NULL: RR_OK without a launch.  With every pointer set the result and the
 * launches are those of the full backward. */
int rr_model_backward(const rr_model_cfg* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p,
                      const float* dscores, rr_params* grads, void* ws, int64_t ws_bytes, void* stream);
/* The same four with per-sub-module widths and dropouts.  The entry points above are these with diff_hidden = ffn_hidden = hidden and
 * diff_dropout = ffn_dropout = dropout; a workspace sized by one must be used with a configuration of the same widths. */
int64_t rr_model_workspace_bytes_ex(const rr_model_cfg_ex* cfg, const rr_graph* r, const rr_graph* p);
int64_t rr_model_buffer_offset_ex(const rr_model_cfg_ex* cfg, const rr_graph* r, const rr_graph* p, const char* name);
int rr_model_forward_ex(const rr_model_cfg_ex* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p,
                        const float* add_features, float* scores, void* ws, int64_t ws_bytes, void* stream);
int rr_model_backward_ex(const rr_model_cfg_ex* cfg, const rr_params* w, const rr_graph* r, const rr_graph* p,
                         const float* dscores, rr_params* grads, void* ws, int64_t ws_bytes, void* stream);
/* Per-kernel-class device timing for bench.py's roofline: between begin and end every launch is bracketed by
 * CUDA events on its own stream; end() waits for them and returns summed milliseconds / launch counts per class
 * (0 gemm_fwd 1 gemm_dgrad 2 gemm_wgrad 3 bond_fwd 4 bond_bwd 5 nbr_fwd 6 nbr_bwd 7 readout 8 elementwise 9 loss 10 misc). */
int rr_profile_begin(void);
int rr_profile_end(double* h_ms_by_class, int64_t* h_launches_by_class, int n_classes);
int rr_profile_classes(void);
/* The RR_MP_V1 environment switch (first-generation gather kernels instead of the row pipeline) is read once, at first use; this reads it
 * again. */
void rr_reload_switches(void);
/* kernels launched on this thread since the last reset (for bench.py's gpu_launches) */
int64_t rr_launch_count(void);
void rr_launch_count_reset(void);

#ifdef __cplusplus
}
#endif
#endif /* RR_SM100_H */
