/*
 * egc_b200.h - C ABI of libegc_b200.so: the B200 (sm_100a) implementation of the EGConv
 * message-passing hot path of shyam196/egc.
 *
 * Every entry point is what a binding of the reference's hot path would call instead of the
 * torch / torch_scatter / torch_sparse / torch_geometric leaf ops.  "ref" citations are
 * relative to /root/reference/ (experiments/optimized_layers.py unless another file is named).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless marked host;
 *   - every function returns 0 (EGC_OK) or a negative egc_status; the message of the last
 *     failure on the calling thread is available from egc_last_error_string();
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); nothing here
 *     allocates or frees caller-visible memory or synchronises the device; scratch space is
 *     a caller-owned workspace whose size comes from the matching *_workspace_bytes();
 *   - features are fp32 (the *_bf16 entry points: bf16 basis rows, see there), row-major, contiguous; graph indices are int32 on the device
 *     (the reference's int64 edge_index / rowptr / col are narrowed by the build functions);
 *   - target-major CSR: row i lists the sources j of the messages node i receives
 *     (= the reference's `adj_t`, ref experiments/utils.py:107-109).
 */
/*
 * Environment switches read once per process (A/B and diagnostics; none changes results except EGC_TC_ABLATE):
 *   EGC_FWD_WARP_PER_ROW=1     forward aggregation: warp-per-row kernel instead of the row-block kernel
 *   EGC_BWD_WARP_PER_COLUMN=1  backward CSC pass: warp-per-column kernel instead of the column-block kernel
 *   EGC_TC_NO_TMA=1            projection GEMM: cp.async producers instead of TMA tensor copies for the A operand
 *   EGC_TC_NO_SWIZZLE=1        projection GEMM: four 16-byte TMA boxes per A chunk instead of one 64-byte-swizzled box
 *   EGC_TC_TMA_STORE=1         projection GEMM: TMA tensor-store epilogue (measured equal to the default)
 *   EGC_TC_MAX_RAW_STAGES=n    projection GEMM: cap the A ring depth (at least 4)
 *   EGC_WGRAD_TRANSPOSE=1      parameter gradients: the transposing kernel (k_wgrad_tc) instead of the MN-major one
 *                              (k_wgrad_mn); it partitions the nodes differently, so results differ in the last bits
 *   EGC_TC_ABLATE=bits         projection GEMM: switch pipeline stages off for timing (WRONG results; tools/gemm_ablate.sh)
 */
#ifndef EGC_B200_H_
#define EGC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EGC_ABI_VERSION 5
#define EGC_MAX_AGGR 8          /* len(aggrs) accepted by one layer */
#define EGC_CHUNK_EDGES 256     /* rows longer than this are split into chunks of this many nnz */

typedef enum egc_status {
  EGC_OK = 0,
  EGC_ERR_INVALID_ARGUMENT = -1,
  EGC_ERR_CUDA = -2,
  EGC_ERR_UNSUPPORTED = -3,
  EGC_ERR_WORKSPACE = -4
} egc_status;

/* Aggregator codes, ref :93 {"sum","mean","symnorm","min","max","var","std"}. */
typedef enum egc_aggr {
  EGC_AGGR_SUM = 0,
  EGC_AGGR_MEAN = 1,
  EGC_AGGR_SYMNORM = 2,
  EGC_AGGR_MIN = 3,
  EGC_AGGR_MAX = 4,
  EGC_AGGR_VAR = 5,
  EGC_AGGR_STD = 6
} egc_aggr;

/* Shape of one EGConv layer invocation (ref :96-108, :195-202). */
typedef struct egc_layer_desc {
  int32_t n_dst;                 /* target nodes = CSR rows = rows of weightings / out            */
  int32_t n_src;                 /* source nodes = rows of bases (== n_dst for EGConv)            */
  int32_t heads;                 /* H                                                             */
  int32_t bases;                 /* B                                                             */
  int32_t dim;                   /* D = out_channels / H; a basis row has B*D floats              */
  int32_t n_aggr;                /* A = len(aggrs), 1..EGC_MAX_AGGR                               */
  int32_t aggr[EGC_MAX_AGGR];    /* egc_aggr codes in the order given to the constructor          */
  int32_t sigmoid;               /* weightings went through sigmoid (ref :183-184)                */
  int32_t relu;                  /* fused epilogue of the stack around the layer (ref mag/models.py:63): out = max(out, 0);
                                    the backward then masks grad_out with out > 0 (egc_aggregate_bwd `out_act`)   */
} egc_layer_desc;

/* Optional fused epilogue of egc_aggregate_fwd (the stack around the layer, SURVEY section 8 f-1), applied per output
 * element c of row i in this order:   y = out[i, c] (+ bias)  ->  y = y * scale[c] + shift[c]  (BatchNorm in eval mode,
 * folded: scale = gamma / sqrt(var + eps), shift = beta - mean * scale; ref arxiv/norm_models.py:35)  ->  y = max(y, 0)
 * when desc->relu (ref :36, mag/models.py:63)  ->  y += add[i, c]  (the residual of ref :38-39, or the running sum of
 * REGConv's relation terms, rmag/models.py:146; `add` may alias `out`).  Any pointer may be NULL. */
typedef struct egc_epilogue {
  const float* scale;            /* [H*D] or NULL (then shift must be NULL too)                  */
  const float* shift;            /* [H*D] or NULL                                                */
  const float* add;              /* [n_dst, H*D] or NULL                                         */
  const float* agg_init;         /* [n_dst, A, B*D] or NULL: partial aggregates of an earlier call over ANOTHER entry subset
                                    of the same rows (agg_out of that call; sum / symnorm aggregators only): added to this
                                    call's sums before they are saved and combined, so  call(local sources) -> call(halo
                                    sources, agg_init) = one call over all of them.  May alias agg_out / saved.          */
} egc_epilogue;

/* Row plan: how long rows of a CSR (or columns of its CSC) are split into chunks so that no
 * warp walks more than EGC_CHUNK_EDGES nnz.  Built once per graph by egc_plan_build(). */
typedef struct egc_row_plan {
  int32_t n_long;                /* rows with more than EGC_CHUNK_EDGES nnz                       */
  int32_t n_chunks;              /* total chunks over those rows                                  */
  const int32_t* long_rows;      /* [n_long]    row id                                            */
  const int32_t* long_chunk_ptr; /* [n_long+1]  first chunk of each long row                      */
  const int32_t* chunk_row;      /* [n_chunks]  row id of the chunk                               */
  const int32_t* chunk_begin;    /* [n_chunks]  first nnz of the chunk; it ends at min(begin+EGC_CHUNK_EDGES, row end) */
} egc_row_plan;

int egc_abi_version(void);
const char* egc_last_error_string(void);      /* host string, valid until the thread's next failing call */
/* compile-time facts of the loaded binary, for INTEGRATION / smoke checks */
const char* egc_build_info(void);

/* Launch accounting / tracing (the reference has no tracing at all, SURVEY.md section 5).
 * egc_launch_count(): kernels launched by this library in this process (always counted).
 * egc_profile_enable(1): from now on every kernel launch is bracketed by CUDA events on its stream;
 * egc_profile_collect() synchronises those events and writes one "name,launches,total_ms\n" line per
 * kernel name into buf (returns the number of bytes written, negative on error) and clears the table. */
uint64_t egc_launch_count(void);
int egc_profile_enable(int32_t on);
int egc_profile_collect(char* buf /* host */, size_t capacity);

/* ------------------------------------------------------------------------------------------
 * Graph preparation (bit-exact integer work)
 * ---------------------------------------------------------------------------------------- */

/* meta[] slots written (device int32[8]) by the graph builders */
#define EGC_META_NNZ 0          /* nnz of the produced CSR                                        */
#define EGC_META_MAX_DEG 1      /* longest row                                                    */
#define EGC_META_N_LONG 2       /* rows longer than EGC_CHUNK_EDGES                               */
#define EGC_META_N_CHUNKS 3     /* chunks over those rows                                         */
#define EGC_META_N_LOOPS 4      /* self-loops appended                                            */
#define EGC_META_SLOTS 8

/* loops: how self-loops are handled for an edge_index input */
#define EGC_LOOPS_NONE 0        /* add_self_loops=False: graph used untouched                     */
#define EGC_LOOPS_ALL_NODES 1   /* gcn_norm(..., num_nodes=N) -> add_remaining_self_loops, ref :131-137 */
#define EGC_LOOPS_UP_TO_MAX_ID 2/* add_remaining_self_loops(edge_index) without num_nodes, ref :164:
                                   only nodes <= edge_index.max() get a loop                      */

size_t egc_csr_from_edges_workspace_bytes(int64_t n_edges, int32_t n_nodes);
/* edge_index (int64, row 0 = source j, row 1 = target i; ref :128-141 / :159-166) -> target-major CSR.
 * Existing self-loops are dropped and one loop per node is appended AFTER all other edges
 * (PyG add_remaining_self_loops); rows keep the edge order of the input (stable sort by target), so
 * "first element wins" ties of min/max resolve as in torch_scatter.
 * Outputs: rowptr[n_nodes+1], col[capacity n_edges + n_nodes] (first meta[NNZ] valid), meta[8]. */
int egc_csr_from_edges(const int64_t* src, const int64_t* dst, int64_t n_edges, int32_t n_nodes,
                       int32_t loops, int32_t* rowptr, int32_t* col, int32_t* meta,
                       void* workspace, size_t workspace_bytes, void* stream);

/* SparseTensor input (ref :143-156, :168-175; torch_sparse fill_diag): narrows an int64 CSR to int32
 * and, if fill_diag != 0, removes every diagonal entry and inserts one per i < min(n_dst, n_src) at
 * its sorted position (diagonal value 1.0 when the matrix carries values).
 * value_in may be NULL.  Outputs: rowptr[n_dst+1], col / value_out [capacity nnz_in + min(n_dst,n_src)], meta[8]. */
size_t egc_csr_fill_diag_workspace_bytes(int32_t n_dst);
int egc_csr_fill_diag(const int64_t* rowptr_in, const int64_t* col_in, const float* value_in,
                      int32_t n_dst, int32_t n_src, int32_t fill_diag, int32_t* rowptr, int32_t* col,
                      float* value_out, int32_t* meta, void* workspace, size_t workspace_bytes, void* stream);

/* gcn_norm (ref :131-137, :146-152): deg[i] = sum of row i's values (nnz count when value == NULL),
 * dis = deg^-1/2 with inf -> 0, val_sym[e] = (value[e] * dis[row(e)]) * dis[col(e)].
 * Requires n_src == n_dst when called for EGConv.  deg / dis may be NULL if not wanted. */
int egc_symnorm_weights(const int32_t* rowptr, const int32_t* col, const float* value, int32_t n_dst,
                        float* deg, float* dis, float* val_sym, void* stream);

/* CSC view used by the backward pass (the reference caches torch_sparse's csr2csc,
 * ref experiments/utils.py:111-113): colptr[n_src+1], rowidx[nnz] (target of each entry),
 * csr2csc[nnz] (CSR position of each CSC entry; stable, i.e. targets ascending inside a column). */
size_t egc_csr_transpose_workspace_bytes(int32_t nnz, int32_t n_dst, int32_t n_src);
int egc_csr_transpose(const int32_t* rowptr, const int32_t* col, int32_t nnz, int32_t n_dst, int32_t n_src,
                      int32_t* colptr, int32_t* rowidx, int32_t* csr2csc, int32_t* meta,
                      void* workspace, size_t workspace_bytes, void* stream);

/* out[k] = in[perm[k]] for fp32 per-nnz values (CSR order -> CSC order). */
int egc_permute_f32(const float* in, const int32_t* perm, int32_t n, float* out, void* stream);

/* Chunk plan of the long rows of a CSR (meta[N_LONG], meta[N_CHUNKS] give the array sizes). */
int egc_plan_build(const int32_t* rowptr, int32_t n_rows, int32_t n_long, int32_t n_chunks,
                   int32_t* long_rows, int32_t* long_chunk_ptr, int32_t* chunk_row, int32_t* chunk_begin,
                   void* workspace, size_t workspace_bytes, void* stream);
size_t egc_plan_build_workspace_bytes(int32_t n_rows);

/* ------------------------------------------------------------------------------------------
 * Dense projections  (ref :180 `torch.matmul(x, bases_weight)`, :182-184 `comb_weight(x)` [+ sigmoid])
 * ---------------------------------------------------------------------------------------- */

#define EGC_GEMM_AUTO 0         /* tcgen05 3xTF32 when the shape allows, else fp32 FFMA            */
#define EGC_GEMM_FP32_SIMT 1    /* exact fp32 FFMA tiles (any shape)                               */
#define EGC_GEMM_3XTF32 2       /* tcgen05 kind::tf32, 3-term split: fp32-level accuracy           */
#define EGC_GEMM_TF32 3         /* tcgen05 kind::tf32, single pass (~1e-3 relative)                */

/* Shapes and alignment of the tensor-core path: f_in, bd and hab multiples of 4 and the weights resident in shared memory
 * next to the operand ring (the forward's and d_x's); the tensors a tensor-core kernel streams 16-byte aligned:
 *   forward: x, bases, weightings and b_comb (when not NULL);
 *   d_x:     d_bases, d_lin and d_x;
 *   d_w_bases / d_w_comb: x, d_bases and d_lin.
 * Contiguous tensors at a storage offset need not be.  EGC_GEMM_AUTO takes the fp32 FFMA kernels for a product whose
 * shape or tensors do not qualify; EGC_GEMM_3XTF32 / EGC_GEMM_TF32 return EGC_ERR_UNSUPPORTED for the forward and d_x
 * instead, while the parameter gradients fall back to the FFMA kernels under every algorithm. */

/* bases[n, bd] = x[n, f_in] . w_bases[f_in, bd]
 * weightings[n, hab] = act(x . w_comb[hab, f_in]^T + b_comb[hab]),  act = sigmoid if `sigmoid`. */
int egc_project_fwd(const float* x, const float* w_bases, const float* w_comb, const float* b_comb,
                    int32_t n, int32_t f_in, int32_t bd, int32_t hab, int32_t sigmoid,
                    float* bases, float* weightings, int32_t algo, void* stream);

/* Opt-in bf16 storage of the basis rows (round to nearest even, packed [n, bd] bf16 = uint16_t bit patterns; bd % 4 == 0 on
 * the tensor-core path): the same products as egc_project_fwd, accumulated in fp32, rounded once when stored.  weightings
 * stay fp32.  The consumers of such `bases` are egc_aggregate_fwd_bf16 / egc_aggregate_bwd_bf16. */
int egc_project_fwd_bf16(const float* x, const float* w_bases, const float* w_comb, const float* b_comb,
                         int32_t n, int32_t f_in, int32_t bd, int32_t hab, int32_t sigmoid,
                         uint16_t* bases, float* weightings, int32_t algo, void* stream);

/* Autograd of the two projections (ref: implicit backward of :180-182).  d_lin is the gradient
 * w.r.t. the pre-activation of comb_weight (sigmoid' already applied by egc_aggregate_bwd).
 *   d_x[n,f_in]       = d_bases . w_bases^T + d_lin . w_comb        (d_x may be NULL)
 *   d_w_bases[f_in,bd] = x^T . d_bases ; d_w_comb[hab,f_in] = d_lin^T . x ; d_b_comb[hab] = colsum(d_lin)
 * Parameter gradients are OVERWRITTEN (not accumulated). */
size_t egc_project_bwd_workspace_bytes(int32_t n, int32_t f_in, int32_t bd, int32_t hab);
int egc_project_bwd(const float* x, const float* w_bases, const float* w_comb,
                    const float* d_bases, const float* d_lin, int32_t n, int32_t f_in, int32_t bd, int32_t hab,
                    float* d_x, float* d_w_bases, float* d_w_comb, float* d_b_comb,
                    int32_t algo, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused multi-aggregator CSR SpMM + per-node/per-head combination
 * (ref :191 propagate -> :215-249 aggregate / :251-278 message_and_aggregate, :195-208 combine + bias)
 * ---------------------------------------------------------------------------------------- */

/* out[i, h*D+d] = bias[h*D+d] + sum_{a,b} weightings[i, h*A*B + a*B + b] * agg_a(i)[b*D + d]
 * where agg_a(i) reduces bases[j, :] over the nnz of CSR row i with aggregator a:
 *   sum / mean (divide by nnz count, min 1) / symnorm (weights val_sym) / min / max (empty row -> 0,
 *   first nnz wins ties) / var = mean(x^2) - mean(x)^2 / std = sqrt(relu(var) + 1e-5).
 * val_sym: per-nnz weights for symnorm (required iff symnorm is requested).
 * val_lin: per-nnz weights applied by every other aggregator (NULL = unweighted; only a valued
 *          SparseTensor without symnorm produces them, ref :256-258).
 * bias may be NULL.  row_subset (may be NULL = all rows): only these rows (of at most EGC_CHUNK_EDGES nnz) are
 * computed as row tasks - a row-partitioned caller aggregates interior rows while the halo exchange is in
 * flight and the boundary rows afterwards; the long rows of `plan` are processed whenever plan != NULL.
 * Every output is optional (NULL to skip), at least one must be given:
 *   out[n_dst, H*D]           the layer output (needs weightings)
 *   agg_out[n_dst, A, B*D]    the aggregated bases before combination (ref :249 / :278)
 *   arg_out[n_dst, A, B*D]    int32 nnz position of the winning element for min/max slots (-1: empty row,
 *                             other slots -1); source id = col[arg]
 *   saved[n_dst, S, B*D]      what egc_aggregate_bwd needs, S = egc_saved_slots(): slot a < A = agg_a (std slots
 *                             negated when relu(var) gated the gradient off), slot A = mean when var/std is present
 *   saved_arg[n_dst, R, B*D]  winning nnz positions of the R = egc_saved_arg_slots() min/max aggregators. */
int32_t egc_saved_slots(const egc_layer_desc* desc);
int32_t egc_saved_arg_slots(const egc_layer_desc* desc);
size_t egc_aggregate_fwd_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* plan);
int egc_aggregate_fwd(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col,
                      const float* val_sym, const float* val_lin, const egc_row_plan* plan,
                      const float* bases, const float* weightings, const float* bias, const egc_epilogue* epilogue,
                      const int32_t* row_subset, int32_t n_subset,
                      float* out, float* agg_out, int32_t* arg_out, float* saved, int32_t* saved_arg,
                      void* workspace, size_t workspace_bytes, void* stream);

/* egc_aggregate_fwd over bf16 basis rows (from egc_project_fwd_bf16): every value is widened to fp32 before any arithmetic,
 * so sums, means, variances and the min/max winners (first nnz wins ties) are those of egc_aggregate_fwd on the widened rows;
 * every output stays fp32 / int32.  Covers B*D in 40..128 with B*D % 8 == 0 and H*D <= 512 (128 when D % 4 != 0), no per-nnz
 * linear weights (val_lin), no row subset and no epilogue agg_init; 16-byte aligned tensors.  Other shapes return
 * EGC_ERR_INVALID_ARGUMENT.  Workspace: egc_aggregate_fwd_workspace_bytes() (never NULL). */
int egc_aggregate_fwd_bf16(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_sym,
                           const egc_row_plan* plan, const uint16_t* bases, const float* weightings, const float* bias,
                           const egc_epilogue* epilogue, float* out, float* agg_out, int32_t* arg_out, float* saved,
                           int32_t* saved_arg, void* workspace, size_t workspace_bytes, void* stream);

/* Training-mode dropout after the fused ReLU (ref mag/models.py:63-64), applied to `out` inside the same epilogue.  The mask
 * is a pure function of (seed, global row, column):
 *   key     = (low 32 bits of *seed, high 32 bits of *seed)         (*seed is read by the kernel: a replayed CUDA graph
 *                                                                    sees whatever the seed buffer holds at replay time)
 *   r       = word (c & 3) of Philox4x32-10(counter = (c >> 2, row_offset + i, 0, 0), key)   for output (i, c), c < H*D
 *   keep    = r < min(floor((1 - p) * 2^32), 2^32 - 1),  k = fp32(1 / (1 - p)),  both from the fp32 `p` widened to double
 *   out     = keep ? relu(y) * k : 0
 * A row-partitioned caller passes its first global row as row_offset and gets its rows of the single-GPU mask.  p == 0 is no
 * dropout; 0 < p < 1 needs desc->relu, `out`, and an epilogue without scale / shift / add (agg_init is allowed: it continues
 * the sums before the combination).  Anything else returns EGC_ERR_INVALID_ARGUMENT.  The backward needs no mask:
 * out > 0 exactly where the ReLU was open and the element kept, so egc_aggregate_bwd with out_act = out and epi_scale = a
 * [H*D] vector filled with k is the exact ReLU + dropout backward. */
typedef struct egc_dropout {
  const uint64_t* seed;          /* device, one word                                              */
  float p;                       /* drop probability, 0 <= p < 1                                  */
  int64_t row_offset;            /* global id of local row 0; row_offset + n_dst <= 2^32          */
} egc_dropout;

/* egc_aggregate_fwd / egc_aggregate_fwd_bf16 with dropout (NULL: the calls above, which are these with dropout = NULL). */
int egc_aggregate_fwd_dropout(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_sym,
                              const float* val_lin, const egc_row_plan* plan, const float* bases, const float* weightings,
                              const float* bias, const egc_epilogue* epilogue, const egc_dropout* dropout,
                              const int32_t* row_subset, int32_t n_subset, float* out, float* agg_out, int32_t* arg_out,
                              float* saved, int32_t* saved_arg, void* workspace, size_t workspace_bytes, void* stream);
int egc_aggregate_fwd_bf16_dropout(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_sym,
                                   const egc_row_plan* plan, const uint16_t* bases, const float* weightings, const float* bias,
                                   const egc_epilogue* epilogue, const egc_dropout* dropout, float* out, float* agg_out,
                                   int32_t* arg_out, float* saved, int32_t* saved_arg, void* workspace, size_t workspace_bytes,
                                   void* stream);

/* Backward of the above (ref: autograd of :191-208; torch_sparse spmm backward over the cached CSC).
 * Pass 1 (per target, streaming over `saved`): d_weightings (times sigmoid' when desc->sigmoid; = gradient
 * w.r.t. the Linear output) and the target-side streams t_sym / t_lin / t_sq; min/max gradients are routed
 * to the single winning source (fp32 atomics into d_bases).  Pass 2 (CSC, per source, atomic-free):
 *   d_bases[j] = sum_e val_sym[e] t_sym[i_e] + val_lin[e] (t_lin[i_e] + 2 bases[j] t_sq[i_e]) + routed.
 * rowptr / col / val_lin are the CSR of the forward (row nnz counts, arg -> source id); colptr / rowidx /
 * csc_val_sym / csc_val_lin its CSC view from egc_csr_transpose + egc_permute_f32 (values NULL like
 * their CSR twins); csr2csc (egc_csr_transpose; may be NULL unless EGC_BWD_DETERMINISTIC is set and the layer has a
 * min/max aggregator) = CSR position of every CSC entry.  The routed min/max gradients are added AFTER pass 2, which
 * writes every row of d_bases.  d_bias (may be NULL) = column sums of grad_out; d_lin_colsum (may be NULL) = column sums of
 * d_weightings = gradient of the comb-weight bias (ref :108, :182), produced here because pass 1 has the rows in
 * registers - egc_project_bwd then takes d_b_comb = NULL.  out_act: the forward's `out` (required iff desc->relu, else
 * NULL): pass 1 uses grad_out[i, c] * (out_act[i, c] > 0) - with an epilogue `add`, pass the post-activation value
 * BEFORE the add (out - add).  epi_scale (or NULL): the forward epilogue's scale; pass 1 multiplies the masked gradient
 * by it (scale / shift themselves are constants: no gradient is produced for them); the gradient w.r.t. `add` is
 * grad_out itself.  d_bias then is the gradient of the bias INSIDE the epilogue (masked and scaled).  Column sums: pass 1
 * accumulates d_bias and d_lin_colsum in registers while H*A*B <= 128 and H*D <= 512 (<= 128 when D % 4 != 0); wider
 * layers take a two-stage column sum after the passes, which applies the same mask and scale to grad_out - so the fused
 * epilogue has no width limit of its own.  tstreams_out (or NULL):
 * where pass 1 writes the target-side streams [n_dst, L, B*D] instead of the workspace (see egc_aggregate_bwd_cols).
 * flags: EGC_BWD_*. */
#define EGC_BWD_DETERMINISTIC 1 /* route min/max gradients with a compare-and-add gather over the CSC instead of fp32
                                   atomics: bit-reproducible from run to run (needs csr2csc; two more gathered rows per
                                   entry and min/max slot) */
#define EGC_BWD_SKIP_ROUTING 4  /* diagnostics only: drop the min/max gradient routing (results are then incomplete) */
#define EGC_BWD_NO_HUB_PRIVATISATION 8 /* tuning: route min/max gradients of hub sources (long CSC columns) with global
                                   fp32 atomics like every other source instead of per-CTA shared-memory accumulators */
#define EGC_BWD_COLS_HEAD 128   /* column phases of a row-partitioned caller (source columns = [own | halo], col_split = number
                                   of own columns): HEAD = pass 1, the min/max routing and pass 2 of the columns >= col_split,
                                   so the halo partial sums can travel to their owners while ...                           */
#define EGC_BWD_COLS_TAIL 256   /* ... TAIL = pass 2 of the columns < col_split runs (same arguments and workspace, after the
                                   HEAD call on the same stream).  Neither bit: the whole backward in one call.             */
size_t egc_aggregate_bwd_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* csc_plan, int32_t flags);
int egc_aggregate_bwd(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_lin,
                      const int32_t* colptr, const int32_t* rowidx, const int32_t* csr2csc, const float* csc_val_sym,
                      const float* csc_val_lin, const egc_row_plan* csc_plan,
                      const float* bases, const float* weightings, const float* saved, const int32_t* saved_arg,
                      const float* grad_out, const float* out_act, const float* epi_scale, float* d_weightings,
                      float* d_bases, float* d_bias, float* d_lin_colsum, float* tstreams_out,
                      int32_t flags, int32_t col_split, void* workspace, size_t workspace_bytes, void* stream);

/* egc_aggregate_bwd for a layer whose forward ran on bf16 basis rows (egc_aggregate_fwd_bf16): `bases` is bf16 (read by the
 * var / std term 2 bases[j] t_sq[i]) and pass 1 stores the target-side streams t_sym / t_lin / t_sq as bf16 (round to
 * nearest even) in the workspace, which pass 2 widens and sums in fp32.  saved, the routed min/max gradients, d_weightings,
 * d_bases, d_bias and d_lin_colsum are fp32 as in egc_aggregate_bwd.  No per-entry linear weights (val_lin);
 * EGC_BWD_DETERMINISTIC and the tuning flags are honoured.  The basis rows must be 36..128 values wide, a multiple of 4,
 * 16-byte aligned.  Workspace: egc_aggregate_bwd_bf16_workspace_bytes().  Equivalent to
 * egc_aggregate_bwd_bf16_partitioned(..., tstreams_out = NULL, flags, col_split = 0, ...). */
size_t egc_aggregate_bwd_bf16_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* csc_plan, int32_t flags);
int egc_aggregate_bwd_bf16(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const int32_t* colptr,
                           const int32_t* rowidx, const int32_t* csr2csc, const float* csc_val_sym, const egc_row_plan* csc_plan,
                           const uint16_t* bases, const float* weightings, const float* saved, const int32_t* saved_arg,
                           const float* grad_out, const float* out_act, const float* epi_scale, float* d_weightings,
                           float* d_bases, float* d_bias, float* d_lin_colsum, int32_t flags, void* workspace,
                           size_t workspace_bytes, void* stream);
/* egc_aggregate_bwd_bf16 for row-partitioned callers: tstreams_out and col_split mean what they mean for egc_aggregate_bwd.
 * EGC_BWD_PASS1_ONLY writes the target-side streams as bf16 (round to nearest even) into the first n_dst rows of
 * tstreams_out [rows, L, B*D] (16-byte aligned) for egc_aggregate_bwd_cols_bf16; EGC_BWD_COLS_HEAD / EGC_BWD_COLS_TAIL split
 * pass 2 at col_split (the routed min/max gradients come first and both pass-2 launches accumulate, as in fp32). */
int egc_aggregate_bwd_bf16_partitioned(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col,
                                       const int32_t* colptr, const int32_t* rowidx, const int32_t* csr2csc,
                                       const float* csc_val_sym, const egc_row_plan* csc_plan, const uint16_t* bases,
                                       const float* weightings, const float* saved, const int32_t* saved_arg,
                                       const float* grad_out, const float* out_act, const float* epi_scale, float* d_weightings,
                                       float* d_bases, float* d_bias, float* d_lin_colsum, uint16_t* tstreams_out,
                                       int32_t flags, int32_t col_split, void* workspace, size_t workspace_bytes, void* stream);

/* Pass 2 alone, for row-partitioned callers that exchange the TARGET-SIDE STREAMS instead of partial sums (layers without
 * min / max; no reference counterpart, DESIGN.md "multi-GPU"): pass 1 runs through egc_aggregate_bwd with
 * EGC_BWD_PASS1_ONLY and tstreams_out = the first n_dst rows of a table [n_rows_ext, L, B*D] (L = number of linear streams:
 * [symnorm] + [sum / mean / var / std] + [var / std], interleaved per row) whose remaining rows the peers fill with the
 * streams of their targets; this call then sums, for every OWN source column j of the TRANSPOSED local adjacency
 * (colptr / rowidx / csc_val_* = that adjacency, rowidx indexing the rows of `tstreams`; desc->n_src = number of columns,
 * desc->n_dst = rows of `tstreams`), d_bases[j] = sum_e val_sym[e] t_sym[i_e] + val_lin[e] (t_lin[i_e] + 2 bases[j] t_sq[i_e])
 * - complete, atomic-free, and over full-degree columns only.  EGC_BWD_ACCUMULATE: d_bases[j] += instead of = (a second
 * launch over another entry subset, e.g. the halo targets after the local ones).  bases may be NULL without var / std. */
#define EGC_BWD_PASS1_ONLY 512  /* egc_aggregate_bwd: stop after pass 1 (needs tstreams_out, no min / max aggregator)          */
#define EGC_BWD_ACCUMULATE 1024 /* egc_aggregate_bwd_cols: add to d_bases instead of overwriting it                            */
size_t egc_aggregate_bwd_cols_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* csc_plan);
int egc_aggregate_bwd_cols(const egc_layer_desc* desc, const int32_t* colptr, const int32_t* rowidx,
                           const float* csc_val_sym, const float* csc_val_lin, const egc_row_plan* csc_plan,
                           const float* tstreams, const float* bases, float* d_bases, int32_t flags,
                           void* workspace, size_t workspace_bytes, void* stream);
/* egc_aggregate_bwd_cols over a bf16 stream table (from egc_aggregate_bwd_bf16_partitioned with EGC_BWD_PASS1_ONLY): the
 * streams are widened and summed in fp32, `bases` are the bf16 basis rows of the columns (NULL without var / std), d_bases
 * is fp32.  No per-entry linear weights.  Workspace: egc_aggregate_bwd_cols_workspace_bytes() (its partials are fp32). */
int egc_aggregate_bwd_cols_bf16(const egc_layer_desc* desc, const int32_t* colptr, const int32_t* rowidx,
                                const float* csc_val_sym, const egc_row_plan* csc_plan, const uint16_t* tstreams,
                                const uint16_t* bases, float* d_bases, int32_t flags, void* workspace, size_t workspace_bytes,
                                void* stream);

/* ------------------------------------------------------------------------------------------
 * Row exchange for row-partitioned graphs (no reference counterpart; see DESIGN.md "multi-GPU")
 * egc_gather_rows and egc_peer_push_rows move rows without arithmetic: `width` counts 4-byte words, so a row of B*D bf16
 * values (the *_bf16 entry points; B*D % 8 == 0) passes width = B*D / 2 and still moves in whole 16-byte pieces.
 * ---------------------------------------------------------------------------------------- */

/* dst[k, :] = src[index[k], :]  (pack halo rows before a send / all-gather), width 4-byte words per row */
int egc_gather_rows(const float* src, const int32_t* index, int32_t n_index, int32_t width, float* dst, void* stream);

/* ------------------------------------------------------------------------------------------
 * NVLink peer-memory exchange (one process per GPU of a node; csrc/peer.cu).  No reference counterpart.
 * A rank allocates ONE peer segment, exports its IPC handle, and maps the segments of the other ranks.
 * Data moves by posted stores into a mapped segment (egc_peer_push_rows); ordering is by epoch flags:
 * flags of a rank = uint32 [n_slots][world] inside its segment, entry [slot][q] written by rank q only.
 * The epoch is a device-resident counter advanced by a kernel, so a step can be replayed from a CUDA graph.
 * ---------------------------------------------------------------------------------------- */
#define EGC_MAX_PEERS 8
/* segments of one egc_peer_push_rows call: one per (peer, table), e.g. 7 peers x 4 node types of a heterogeneous layer */
#define EGC_MAX_PUSH_SEGMENTS 64
typedef struct egc_ipc_handle { unsigned char bytes[64]; } egc_ipc_handle;

/* cudaMalloc + zero-fill + cudaIpcGetMemHandle (setup time; synchronises) */
int egc_peer_alloc(size_t bytes, void** ptr, egc_ipc_handle* handle);
int egc_peer_free(void* ptr);
/* map another rank's segment into this process (enables peer access lazily) / unmap it */
int egc_peer_open(const egc_ipc_handle* handle, void** ptr);
int egc_peer_close(void* ptr);

/* For each segment s < n_seg (HOST arrays src/dst/seg_ptr, n_seg <= EGC_MAX_PUSH_SEGMENTS): rows k in
 * [seg_ptr[s], seg_ptr[s+1]) of the concatenated list:  dst[s][(k - seg_ptr[s]), :] = src[s][index[k], :]
 * (index == NULL: src[s][k - seg_ptr[s], :]).  dst may point into a mapped peer segment.
 * Fused signal (flags != NULL, slot_mask != 0): the last CTA to finish, after a system-scope fence, raises
 * flags[q][slot * world + rank] = *epoch for every peer q and every slot bit of slot_mask; `counter` is a
 * device word that is zero between calls. */
int egc_peer_push_rows(int32_t n_seg, const float* const* src, float* const* dst, const int32_t* seg_ptr,
                       const int32_t* index, int32_t width, uint32_t* const* flags, int32_t world, int32_t rank,
                       uint32_t slot_mask, const uint32_t* epoch, uint32_t* counter, void* stream);

/* Stream-ordered copy of `bytes` from local memory into (or out of) a mapped peer segment by the COPY ENGINE
 * (cudaMemcpyAsync): unlike egc_peer_push_rows it occupies no SM, so it overlaps a compute kernel on another stream
 * whatever that kernel's occupancy - the rows are packed first (egc_gather_rows) and sent as one contiguous block per
 * peer.  Capturable in a CUDA graph (a memcpy node). */
int egc_peer_copy(void* dst, const void* src, size_t bytes, void* stream);

/* *epoch += 1 (device counter) */
int egc_peer_epoch_advance(uint32_t* epoch, void* stream);
/* flags[q][slot * world + rank] = *epoch for every peer q != rank and every slot bit of slot_mask (HOST array of
 * mapped flag arrays); release at system scope: everything earlier on the stream is visible to a peer that
 * observes the flag */
int egc_peer_signal(uint32_t* const* flags, int32_t world, int32_t rank, uint32_t slot_mask, const uint32_t* epoch,
                    void* stream);
/* (advance != 0: *epoch += 1 first - a new step starts.)  Block the stream until my_flags[slot * world + q] >=
 * *epoch - lag for every q != rank; after timeout_ns the kernel records *err = 1 + slot (device word) and TRAPS:
 * nothing downstream may run on stale peer data, so the stream and every later CUDA call of the process fail */
int egc_peer_wait(const uint32_t* my_flags, int32_t world, int32_t rank, int32_t slot, uint32_t* epoch,
                  uint32_t lag, int32_t advance, uint64_t timeout_ns, uint32_t* err, void* stream);

/* into[rows[r], :] += sum_{t in [ptr[r], ptr[r+1])} staging[entry[t], :]   (fixed order: deterministic) */
int egc_peer_reduce_rows(const float* staging, const int32_t* rows, const int32_t* ptr, const int32_t* entry,
                         int32_t n_rows, int32_t width, float* into, void* stream);
/* One-shot all-reduce (sum) of a small replicated vector in ONE kernel: src[n] is stored into slot [rank] of every
 * rank (slot_of_me[q] = mapped address of rank q's slot [rank], own rank included), flag `slot` is raised at *epoch,
 * the kernel waits for the same flag of every peer (traps after timeout_ns, *err = 1 + slot) and writes
 * out[i] = sum_r my_slots[r * n + i] in rank order - identical bits on every rank.  n % 4 == 0, 16-byte aligned buffers,
 * *counter == 0 on entry (and again on exit). */
int egc_peer_allreduce(const float* src, float* const* slot_of_me, const float* my_slots, uint32_t* const* flags,
                       const uint32_t* my_flags, int32_t world, int32_t rank, int32_t slot, const uint32_t* epoch,
                       uint32_t* counter, int32_t n, float* out, uint64_t timeout_ns, uint32_t* err, void* stream);

/* out[i] = sum_q slots[q * n + i] in rank order (the one-shot all-reduce of the replicated parameter gradients) */
int egc_peer_sum_slots(const float* slots, int32_t world, int32_t n, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Mini-batch plumbing (SURVEY.md section 8 f-4; csrc/batch.cu).  Replaces, on the device, what the reference
 * gets from PyG on the CPU: DataLoader / Batch.from_data_list collation (experiments/zinc/configs.py:36-45,60-67,
 * experiments/cifar/configs.py:42-53) and the graph readout global_{add,mean,max}_pool
 * (experiments/zinc/models.py:46-53,73).  Graph g of a collated batch owns the contiguous node range
 * [node_ptr[g], node_ptr[g+1]).
 * ---------------------------------------------------------------------------------------- */
#define EGC_POOL_SUM 0
#define EGC_POOL_MEAN 1  /* divides by max(count, 1), as scatter(reduce="mean") */
#define EGC_POOL_MAX 2   /* empty graph -> 0; the gradient goes to the first maximal node, as scatter_max */

/* Block-diagonal collation: edge e of graph g (edge_ptr[g] <= e < edge_ptr[g+1], graph-local node ids) becomes
 * (src + node_ptr[g], dst + node_ptr[g]); batch_out[i] (may be NULL) = graph of node i.  *flags bit 0 is raised when a
 * local id lies outside its graph. */
int egc_collate_edges(const int64_t* src_local, const int64_t* dst_local, const int32_t* edge_ptr, const int32_t* node_ptr,
                      int32_t n_graphs, int64_t n_edges, int64_t n_nodes, int64_t* src_out, int64_t* dst_out,
                      int64_t* batch_out, int32_t* flags, void* stream);
/* node_ptr [n_graphs + 1] from a sorted PyG `batch` vector.  *flags: bit 0 unsorted, bit 1 id outside [0, n_graphs). */
int egc_segment_ptr(const int64_t* batch, int64_t n, int32_t n_graphs, int32_t* ptr, int32_t* flags, void* stream);
/* out[g, :] = reduce over the nodes of graph g of x[i, :]  (x [n, f] row-major); arg [n_graphs, f] (EGC_POOL_MAX, may be
 * NULL in inference) = winning node id or -1 */
int egc_segment_pool_fwd(const float* x, const int32_t* ptr, int32_t n_graphs, int32_t f, int32_t mode, float* out,
                         int32_t* arg, void* stream);
/* d_x[i, :] for every node of every graph (all n rows are written when ptr covers them) */
int egc_segment_pool_bwd(const float* d_out, const int32_t* ptr, const int32_t* arg, int32_t n_graphs, int32_t f,
                         int32_t mode, float* d_x, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EGC_B200_H_ */
