/* ddp_b200.h -- C ABI of the B200-native DiffDock-Pocket score-model hot path.
 *
 * The reference (plainerman/DiffDock-Pocket) is pure Python; the native code it runs for this path
 * lives in third-party wheels (SURVEY.md 2.1).  Each entry point below replaces one of those call
 * sites; the Python host (diffdock_pocket_b200/*.py) binds them with ctypes and mirrors the
 * reference's operator interfaces.  Conventions:
 *   - every pointer is a DEVICE pointer unless named *_host; the caller owns all buffers,
 *     kernels never allocate; `stream` is a cudaStream_t passed as void*;
 *   - indices are int32 on the device; floating data is fp32 row-major unless stated;
 *   - dynamic edge sets live in fixed-capacity buffers `edge[2][cap]` with the live count in a
 *     device int (`n_edges_dev`), so no call needs a host synchronisation;
 *   - return value: 0 = ok, <0 = invalid argument (DDP_E_*), >0 = cudaError_t of the launch.
 *     No exceptions cross the ABI.
 */
#ifndef DDP_B200_H
#define DDP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDP_E_ARG   (-1)
#define DDP_E_SHAPE (-2)
#define DDP_E_UNSUPPORTED (-3)

/* Library / build identification ("sm_100a"). */
const char *ddp_version(void);

/* ------------------------------------------------------------------------------------------------
 * Deterministic accumulation.  The scatter-adds of the convolutions (forward and backward) add partial sums that
 * arrive in whatever order the GPU schedules them; in fp32 the low bits of the result then depend on that order.  The
 * *_fixed entry points below accumulate instead in signed 64-bit fixed point with ONE binary scale 2^S:
 *   q = llrint(v * 2^S)   per partial sum v (multiplying by a power of two is exact: one rounding, to 2^-S absolute),
 *   sum += q              integer addition is associative, so every arrival order gives the same bits,
 *   v' = (float)sum * 2^-S  once, by the consumer (ddp_node_update*_fixed, ddp_fixed_to_float).
 * S = 32: a partial may lie in (-2^31, 2^31) and is resolved to 2.3e-10.  The convolution outputs are O(1) to O(100)
 * (BatchNorm-scaled features and their mean over <= a few hundred edges), so the range leaves > 20 bits of headroom, and
 * a sum of even 10^5 partials carries at most 10^5 * 2^-33 = 1.2e-5 of rounding in ABSOLUTE terms -- more than 1e3 below the
 * 1e-4 relative / per-channel gates the fp32 path is held to, and a sum of 2^32 full-range partials cannot wrap the
 * int64.  A partial that is not finite or lies outside the range is not converted (it adds 0) and sets
 * DDP_STATUS_FIXED_RANGE in the caller's sticky device status word (uint32, zeroed by the caller, bits are OR-ed in;
 * kernels never trap): the host reads the word at a synchronisation point it already has and reports the error. */
#define DDP_ACC_FIXED_SHIFT 32
#define DDP_STATUS_FIXED_RANGE 1u

/* dst[i] = (float)src[i] * 2^-DDP_ACC_FIXED_SHIFT for i < n (the single conversion back of a fixed-point sum). */
int ddp_fixed_to_float(const int64_t *src, int64_t n, float *dst, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Graph construction.  Replaces torch_cluster.radius / radius_graph / knn_graph (pytorch-cluster
 * 1.6.1 CUDA kernels; reference call sites models/all_atom_score_model.py:457,524,545-550,563,607,627).
 * Bit-exact with those kernels: fp32 squared distance accumulated x,y,z with FMA, strict `<`,
 * first-`max_nbr` hits in ascending index order, kNN ties broken by lower index.
 *
 * ddp_radius: for every query y_j (example b given by ptr_y) scan x[ptr_x[b] .. ptr_x[b+1]).
 *   inv_scale: optional per-example divisor c_b (may be NULL): coordinates are divided by c_b
 *              before the distance test (the dynamic cross cutoff of all_atom_score_model.py:545-547).
 *   mode bit0 (DDP_RADIUS_GRAPH): x and y are the same set; the scan cap counts the centre itself
 *              (max_nbr = K+1) but the self pair is not emitted, and rows are swapped so that
 *              edge[0] = neighbour, edge[1] = centre (torch_cluster.radius_graph, flow
 *              source_to_target).  Otherwise edge[0] = j (index into y), edge[1] = i (index into x).
 *   prefix:    number of edges already present at the front of `edge` (ligand bond edges are
 *              concatenated before the radius edges, all_atom_score_model.py:466); the live count
 *              written to n_edges_dev includes it.
 *   slab:      workspace int32 [n_y * slab_w], slab_w >= min(max_nbr, longest x segment);
 *   counts:    workspace int32 [n_y + 1].
 */
#define DDP_RADIUS_GRAPH 1
int ddp_radius(const float *x, const float *y, const int32_t *ptr_x, const int32_t *ptr_y,
               int32_t num_examples, int32_t n_y, const float *inv_scale, float r, int32_t max_nbr,
               int32_t mode, int32_t prefix, int32_t *slab, int32_t slab_w, int32_t *counts,
               int32_t *edge, int32_t edge_cap, int32_t *n_edges_dev, void *stream);

/* ddp_knn_graph: torch_cluster.knn_graph(x, k, batch, loop=False): edge[0] = neighbour (ascending
 * distance per centre), edge[1] = centre.  Same workspace contract, slab_w >= k + 1. */
int ddp_knn_graph(const float *x, const int32_t *ptr, int32_t num_examples, int32_t n, int32_t k,
                  int32_t *slab, int32_t slab_w, int32_t *counts, int32_t *edge, int32_t edge_cap,
                  int32_t *n_edges_dev, void *stream);
/* Search strategy of the filtered k-NN (k = 8 / 12): 0 = ordered scan of the staged example (default), 1 = grid-binned
 * (cell list built per block in shared memory; same edge lists, measured slower at pocket sizes -- see csrc/graph.cu).
 * Returns the previous setting (-1: not set yet, DDP_KNN_GRID in the environment decides on first use). */
int ddp_knn_set_grid(int32_t mode);

/* ddp_calpha_graph: the receptor's residue contact graph, built once per complex by the reference's preprocessing
 * (datasets/process_mols.py:661-677): for every residue i of its complex the residues closer than r, in index order;
 * if there are more than max_nbr, the max_nbr nearest in ascending distance instead; if there are none, the nearest
 * one.  edge[0] = i (repeated), edge[1] = neighbour.  Same workspace contract as ddp_radius, slab_w >= max_nbr. */
int ddp_calpha_graph(const float *pos, const int32_t *ptr, int32_t num_examples, int32_t n, float r, int32_t max_nbr,
                     int32_t *slab, int32_t slab_w, int32_t *counts, int32_t *edge, int32_t edge_cap,
                     int32_t *n_edges_dev, void *stream);

/* In-degree of every node on one side of an edge list (the `count` of torch_scatter's mean,
 * models/score_model.py:117): deg[idx[e]] += 1 for e < *n_edges_dev.  deg must be zeroed by the caller. */
int ddp_degree(const int32_t *idx, const int32_t *n_edges_dev, int32_t edge_cap, int32_t *deg, void *stream);

/* Several degree counts in one launch: deg[idx[e]] += 1 for start <= e < min(*n_edges_dev, edge_cap), per job
 * (the dynamic edge sets of one forward; static ones are counted once per complex by the host). */
typedef struct { const int32_t *idx; const int32_t *n_edges_dev; int32_t edge_cap; int32_t start; int32_t *deg; } ddp_degree_job_t;
int ddp_degree_multi(const ddp_degree_job_t *jobs_host, int32_t n_jobs, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Edge geometry + edge embedding.  Replaces the per-edge-set blocks of build_*_conv_graph
 * (all_atom_score_model.py:476-481, 501-508, 527-534, 552-556, 566-570, 575-579, 594-598, 609-613):
 *   vec = pos_b[edge[1]] - pos_a[edge[0]];  sh = [1, sqrt(3) vec/|vec|];  rbf = GaussianSmearing(|vec|)
 *   emb = W2 relu(Wpre pre + Wrbf rbf + u[graph_of_edge]) + b2
 * where u = Wsig sigma_emb(t_graph) + b1 is precomputed per graph (ddp_graph_sigma_proj).
 * Outputs: sh [cap,4], emb [cap,ns].  pre (n_pre columns, e.g. the 4 bond one-hots, zero for rows
 * >= n_pre_rows) may be NULL.  graph_of_a maps node index on side a -> graph (NULL => edge[0] is
 * already the graph index, used by the centre graph).  u may be NULL (torsion-bond embedding).
 * Folded form (mlp->w2 == NULL): emb receives the hidden activations relu(...) instead; the caller has folded W2 / b2
 * into the first Linear of every convolution that consumes this edge embedding (W1[:, :ns] W2, b1 + W1[:, :ns] b2),
 * which halves the per-edge work of this kernel.
 */
typedef struct {
    const float *w_pre;  /* [n_pre][ns]  (input-major) or NULL */
    const float *w_rbf;  /* [n_rbf][ns] */
    const float *w2;     /* [ns][ns] input-major */
    const float *b2;     /* [ns] */
    const float *b1;     /* [ns], used only when u == NULL */
    const float *rbf_offset; /* [n_rbf] GaussianSmearing.offset (torch.linspace, fp32) */
    float rbf_coeff;         /* GaussianSmearing.coeff = -0.5 / (offset[1]-offset[0])^2 */
    int32_t n_pre, n_rbf, ns;
    int32_t sh_dim;          /* 4 (lmax 1) or 9 (lmax 2) */
} ddp_edge_mlp_t;

int ddp_edge_embed(const float *pos_a, const float *pos_b, const int32_t *edge, int32_t edge_cap,
                   const int32_t *n_edges_dev, const int32_t *graph_of_a, const float *pre,
                   int32_t n_pre_rows, const float *u, const ddp_edge_mlp_t *mlp,
                   float *sh, float *emb, void *stream);

/* sigma embedding + per-graph projections: sig[g] = [sin|cos]((scale * t[g]) * freq[i]) (utils/
 * diffusion_utils.py:73-84; freq = exp(-i ln(1e4)/(half-1)) tabulated by the host in fp32 exactly as
 * torch does), out[m][g][:] = W_m sig[g] + b_m for n_proj matrices of shape [sig_dim][ns]
 * (input-major) stacked in w / b.  out: [n_proj][n_graphs][ns]; sig: [n_graphs][sig_dim]. */
int ddp_graph_sigma_proj(const float *t, int32_t n_graphs, float scale, const float *freq, int32_t sig_dim,
                         const float *w, const float *b, int32_t n_proj, int32_t ns, float *sig, float *out,
                         void *stream);

/* Static (time-independent) part of AtomEncoder.forward (models/score_model.py:74-82; OldAtomEncoder :38-52 after
 * folding its two Linears on the host), computed ONCE per complex and cached (SURVEY 8(f)-1: the receptor's Linear runs
 * over 1280 ESM dims):  out[n][:] = (sum_k table[table_off[k] + cat[n][k]][:]) W_emb + lm[n][:] W_lm.
 * cat: [n][n_cat] int64 categorical features; table: all embedding tables stacked, [rows][ns]; lm: [n][n_lm] or NULL;
 * w_emb_t: [ns][ns] input-major or NULL (identity); w_lm_t: [n_lm][ns] input-major; out: [n][ns]. */
int ddp_node_static_embed(const int64_t *cat, int32_t n, int32_t n_cat, const float *table, const int32_t *table_off,
                          const float *lm, int32_t n_lm, const float *w_emb_t, const float *w_lm_t, int32_t ns,
                          float *out, void *stream);

/* node_attr[n][:ns] = static_part[n][:] + u[graph_of[n]][:]  (AtomEncoder, models/score_model.py:74-82,
 * with the time-independent part of the Linear precomputed once per complex). */
int ddp_node_init(const float *static_part, const float *u, const int32_t *graph_of, int32_t n, int32_t ns,
                  float *out, int32_t ld_out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Tensor-product convolution.  Replaces TensorProductConvLayer.forward (models/score_model.py:108-125)
 * with FasterTensorProduct (models/layers.py:34-85) or e3nn FullyConnectedTensorProduct, fused:
 *   h   = relu(W1 [emb | p1[i1[e]][:ns] | p2[i2[e]][:ns]] + b1)
 *   w   = W2 h + b2                       (never written to memory)
 *   out = TP(x[gather[e]], sh[e], w)      (row groups, see ddp_tp_group_t)
 *   sum[agg[e]] += ew[e] * out            (scatter; the mean / BatchNorm / residual are ddp_node_update)
 *
 * The tensor product is described by row groups.  Group g contributes, for each of its mul_in rows u
 * and each output channel o < mul_out, with d = d_out components k:
 *   basis[u][k] = sum_{i<d1, j<d2} C_g[i][j][k] * x[x_off + u*d1 + i] * sh[sh_off + j]
 *   out[out_off + o*d + k] += w[w_off + u*mul_out + o] * basis[u][k]
 * (C_g already carries the path normalisation: 1/sqrt(in_k) for FasterTensorProduct blocks,
 *  sqrt((2l+1)/fan_in) * wigner_3j for e3nn paths.)
 */
typedef struct {
    int32_t d1, d2, d_out;      /* 2l+1 of input irrep, sh irrep, output irrep */
    int32_t x_off, mul_in;      /* slice of the gathered node features */
    int32_t sh_off;             /* first component of the sh irrep */
    int32_t w_off;              /* first weight column of the group */
    int32_t out_off, mul_out;   /* slice of the output features */
    int32_t c_off;              /* offset into the coefficient table (d1*d2*d_out floats) */
} ddp_tp_group_t;

typedef struct {
    /* edge MLP, fp32, input-major ("transposed") so that output columns are contiguous */
    const float *w1t;  /* [k1][hid] */
    const float *b1;   /* [hid] */
    const float *w2t;  /* [hid][w_numel] */
    const float *b2;   /* [w_numel] */
    int32_t k1, hid, w_numel;
    int32_t n_emb, ns;            /* k1 == n_emb + ns * (#node parts) */
    /* tensor product */
    const ddp_tp_group_t *groups; /* device array [n_groups] */
    const float *ctab;            /* device coefficient table [ctab_len] */
    int32_t ctab_len;
    const uint8_t *col_group;     /* device [w_numel]: group of each weight column */
    int32_t n_groups;
    int32_t f_in, f_out, sh_dim;
} ddp_tpconv_t;

typedef struct {
    const float *emb;             /* [cap][n_emb] */
    const float *p1; const int32_t *i1; int32_t ld1;  /* first node part (NULL to skip) */
    const float *p2; const int32_t *i2; int32_t ld2;  /* second node part (NULL to skip) */
    const float *x;  const int32_t *gather; int32_t ldx; /* node features gathered at edge_index[1] */
    const float *sh;              /* [cap][sh_dim] */
    const int32_t *agg;           /* edge_index[0] */
    const float *ew;              /* optional per-edge weight (smooth_edges) */
    const int32_t *n_edges_dev; int32_t edge_cap;
    /* optional pre-normalised accumulation: sum[agg][c] += out[c] * out_scale[c] / max(agg_deg[agg], 1), i.e. the
     * scatter-MEAN and the BatchNorm scale of this conv applied on the fly, so that several convs of a layer can
     * accumulate into ONE buffer (ddp_node_update then adds only their shifts).  Both NULL: plain sums.  Either may
     * be given alone (the host mirror folds the BatchNorm scale into the packed weights and passes only agg_deg). */
    const float *out_scale;       /* [f_out] */
    const int32_t *agg_deg;       /* [n_out] in-degree of the aggregation nodes for this edge set */
} ddp_tpconv_edges_t;

/* fp32 CUDA-core path: exact-arithmetic mode and fallback for irreps the tensor-core kernel does not
 * specialise (lmax = 2, torsion FCTP).  sum: [n_out][f_out], zeroed by the caller. */
int ddp_tpconv_fp32(const ddp_tpconv_t *conv, const ddp_tpconv_edges_t *edges, float *sum, void *stream);
/* Same convolution with deterministic accumulation (see DDP_ACC_FIXED_SHIFT): both the per-tile accumulation in shared
 * memory and the scatter-add into sum are fixed point.  sum: int64 [n_out][f_out], zeroed by the caller; status: the
 * sticky device status word. */
int ddp_tpconv_fp32_fixed(const ddp_tpconv_t *conv, const ddp_tpconv_edges_t *edges, int64_t *sum, uint32_t *status,
                          void *stream);

/* Tensor-core path (tcgen05 / TMEM, bf16 operands, fp32 accumulate), for FasterTensorProduct-shaped
 * convs (l <= 1 row groups, k1 == hid == 3*ns).  mode: 0 = bf16 single pass, 1 = bf16x3 split
 * (hi*hi + lo*hi + hi*lo: fp32-grade products).
 * ddp_tpconv_pack builds the weight image the kernel streams with TMA bulk copies: UMMA core-matrix order,
 * consumption order, biases folded into a constant-one K slot, path normalisation folded into the weights.
 * All its pointers are HOST pointers (groups_host / ctab_host mirror conv->groups / conv->ctab; w1 [hid][k1],
 * b1 [hid], w2 [w_numel][hid], b2 [w_numel] in nn.Linear layout).  packed_host == NULL returns the image size
 * in bytes; otherwise 0 on success; negative DDP_E_* (DDP_E_UNSUPPORTED: not tensor-core eligible). */
int64_t ddp_tpconv_pack(const ddp_tpconv_t *conv, const ddp_tp_group_t *groups_host, const float *ctab_host,
                        const float *w1_host, const float *b1_host, const float *w2_host, const float *b2_host,
                        int32_t mode, void *packed_host);
/* `packed` is the device copy of that image.  Requires p1 and p2 (three 'ns'-wide edge-attribute parts). */
int ddp_tpconv_umma(const ddp_tpconv_t *conv, const void *packed, int32_t mode,
                    const ddp_tpconv_edges_t *edges, float *sum, void *stream);

/* Grouped launch: n_jobs (<= 9) convolutions that share irreps (same f_in / f_out / weight layout, e.g. the nine
 * convs of one interaction layer, all_atom_score_model.py:274-312) run as ONE persistent kernel over the union of
 * their 128-edge tiles, so small edge sets do not leave SMs idle.  Arrays of n_jobs HOST pointers. */
int ddp_tpconv_umma_group(const ddp_tpconv_t *const *convs, const void *const *packed, int32_t mode,
                          const ddp_tpconv_edges_t *const *edges, float *const *sums, int32_t n_jobs, void *stream);
/* Deterministic accumulation (see DDP_ACC_FIXED_SHIFT): the same kernels, but every partial sum of the segmented
 * pre-reduction is converted to fixed point and added with a 64-bit integer reduction.  sums: int64 [n_out][f_out] each,
 * zeroed by the caller; status: the sticky device status word.  Same packed images, modes and restrictions. */
int ddp_tpconv_umma_fixed(const ddp_tpconv_t *conv, const void *packed, int32_t mode, const ddp_tpconv_edges_t *edges,
                          int64_t *sum, uint32_t *status, void *stream);
int ddp_tpconv_umma_group_fixed(const ddp_tpconv_t *const *convs, const void *const *packed, int32_t mode,
                                const ddp_tpconv_edges_t *const *edges, int64_t *const *sums, int32_t n_jobs, uint32_t *status,
                                void *stream);

/* Training path (SURVEY 8(f) row 3): backward of the tensor product of one TensorProductConvLayer.  Replaces what
 * autograd does for `self.tp(node_attr[edge_dst], edge_sh, self.fc(edge_attr))` under `loss.backward()`
 * (models/score_model.py:112-114, models/layers.py:40-85 / e3nn FullyConnectedTensorProduct; utils/training.py:147-191):
 *   g_w[e][col]            = sum_k basis_k(x, sh) g_out[e][out(col)][k]
 *   g_x[gather[e]][...]   += w[e][col] sum_{j,k} C[i][j][k] sh[e][j] g_out[e][...][k]      (atomic; may be NULL)
 *   g_sh[e][j]            += w[e][col] sum_{i,k} C[i][j][k] x[...][i] g_out[e][...][k]       (atomic; may be NULL)
 * w / g_w: [n_edges][w_numel] (the per-edge weights fc(edge_attr) and their gradient, materialised per chunk of
 * edges by the caller), g_out: [n_edges][f_out] per-EDGE output gradients (the caller has applied the scatter-mean:
 * g_sum[agg[e]] / deg).  The Linear / ReLU gradients around it are plain GEMMs on the caller's side
 * (diffdock_pocket_b200/score_model.py:_ConvFn).  Uses conv->groups, ctab, n_groups, w_numel, f_out, sh_dim; irrep
 * dimensions of the groups must be <= 5 (l <= 2). */
int ddp_tp_backward(const ddp_tpconv_t *conv, int32_t rows_per_edge /* sum of mul_in over conv->groups */, const float *x,
                    const int32_t *gather, int32_t ldx, const float *sh, const float *w, const float *g_out, int32_t n_edges,
                    float *g_w, float *g_x, float *g_sh, void *stream);
/* Same, with g_x / g_sh accumulated deterministically in fixed point (see DDP_ACC_FIXED_SHIFT): int64 buffers of the same
 * shapes, zeroed by the caller (they may collect several chunks of edges) and converted once with ddp_fixed_to_float;
 * status: the sticky device status word.  g_w is written directly, as above. */
int ddp_tp_backward_fixed(const ddp_tpconv_t *conv, int32_t rows_per_edge, const float *x, const int32_t *gather, int32_t ldx,
                          const float *sh, const float *w, const float *g_out, int32_t n_edges, float *g_w, int64_t *g_x,
                          int64_t *g_sh, uint32_t *status, void *stream);

/* Developer aid: when trace_dev != NULL, CTA 0 of every following tensor-core conv launch records clock64()
 * timestamps of its MMA-issue and epilogue roles per weight tile into trace_dev (device int64 buffer); NULL turns
 * it off.  Returns the number of int64 slots the buffer must hold, or DDP_E_UNSUPPORTED when the library was built
 * without -DDDP_UMMA_TRACE (the default: the hooks cost epilogue instructions).  Not part of the reference surface. */
int ddp_tpconv_umma_set_trace(void *trace_dev);

/* node update (all_atom_score_model.py:315-324 + scatter-mean + e3nn BatchNorm eval, score_model.py:117,123):
 *   new[n][c] = (c < f_old ? old[n][c] : 0) + sum_u live_u * (sum_u[n][c] / max(deg_u[n],1) * scale_u[c] + shift_u[c])
 * live_u = (*n_edges_u > 0) reproduces `return 0` for an empty edge set (score_model.py:109-111).
 * old may be NULL (heads).  deg == NULL: sum is already normalised (see ddp_tpconv_edges_t.out_scale / agg_deg; scale
 * is then ignored); sum == NULL: the update contributes only its shift. */
typedef struct {
    const float *sum; const int32_t *deg; const float *scale; const float *shift; const int32_t *n_edges_dev;
} ddp_update_t;
int ddp_node_update(const float *old_x, int32_t f_old, int32_t ld_old, const ddp_update_t *updates, int32_t n_updates,
                    int32_t n, int32_t f_new, float *new_x, int32_t ld_new, void *stream);
/* The node updates of one interaction layer (ligand, atom, receptor) in one launch; widths / strides even and
 * bases 8-byte aligned (the resident plan's buffers). */
typedef struct {
    const float *old_x; int32_t f_old, ld_old;
    ddp_update_t updates[4]; int32_t n_updates;
    int32_t n, f_new; float *new_x; int32_t ld_new;
} ddp_node_update_job_t;
int ddp_node_update_multi(const ddp_node_update_job_t *jobs_host, int32_t n_jobs, void *stream);
/* The same two updates for sums accumulated in fixed point by the *_fixed convolutions: every non-NULL
 * ddp_update_t.sum points at int64 [n][f_new] (cast to const float * in the struct), converted with 2^-DDP_ACC_FIXED_SHIFT
 * before the divide-by-degree, scale and shift above.  Everything else is unchanged. */
int ddp_node_update_fixed(const float *old_x, int32_t f_old, int32_t ld_old, const ddp_update_t *updates, int32_t n_updates,
                          int32_t n, int32_t f_new, float *new_x, int32_t ld_new, void *stream);
int ddp_node_update_multi_fixed(const ddp_node_update_job_t *jobs_host, int32_t n_jobs, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Heads (all_atom_score_model.py:329-434). */

/* out[g][c] = mean over i in [ptr[g], ptr[g+1]) of src[idx ? idx[i] : i][c] (0 for an empty segment):
 * ligand centroid (build_center_conv_graph, :590-592) and the confidence pooling (:331,339). */
int ddp_segment_mean(const float *src, const int32_t *idx, const int32_t *ptr, int32_t n_seg, int32_t width,
                     int32_t ld, float *out, int32_t ld_out, void *stream);

/* bond geometry: mid = (pos[b0]+pos[b1])/2, y2 = Y_2(pos[b1]-pos[b0]) (component normalised, e3nn
 * basis), attr = x[b0] + x[b1] (first ns columns)  (:391-394, :604, :415-418, :624). */
int ddp_bond_geometry(const float *pos, const int32_t *bonds, int32_t n_bonds, const float *x, int32_t ldx, int32_t ns,
                      float *mid, float *y2, float *attr, void *stream);

/* sh_tor[e] = [1, 1o component of FullTensorProduct(sh_edge (1x0e+1x1o), Y2[bond])]  (:395, :419); the leading 1
 * pads the row to the [s0 | s1] layout of the conv kernels (4 floats per edge). */
int ddp_tor_edge_sh(const float *sh, int32_t sh_dim, const float *y2, const float *c121 /* [3][5][3], sqrt(3) folded */,
                    const int32_t *edge, const int32_t *n_edges_dev, int32_t edge_cap, float *sh_tor, void *stream);

/* General form for sh_lmax = 2 (all_atom_score_model.py:193,219,395,419): the l <= 1 output irreps of
 * FullTensorProduct(sh_edge, Y2[bond]) that the torsion convolutions can couple to (0e from 2e x 2e, 1o from 1o x 2e,
 * 1e from 2e x 2e), written contiguously to out [cap][out_dim].  Path q:
 *   out[e][out_off + k] = sum_{i < d_in, j < 5} ctab[c_off + (i * 5 + j) * d_out + k] * sh[e][in_off + i] * y2[bond][j]
 * with ctab = sqrt(2 l_out + 1) * wigner_3j(l_in, 2, l_out) (e3nn FullTensorProduct, component normalisation). */
typedef struct { int32_t in_off, d_in, out_off, d_out, c_off; } ddp_ftp_path_t;
int ddp_tor_edge_sh_generic(const float *sh, int32_t sh_dim, const float *y2, const ddp_ftp_path_t *paths_host, int32_t n_paths,
                            const float *ctab, const int32_t *edge, const int32_t *n_edges_dev, int32_t edge_cap, float *out,
                            int32_t out_dim, void *stream);

/* row MLP (tor_final_layer / sc_tor_final_layer :402,427; confidence_predictor :344 with BatchNorm1d folded):
 * x <- act_l(W_l x + b_l) for up to 4 layers (W input-major [n_in][n_out], b may be NULL; act 0 none,
 * 1 relu, 2 tanh), then out[row][:] = x * (row_scale ? row_scale[row] : 1).  Widths <= 256. */
typedef struct { const float *wt; const float *b; int32_t n_in, n_out, act; } ddp_mlp_layer_t;
int ddp_row_mlp(const float *in, int32_t n, int32_t ld_in, const ddp_mlp_layer_t *layers_host, int32_t n_layers,
                const float *row_scale, float *out, int32_t ld_out, void *stream);

/* tr / rot magnitude heads (:365-384): g [B][12] conv output, sig [B][sig_dim];
 * out_tr = v_tr/|v_tr| * mlp_tr([|v_tr| | sig]) / tr_sigma;  out_rot likewise * so3_norm. */
int ddp_tr_rot_head(const float *g, const float *sig, int32_t sig_dim, int32_t n_graphs, const float *tr_w1t,
                    const float *tr_b1, const float *tr_w2, const float *tr_b2, const float *rot_w1t, const float *rot_b1,
                    const float *rot_w2, const float *rot_b2, int32_t hid, const float *tr_sigma, const float *so3_norm,
                    float *tr_out, float *rot_out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Pose update: one launch per reverse-diffusion step (utils/sampling.py:129-251 +
 * utils/diffusion_utils.py:37-70 + utils/torsion.py:68-94,251-278 + utils/geometry.py:39-86,209-243).
 * Per sample s:  perturb = a * score + b * z  for tr, rot, tor, sc_tor (a, b host scalars of the step);
 * side-chain bonds are rotated in order, then the ligand is moved rigidly, its torsions are applied in
 * order and the flexed conformer is Kabsch-aligned back onto the rigid pose. */
typedef struct {
    float a_tr, b_tr, a_rot, b_rot, a_tor, b_tor, a_sc, b_sc;
} ddp_step_coef_t;
typedef struct {
    int32_t n_samples;
    /* ligand */
    float *lig_pos; const int32_t *lig_ptr;              /* [NL][3], [n_samples+1] */
    const int32_t *tor_ptr;                              /* [n_samples+1] into tor arrays */
    const int32_t *tor_bonds;                            /* [T][2] global atom indices (u, v) */
    const uint8_t *mask_rotate; const int32_t *mask_ptr; /* row t: atoms of its sample, bytes; mask_ptr[T+1] */
    /* side chains */
    float *atom_pos;                                     /* [NA][3] */
    const int32_t *sc_ptr;                               /* [n_samples+1] into sc arrays */
    const int32_t *sc_bonds;                             /* [S][2] global atom indices (u, v) */
    const int32_t *sc_sub_ptr; const int32_t *sc_sub;    /* [S+1], global atom indices of each subcomponent */
    /* scores and noise */
    const float *tr_score, *rot_score, *tor_score, *sc_score;
    const float *tr_z, *rot_z, *tor_z, *sc_z;
} ddp_pose_t;
int ddp_pose_update(const ddp_pose_t *pose, const ddp_step_coef_t *coef, void *stream);
/* Largest ligand (atoms of one sample) the fused kernel handles: its flexible / rigid copies live in shared memory.
 * The caller must check its per-sample atom counts against this (the kernel traps on a larger ligand instead of
 * leaving it unmoved). */
int ddp_pose_max_ligand_atoms(void);
/* Same, with the step coefficients read from DEVICE memory (8 floats): lets the whole step be replayed as a
 * CUDA graph while the per-step scalars change. */
int ddp_pose_update_dev(const ddp_pose_t *pose, const ddp_step_coef_t *coef_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif
