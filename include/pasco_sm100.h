/* pasco_sm100.h — C ABI of libpasco_sm100.so, the sm_100a sparse-voxel engine that sits
 * underneath PaSCo's operator surface.
 *
 * Every entry point replaces one granule of the MinkowskiEngine 0.5.4 pybind backend
 * (`MinkowskiEngineBackend._C`, not vendored in /root/reference) that the reference reaches
 * through `import MinkowskiEngine as ME`; the reference call site each one serves is cited
 * as pasco/<file>:<line> (paths relative to /root/reference).
 *
 * Conventions
 *   - plain C types, raw DEVICE pointers, caller-owned memory (the library never allocates);
 *   - every call takes the CUDA stream to launch on (pass torch's current stream);
 *   - returns 0 on success, negative on error; pasco_last_error() gives the message of the
 *     last failure on the calling thread;
 *   - coordinates are int32 rows (b, x, y, z), each component in [-32768, 32767];
 *   - features are row-major float32 [N, C]; row indices are int32, −1 == "no row";
 *   - a neighbour table `nbr` is int32 [K, N_out]: nbr[k*N_out + o] = input row feeding
 *     output row o through kernel offset k, or −1.  Offsets enumerate x fastest; odd kernel
 *     sizes are centred, even ones span [0, k)·stride  (ME convention, SURVEY.md §8b).
 */
#ifndef PASCO_SM100_H_
#define PASCO_SM100_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* pasco_stream_t; /* cudaStream_t */

const char* pasco_last_error(void);
int pasco_abi_version(void);
/* fills sm count / smem per block opt-in / compute capability major*10+minor of the current device */
int pasco_device_info(int* sm_count, int* smem_optin, int* cc);

/* ---- coordinate maps (ME CoordinateMapManager::insert_and_map / stride / kernel_map) ----
 * Hash table = open addressing over `capacity` (power of two ≥ 2N) slots:
 *   table_keys  uint64[capacity]  (caller fills with 0xFF bytes before the first insert)
 *   table_vals  int32 [capacity]  (caller fills with 0x7F bytes)                            */

/* ME.SparseTensor(F, C) — pasco/models/net_panoptic_sparse.py:323, unet3d_sparse_v2.py:207.
 * Inserts n rows; on return table_vals[slot(key)] = smallest row index holding that key and
 * first_row[i] = that winning row for input row i (first_row[i]==i ⇔ row i is kept).
 * Keys pack 16 bits per component: a coordinate or batch index outside [-32768, 32767] sets *err_flag = 2 on the
 * device (err_flag may be NULL) and the host wrapper raises; MinkowskiEngine accepts the full int32 range.          */
int pasco_hash_insert(const int32_t* coords, int64_t n, uint64_t* table_keys, int32_t* table_vals,
                      int64_t capacity, int32_t* first_row, int32_t* err_flag, pasco_stream_t s);

/* After compaction: rewrite table values old_row → new_row[old_row] (new_row[i] = −1 for dropped rows). */
int pasco_hash_remap(int32_t* table_vals, int64_t capacity, const int32_t* new_row, pasco_stream_t s);

/* row of each query coordinate (−1 if absent) — union map (decoder_v3.py:163) and tests */
int pasco_hash_lookup(const int32_t* query, int64_t nq, const uint64_t* table_keys, const int32_t* table_vals,
                      int64_t capacity, int32_t* out_row, pasco_stream_t s);

/* out[i] = (b, floor(x/s)*s, ...) — ME stride map for k=2,s=2 convs (pasco/maskpls/mink.py:509-511)
 * and max-pool (transformer_predictor_v2.py:100-102).  Floors toward −inf.                     */
int pasco_coords_floor(const int32_t* coords, int64_t n, int32_t sx, int32_t sy, int32_t sz, int32_t* out,
                       pasco_stream_t s);

/* generative transposed conv output coordinates (mink.py:524-527): child row 8*p + k =
 * parent p + offset_k * out_stride, offsets x fastest in {0,1}^3; kernel_size fixed to 2.     */
int pasco_coords_generate_k2(const int32_t* coords, int64_t n, int32_t out_sx, int32_t out_sy, int32_t out_sz,
                             int32_t* out, pasco_stream_t s);

/* nbr[k, o] for an odd kernel (k=3) between an input map (hash table) and output coords:
 * probes out + offset_k*dilation*stride  (every ME.MinkowskiConvolution k=3: mink.py:625-638,
 * decoder_v3.py:267-282).                                                                      */
int pasco_kernel_map_probe(const int32_t* out_coords, int64_t n_out, const uint64_t* table_keys,
                           const int32_t* table_vals, int64_t capacity, int32_t kernel_size, int32_t sx,
                           int32_t sy, int32_t sz, int32_t* nbr, pasco_stream_t s);

/* same for an anisotropic odd box kernel (kx,ky,kz), K = kx*ky*kz offsets x fastest — the dense bottleneck
 * kernels (3,3,1), (5,5,3), (7,7,5) of pasco/models/layers.py:656-702 run as sparse convs over the full
 * stride-8 grid.                                                                                  */
int pasco_kernel_map_box(const int32_t* out_coords, int64_t n_out, const uint64_t* table_keys,
                         const int32_t* table_vals, int64_t capacity, int32_t kx, int32_t ky, int32_t kz,
                         int32_t sx, int32_t sy, int32_t sz, int32_t* nbr, pasco_stream_t s);

/* even kernel == stride (k=2 s=2 conv, k=s max-pool): every child has one parent.
 *   parent_of[i] = row of floor(child_i) in the parent table
 *   slot_of[i]   = kernel offset index of the child inside its parent block (x fastest)
 *   nbr[k, p]    = child row (written when nbr != NULL; K = ks^3 rows of n_parent)              */
int pasco_kernel_map_down(const int32_t* child_coords, int64_t n_child, const uint64_t* table_keys,
                          const int32_t* table_vals, int64_t capacity, int32_t ks, int32_t child_sx,
                          int32_t child_sy, int32_t child_sz, int32_t* parent_of, int32_t* slot_of, int32_t* nbr,
                          int64_t n_parent, pasco_stream_t s);

/* ---- row compaction (ME.MinkowskiPruning: decoder_v3.py:159,421,496; misc.py:17-26) ----------
 * step 1: block_counts[b] = popcount of mask over rows [b*1024, (b+1)*1024)
 * (caller turns counts into exclusive offsets — a length-ceil(n/1024) scan)
 * step 2: new_row[i] = compacted index or −1, kept_rows[new] = i (order preserving)             */
int pasco_mask_block_counts(const uint8_t* mask, int64_t n, int32_t* block_counts, pasco_stream_t s);
int pasco_mask_compact(const uint8_t* mask, int64_t n, const int32_t* block_offsets, int32_t* new_row,
                       int32_t* kept_rows, pasco_stream_t s);

/* out[r, :] = rows[r] >= 0 ? src[rows[r], :] : 0   (row gather; also the backward of scatter) */
int pasco_gather_rows(const float* src, const int32_t* rows, int64_t n_rows, int32_t C, float* out,
                      pasco_stream_t s);
/* dst[rows[r], :] (+)= src[r, :]; rows unique, −1 skipped (union add, decoder_v3.py:163) */
int pasco_scatter_rows(const float* src, const int32_t* rows, int64_t n_rows, int32_t C, float* dst,
                       int32_t accumulate, pasco_stream_t s);
/* same for int32 [N,4] coordinate rows */
int pasco_gather_coords(const int32_t* src, const int32_t* rows, int64_t n_rows, int32_t* out, pasco_stream_t s);

/* ---- dense <-> sparse (SparseTensor.dense / ME.to_sparse: augmenter.py:15-22,
 *      unet3d_sparse_v2.py:196-202, transformer_predictor_v2.py:263-274) ----------------------
 * dense is [B, C, X, Y, Z] float32; cell = (coord - min) / stride.  A row whose cell lies outside the volume is
 * skipped (to_dense) / reads as zero (from_dense) and sets *err_flag = 1 on the device (err_flag may be NULL); the
 * host wrapper raises at its next synchronisation point, where MinkowskiEngine raises immediately.              */
int pasco_to_dense(const float* feats, const int32_t* coords, int64_t n, int32_t C, const int32_t min_c[3],
                   const int32_t stride[3], float* dense, int32_t B, int32_t X, int32_t Y, int32_t Z,
                   int32_t* err_flag, pasco_stream_t s);
int pasco_from_dense(const float* dense, const int32_t* coords, int64_t n, int32_t C, const int32_t min_c[3],
                     const int32_t stride[3], float* feats, int32_t B, int32_t X, int32_t Y, int32_t Z,
                     int32_t* err_flag, pasco_stream_t s);
/* occupancy[b,x,y,z] = (sum_c |dense[b,c,x,y,z]|) != 0  → uint8 mask in (b,x,y,z) order */
int pasco_dense_occupancy(const float* dense, int32_t B, int32_t C, int64_t cells, uint8_t* mask,
                          pasco_stream_t s);

/* ---- sparse convolution (ME ConvolutionForward/Backward: every conv on the path) -------------
 * out[o,:] = sum_k in[nbr[k,o],:] @ W[k]        W: float32 [K, Cin, Cout]
 *
 * Tensor-core path (tcgen05, bf16 split operands, fp32 accumulate in TMEM):
 *   precision 1 = bf16 operands (1 MMA / k-step), 3 = bf16x3 split (hi·hi + lo·hi + hi·lo,
 *   ~2^-16 relative: the "fp32" mode of BASELINE.json configs[1]).
 *   Requires Cin % 64 == 0, Cout % 16 == 0, 16 <= Cout <= 256.
 * Weights are first packed into the UMMA shared-memory image:
 *   transpose=0: B[n=co][k=ci] = W[k][ci][co]      (forward)
 *   transpose=1: B[n=ci][k=co] = W[k][ci][co]      (input gradient; swap Cin/Cout in the conv call)
 * packed size in bytes = pasco_conv_packed_bytes(K, Cin, Cout).                                 */
int64_t pasco_conv_packed_bytes(int32_t K, int32_t Cin, int32_t Cout);
int pasco_conv_pack_weights(const float* W, int32_t K, int32_t Cin, int32_t Cout, int32_t transpose, void* packed,
                            pasco_stream_t s);
/* koff_map (host int32[K] or NULL): packed weight slice used for table row k; must be the identity
 * (NULL) or the reversal K-1-k (mirrored offsets of the input gradient).  K <= 1024.
 * bias: float32[Cout] or NULL.  in_scale/in_shift: optional per-input-channel affine applied
 * in the gather prologue (fused BatchNorm), in_act: 0 none, 1 ReLU, 2 LeakyReLU(0.01) after it.
 * stats: optional float64[2*Cout] accumulating column sum / sum of squares of the output.
 * in_pitch / out_pitch: row strides in floats (0 = Cin / Cout) so that a column block of a wider matrix can be
 * read / written in place — dense Linear layers run as K = 1, nbr = NULL convolutions in column chunks <= 256.  */
int pasco_conv_forward_tc(const float* in, int64_t n_in, const int32_t* nbr, int32_t K, int64_t n_out,
                          int32_t Cin, int32_t Cout, const void* packed_w, const int32_t* koff_map,
                          const float* bias, const float* in_scale, const float* in_shift, int32_t in_act,
                          double* stats, float* out, int32_t precision, int64_t in_pitch, int64_t out_pitch,
                          pasco_stream_t s);
/* Split-K form of the same convolution for shapes with few output tiles and many offsets (the dense bottleneck of
 * layers.py:646-726 runs as 32 tiles x 245 offsets: one CTA per tile would leave 116 of 148 SMs idle).  The offsets are
 * cut into ranges, every (tile, range) pair is a work item whose partial result goes to the caller's workspace, and a
 * second kernel adds the partials in a fixed order (+ bias) — still deterministic, no atomics.
 * pasco_conv_splitk_workspace_bytes returns 0 when the shape is not worth splitting (then call pasco_conv_forward_tc). */
int64_t pasco_conv_splitk_workspace_bytes(int32_t K, int64_t n_out, int32_t Cout);
int pasco_conv_forward_splitk(const float* in, int64_t n_in, const int32_t* nbr, int32_t K, int64_t n_out, int32_t Cin,
                              int32_t Cout, const void* packed_w, const int32_t* koff_map, const float* bias,
                              const float* in_scale, const float* in_shift, int32_t in_act, float* out, int32_t precision,
                              int64_t in_pitch, int64_t out_pitch, void* workspace, int64_t workspace_bytes,
                              pasco_stream_t s);

/* Plane-gather path (the default for every gathered convolution): the activations are split ONCE per tensor into bf16
 * planes x = hi + lo (lo = NULL for precision 1) by pasco_split_planes — optionally fused with y = act(x*scale + shift),
 * the BatchNorm + activation of the producing layer — and the convolution / weight-gradient producers move plane rows
 * with 16-byte cp.async copies straight into the swizzled UMMA tiles (missing neighbours are zero-fill copies that touch
 * no memory).  Planes are bf16 [N, C] with a row pitch in ELEMENTS (0 = C); C % 8 == 0.
 * pasco_conv_forward_planes: forward and input gradient (same contract as pasco_conv_forward_tc: koff_map, bias, fused
 * BatchNorm statistics of `out` in `stats`);  pasco_conv_wgrad_planes: dW (zeroed by the caller) from the planes of the
 * layer input and of the output gradient.                                                                          */
int pasco_split_planes(const float* x, int64_t n, int32_t C, int64_t pitch, const float* scale, const float* shift,
                       int32_t act, void* hi, void* lo, pasco_stream_t s);
int pasco_conv_forward_planes(const void* hi, const void* lo, int64_t n_in, const int32_t* nbr, int32_t K, int64_t n_out,
                              int32_t Cin, int32_t Cout, const void* packed_w, const int32_t* koff_map, const float* bias,
                              double* stats, float* out, int32_t precision, int64_t plane_pitch, int64_t out_pitch,
                              pasco_stream_t s);
int pasco_conv_wgrad_planes(const void* in_hi, const void* in_lo, int64_t n_in, const int32_t* nbr, int32_t K,
                            int64_t n_out, int32_t Cin, int32_t Cout, const void* g_hi, const void* g_lo, float* dW,
                            int32_t precision, int64_t in_pitch, int64_t gout_pitch, float* workspace,
                            int64_t workspace_bytes, pasco_stream_t s);

/* dW[k] = sum_o in[nbr[k,o],:]^T @ gout[o,:]   (tcgen05, MN-major operands); dW float32 [K,Cin,Cout] zeroed by caller.
 * Both weight-gradient kernels store each CTA's partial dW in `workspace` (pasco_conv_wgrad_workspace_bytes) and add the
 * partials in a fixed order, so dW is the same from run to run.                                                       */
int64_t pasco_conv_wgrad_workspace_bytes(int32_t K, int64_t n_out, int32_t Cin, int32_t Cout);
int pasco_conv_wgrad_tc(const float* in, int64_t n_in, const int32_t* nbr, int32_t K, int64_t n_out, int32_t Cin,
                        int32_t Cout, const float* gout, const float* in_scale, const float* in_shift,
                        int32_t in_act, float* dW, int32_t precision, int64_t in_pitch, int64_t gout_pitch,
                        float* workspace, int64_t workspace_bytes, pasco_stream_t s);

/* CUDA-core fp32 reference path of the same contraction (any Cin/Cout; validation + odd shapes) */
int pasco_conv_forward_simt(const float* in, const int32_t* nbr, int32_t K, int64_t n_out, int32_t Cin,
                            int32_t Cout, const float* W, int32_t w_transposed, const int32_t* koff_map,
                            const float* bias, float* out, pasco_stream_t s);
int64_t pasco_conv_wgrad_simt_workspace_bytes(int32_t K, int64_t n_out, int32_t Cin, int32_t Cout);
int pasco_conv_wgrad_simt(const float* in, const int32_t* nbr, int32_t K, int64_t n_out, int32_t Cin, int32_t Cout,
                          const float* gout, float* dW, float* workspace, int64_t workspace_bytes, pasco_stream_t s);

/* ---- pooling / reductions --------------------------------------------------------------------
 * ME.MinkowskiMaxPooling(k=s, stride=s) (transformer_predictor_v2.py:100-102): out rows
 * pre-filled with -inf by the caller; out[parent_of[i], c] = max(...)                            */
int pasco_maxpool_forward(const float* in, const int32_t* parent_of, int64_t n_in, int32_t C, float* out,
                          pasco_stream_t s);
/* torch_scatter.scatter_max(src, index, dim=0) (unet3d_sparse_v2.py:79): out pre-filled with -inf,
 * second pass writes argmax (smallest row attaining the max) and zero-fills empty segments        */
int pasco_scatter_max(const float* src, const int64_t* index, int64_t n, int32_t C, float* out, int64_t n_seg,
                      int64_t* argmax, pasco_stream_t s);

/* ---- BatchNorm over rows (ME.MinkowskiBatchNorm == BatchNorm1d on [N,C]; mink.py:512,623,631) ---
 * stats float64[2*C] (sum, sumsq) zeroed by the caller; apply: y = act(x*scale[c] + shift[c])      */
int pasco_bn_stats(const float* x, int64_t n, int32_t C, double* stats, pasco_stream_t s);
int pasco_affine_act(const float* x, int64_t n, int32_t C, const float* scale, const float* shift, int32_t act,
                     const float* residual, float* y, pasco_stream_t s);
/* per-channel coefficients in one launch each: stats -> scale/shift (+ mean, rstd, running-statistics update);
 * backward sums -> (ca, cb, cc) of dx = ca*dz + cb*x + cc and the gamma/beta gradients (divided by grad_div).
 * count_dev (device double, e.g. the all-reduced SyncBatchNorm row count) overrides `count` when not NULL.       */
int pasco_bn_finalize(const double* stats, const double* count_dev, double count, int32_t C, const float* gamma,
                      const float* beta, float eps, float momentum, float* scale, float* shift, float* mean, float* rstd,
                      float* running_mean, float* running_var, pasco_stream_t s);
int pasco_bn_bwd_coefs(const double* sums, const double* count_dev, double count, int32_t C, const float* gamma,
                       const float* mean, const float* rstd, float grad_div, float* ca, float* cb, float* cc, float* ggamma,
                       float* gbeta, pasco_stream_t s);
/* backward: given dy, x (pre-BN), scale/shift/act → sums float64[2*C] = (Σ dz, Σ dz·x̂·…) and dx */
int pasco_bn_bwd_reduce(const float* dy, const float* x, int64_t n, int32_t C, const float* scale,
                        const float* shift, int32_t act, double* sums, pasco_stream_t s);
int pasco_bn_bwd_apply(const float* dy, const float* x, int64_t n, int32_t C, const float* scale,
                       const float* shift, int32_t act, const float* coef_a, const float* coef_b,
                       const float* coef_c, float* dx, pasco_stream_t s);

/* ---- MaskPLS masked cross-attention (pasco/models/transformer/blocks.py:73-92 with the attention mask of
 *      transformer_predictor_v2.py:220-289): Q <= 128 queries against all P voxels, H heads of width D <= 64 ------
 * q [Q, H*D], k / v [P, H*D] float32 (already projected); logits = scale * q.k; mask = bit rows
 * uint32 [Q, 2*ceil(P/64)] (bit j of word 2t + j/32 set = key 64t + j masked) or NULL; out [Q, H*D] ZEROED by the
 * caller; lse [H, Q] receives log-sum-exp per row (needed by the backward).  Two streaming passes over K (row
 * statistics, then output), tcgen05 for both GEMMs, bf16x3 split operands.                                        */
int64_t pasco_xattn_workspace_bytes(int32_t Q, int64_t P, int32_t H, int32_t D);
int pasco_xattn_forward(const float* q, const float* k, const float* v, const uint32_t* mask, int32_t Q, int64_t P,
                        int32_t H, int32_t D, float scale, float* out, float* lse, float* workspace,
                        int64_t workspace_bytes, pasco_stream_t s);
/* backward of the above: recomputes the probabilities from lse; dq [Q, H*D] ZEROED by the caller (the key chunks'
 * partial dq go to `workspace`, sized by pasco_xattn_workspace_bytes, and are added in chunk order), dk / dv [P, H*D]
 * are fully overwritten (every row written exactly once, no atomics).                                            */
int pasco_xattn_backward(const float* q, const float* k, const float* v, const uint32_t* mask, const float* lse,
                         const float* out, const float* dout, int32_t Q, int64_t P, int32_t H, int32_t D, float scale,
                         float* dq, float* dk, float* dv, float* workspace, int64_t workspace_bytes, pasco_stream_t s);

/* ---- evaluation (pasco/models/metrics.py SSCMetrics + UncertaintyMetrics, pasco/loss/panoptic_quality.py) ---------
 * Calibration binning is torchmetrics' binary_calibration_error: bounds = torch.linspace(0, 1, n_bins + 1) in fp32,
 * slot = bucketize(conf, bounds, right=True) - 1 over n_bins + 1 slots (NB below).  Integer outputs are ACCUMULATED
 * (+=, the caller zeroes them once); fp64 sums are accumulated too and are the same from run to run.  A label >= K
 * (other than 255 = unknown) or a segment id outside its table sets *err_flag = 3 and the cell or row is skipped.
 *
 * One sweep over a scene's cells: prob float [K, cells] (class-major, empty cells one-hot class 0), label uint8 [cells].
 * Per cell: pred = argmax (first maximum), conf = max prob.
 * Everything is over known cells (SSCMetrics.add_batch zeroes unknown cells, then masks them out).
 *   counts int64 [K*K + 4*NB]: confusion[target][pred] (SSCMetrics.add_batch), then split by pred == 0 / pred != 0:
 *     calibration counts [2][NB], correct (pred == label) counts [2][NB];
 *   sums double [2*NB + 2]: Σ conf [2][NB], Σ -log(p[label] + 1e-12) [2] (add_batch_ece).                           */
int64_t pasco_eval_ssc_workspace_bytes(int64_t cells, int32_t n_bins);
int pasco_eval_ssc(const float* prob, const uint8_t* label, int64_t cells, int32_t K, const float* bounds,
                   int32_t n_bins, int64_t* counts, double* sums, double* workspace, int64_t workspace_bytes,
                   int32_t* err_flag, pasco_stream_t s);
/* Intersection table of GT panoptic ids (gt_id int32 [cells], 0..n_gt) and predicted ids (pred_id int32 [n_rows],
 * 0..n_pred, at cell row_cell[r]; cells without a row are id 0) over known cells: table int64 [(n_gt+1) * (n_pred+1)].
 * Column sums are the predicted areas, row sums the GT areas, both after unknown cells are zeroed.                  */
int pasco_eval_pairs(const int32_t* pred_id, const int64_t* row_cell, int64_t n_rows, const int32_t* gt_id,
                     const uint8_t* label, int64_t cells, int32_t n_gt, int32_t n_pred, int64_t* table, int32_t* err_flag,
                     pasco_stream_t s);
/* Binned calibration of per-row mask confidences (UncertaintyMetrics.compute_ece_panop): rows whose cell is known with
 * gt_id != 0 and conf != 0; correct when match[pred_id] (int32 [n_pred+1], the GT id matched to each predicted
 * segment, 0 = none) == gt_id.  counts int64 [2*NB] (count, correct), sums double [NB] (Σ conf).                     */
int64_t pasco_eval_calib_workspace_bytes(int64_t n_rows, int32_t n_bins);
int pasco_eval_calib(const float* conf, const int32_t* pred_id, const int64_t* row_cell, int64_t n_rows,
                     const int32_t* gt_id, const uint8_t* label, int64_t cells, const int32_t* match, int32_t n_pred,
                     const float* bounds, int32_t n_bins, int64_t* counts, double* sums, double* workspace,
                     int64_t workspace_bytes, int32_t* err_flag, pasco_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* PASCO_SM100_H_ */
