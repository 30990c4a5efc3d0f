/*
 * b200pose.h - C ABI of libb200pose.so: the B200 (sm_100a) kernels of the per-frame inference hot
 * path of gnns4hri/3D_multi_pose_estimator.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; the caller allocates all
 *     outputs (the Python host layer does so through torch); no ownership is transferred;
 *   - every entry point enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 *     without synchronising; it is re-entrant per stream and keeps no global mutable state;
 *   - return value: 0 = ok, negative = error (B200POSE_E_*); b200pose_last_error() returns a
 *     thread-local message. Nothing aborts the process: the reference's callers wrap the model call
 *     in `try/except: continue` (test/metrics_from_model.py:200-213) and the Python layer raises.
 *   - "planes": an fp32 matrix X stored as two bf16 matrices hi = bf16(X), lo = bf16(X - hi) with a
 *     common leading dimension (multiple of 64 elements). All tensor-core GEMMs consume and produce
 *     planes and compute hi*hi + lo*hi + hi*lo with fp32 accumulation (3-term split-bf16).
 *
 * Each entry point cites the reference interface it replaces (paths relative to the reference root).
 */
#ifndef B200POSE_H
#define B200POSE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200POSE_OK             0
#define B200POSE_E_INVALID     -1   /* bad argument (shape, alignment, null pointer) */
#define B200POSE_E_CUDA        -2   /* a CUDA runtime / driver call failed */
#define B200POSE_E_UNSUPPORTED -3   /* configuration outside the compiled limits */

#define B200POSE_N_JOINTS        18  /* COCO-18, parameters.py:8 */
#define B200POSE_MAX_CAMERAS     32  /* camera sets are 32-bit masks in the clustering kernel */

const char* b200pose_last_error(void);
int b200pose_version(void);
/* compute capability of the current device as major*10+minor (100 on B200); <0 on error */
int b200pose_device_cc(void);

/* ---------------------------------------------------------------------------------------------
 * Camera tables (replaces the module-import globals of skeleton_matching/graph_generator.py:32-52
 * and utils/pose_estimator_dataset_from_json.py:28-47). C = number of cameras (parameters.camera_names
 * order). The struct itself lives on the HOST (it is read when a call is made); its array members are
 * DEVICE pointers to small tables uploaded once per configuration.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_cameras;                 /* C */
    int32_t v_sm;                      /* len(used_cameras_skeleton_matching) */
    int32_t v_pe;                      /* len(used_cameras) */
    float   image_width, image_height;
    const int32_t* sm_slot;            /* [C] camera -> index in used_cameras_skeleton_matching or -1 */
    const int32_t* pe_slot;            /* [C] camera -> index in used_cameras or -1 */
    const float*   kinv32;             /* [C,3,3] torch.inverse(K_fp32) the head features of camera c read (graph_generator.py:50, see below) */
    const float*   t_cam2root32;       /* [C,4,4] fp32(inv(T_root->cam)) of camera c    (dataset.py:38-41, indexed by camera_names.index) */
    const double*  k64;                /* [C,4]   fx,fy,cx,cy of fp64(K_fp32)    (dataset.py:43) */
    const double*  dist64;             /* [C,5]   k1,k2,p1,p2,k3                 (dataset.py:45) */
    const double*  p64;                /* [C,3,4] T_root->cam[0:3,:]             (dataset.py:47) */
    /* [C,4,4] the camera->root table HumanGraphFromView reads for camera c. graph_generator.py:38-52 appends its tables
     * walking camera_names (keeping the cameras in used_cameras_skeleton_matching) but :232-233 indexes them with
     * used_cameras_skeleton_matching.index(camera): slot s holds the s-th used camera IN RIG ORDER. Equal to
     * t_cam2root32 whenever the used list is in rig order (every shipped configuration); kinv32 follows the same rule. */
    const float*   t_cam2root32_sm;
} b200pose_cameras;

/* ---------------------------------------------------------------------------------------------
 * Packed skeleton batch (replaces the JSON strings the reference re-parses per frame,
 * graph_generator.py:587-588). S skeletons ("heads") of B frames, in head order: frame-dict camera
 * order, then skeleton order, skeletons without joints dropped (graph_generator.py:583-601).
 *   sk_xy   [S,18,2] fp64  pixel x,y exactly as the JSON carried them
 *   sk_vp   [S,18,2] fp32  valid, prob
 *   sk_mask [S]      u32   bit j set <=> joint key j present in the skeleton dict
 *   sk_cam  [S]      i32   camera index (parameters.camera_names order)
 *   head_off[B+1]    i32   first head of each frame
 *   node_off[B+1]    i32   first graph node of each frame  (N_b = H_b + M_b)
 * ------------------------------------------------------------------------------------------- */

/* Stage 1a. CSR/COO graph of every frame: MergedMultipleHumansDataset.process_test +
 * add_edge_node_to_graph (graph_generator.py:813-876, 627-656) without DGL.
 * Outputs (E_b = H_b + 5*M_b edges per frame, edge_off[b] = head_off[b] + 5*(node_off[b]-head_off[b])):
 *   src,dst  [E_tot] i32 frame-local node ids in the reference's edge-id order
 *   row_ptr  [N_tot+1] i32, col [E_tot] i32: CSR by destination, GLOBAL node ids, in-edges of a node
 *            in ascending reference edge id
 *   pairs    [M_tot,2] i32 frame-local (head1, head2) of every edge-node, edge-node order
 *   node_cam [N_tot] i32 index into used_cameras_skeleton_matching, -1 for edge-nodes ('' in the reference)
 * Any output pointer may be null to skip it. */
int b200pose_build_graph(int32_t n_frames, const int32_t* head_off, const int32_t* node_off,
                         const int32_t* sk_cam, const b200pose_cameras* cams_host,
                         int32_t* src, int32_t* dst, int32_t* row_ptr, int32_t* col,
                         int32_t* pairs, int32_t* node_cam, void* stream);

/* Stage 1a', training-side topology. The same five edges per edge-node (add_edge_node_to_graph,
 * graph_generator.py:627-656) for an EXPLICIT edge-node list: process_training (:672-810) orders edge-nodes by its
 * people / other-people / spurious loops and creates both (h1,h2) and (h2,h1), and dgl.batch
 * (train_skeleton_matching.py:80, sm_metrics_without_gt.py:60) concatenates graphs - "frames" here are graphs of a
 * block-diagonal batch, nodes of a graph = its heads then its edge-nodes.
 *   pairs [M_tot,2] i32 graph-local (head1, head2) of every edge-node, in edge-node order (input)
 *   max_heads_per_graph sizes the per-graph scan; outputs as b200pose_build_graph (CSR in ascending edge id). */
int b200pose_build_graph_pairs(int32_t n_graphs, const int32_t* head_off, const int32_t* node_off,
                               const int32_t* sk_cam, const b200pose_cameras* cams, const int32_t* pairs,
                               int32_t max_heads_per_graph,
                               int32_t* src, int32_t* dst, int32_t* row_ptr, int32_t* col,
                               int32_t* node_cam, void* stream);

/* Stage 1b. Node features of alternative '3' (HumanGraphFromView.initializeWithAlternative3,
 * graph_generator.py:444-508), bit-exact fp32.
 *   feats_f32 != null : dense [N_tot, ld_f32] rows for every node (edge-nodes: one-hot column 1) - what
 *                       the reference stores in g.ndata['h'];
 *   head_hi/lo != null: planes [S+1, ld_planes] holding the S head rows plus ONE edge-node row (row S);
 *                       all edge-node rows are identical, so layer 0 of the GAT only projects S+1 rows. */
int b200pose_node_features(int32_t n_frames, int32_t n_heads_total, int32_t n_nodes_total, const int32_t* head_off,
                           const int32_t* node_off, const double* sk_xy, const float* sk_vp,
                           const uint32_t* sk_mask, const int32_t* sk_cam,
                           const b200pose_cameras* cams_host,
                           float* feats_f32, int32_t ld_f32,
                           uint16_t* head_hi, uint16_t* head_lo, int32_t ld_planes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dense projections (nn.Linear of gat2.py:53,55 and utils/mlp.py:8-28):
 *   out = act(A[M,K] * W[N,K]^T + bias[N]),  act(x) = x >= 0 ? x : slope*x   (slope = 1 -> identity)
 * A, W as planes (K-major, lda/ldw multiples of 64, K zero-padded up to a multiple of 64).
 * Outputs (either or both): out_f32 [M, ld_out] and/or planes out_hi/out_lo [M, ld_planes]. Plane
 * padding columns (>= N) are only ever written as zero; the caller zero-initialises plane buffers once
 * so the padding can be consumed as K padding by the next GEMM.
 * out_scale multiplies the result after the activation (x10 of metrics_from_model.py:282).
 * impl: 0 = persistent tcgen05 + TMA tensor-core kernel (the product path; CTA pairs with cta_group::2 MMAs and
 * 256-row tiles above 512 rows, single CTAs below); m <= 8 rows (the pose MLP of a live frame) go to a weight-streaming
 * kernel that keeps A in registers and splits k over the lanes of a CTA, 9..16 rows to one that stages A in shared memory
 * and gives every warp an output column - either way every hi/lo weight is read once;
 * 4 / 5 / 7 force single CTAs / CTA pairs / the few-row kernels (m <= 16; more rows go to the dispatch's persistent kernel).
 * Any other value is refused with B200POSE_E_INVALID.
 * ------------------------------------------------------------------------------------------- */
int b200pose_linear(const uint16_t* a_hi, const uint16_t* a_lo, int32_t lda,
                    const uint16_t* w_hi, const uint16_t* w_lo, int32_t ldw,
                    const float* bias, int32_t m, int32_t n, int32_t k, float slope, float out_scale,
                    float* out_f32, int32_t ld_out,
                    uint16_t* out_hi, uint16_t* out_lo, int32_t ld_planes,
                    int32_t impl, void* stream);
/* b200pose_linear for a CAPACITY of rows (the buffers and tensor maps cover m_capacity rows) with the number of valid
 * rows read from the device when the kernel starts: m-tiles past it are not computed. */
int b200pose_linear_n(const uint16_t* a_hi, const uint16_t* a_lo, int32_t lda,
                      const uint16_t* w_hi, const uint16_t* w_lo, int32_t ldw,
                      const float* bias, int32_t m_capacity, const int32_t* m_dev, int32_t n, int32_t k,
                      float slope, float out_scale,
                      float* out_f32, int32_t ld_out, uint16_t* out_hi, uint16_t* out_lo, int32_t ld_planes,
                      int32_t impl, void* stream);
/* Two projections in one launch when the second is only a few columns wide (the last GAT layer: fc1 150 -> 150, then
 * fc2 + attention dots 150 -> 3, gat2.py:53-58 with num_heads = 1, out_dim = 1):
 *   out2[m, n2] = LeakyReLU_slope1(A W1^T + b1) W2^T + b2,  n1 <= 256, n2 <= 4.
 * The first projection runs on the tensor cores as in b200pose_linear; its activated rows never leave the epilogue
 * registers - each is dotted with the n2 fp32 rows of W2 there (w2_f32 [n2, ldw2], rows padded with zeros to a multiple of
 * 64 columns, 16-byte aligned). Saves writing and re-reading the intermediate planes (2 x 141 MB at 184 k rows). */
int b200pose_linear_fused2(const uint16_t* a_hi, const uint16_t* a_lo, int32_t lda,
                           const uint16_t* w1_hi, const uint16_t* w1_lo, int32_t ldw1, const float* bias1,
                           int32_t m, int32_t n1, int32_t k, float slope1,
                           const float* w2_f32, int32_t ldw2, const float* bias2, int32_t n2,
                           float* out2_f32, int32_t ld_out2, void* stream);

/* fp32 [rows, ld_in] -> planes [rows, ld_planes] (used once per weight matrix at load time, and by tests) */
int b200pose_split_planes(const float* x, int32_t rows, int32_t cols, int32_t ld_in,
                          uint16_t* hi, uint16_t* lo, int32_t ld_planes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Stage 2a. Fused attention logits + edge-softmax + neighbour aggregation of one GAT layer:
 * GraphAttention2.forward lines gat2.py:59-68 (apply_edges edge_attention :78-81, edge_softmax
 * :83-88, update_all(u_mul_e, sum) :66), one warp per destination node over the CSR.
 *   z [rows, ldz] fp32: per source row [ ft2 (heads*dim) | a1 (heads) | a2 (heads) ] as produced by
 *     b200pose_linear with the attention vectors folded into the projection;
 *   layer0 != 0: z holds S+1 compact rows (heads + the shared edge-node row, see node_features);
 *   max_heads_per_frame / max_enodes_per_frame size the shared-memory plan of a frame (0 = unknown);
 *   impl: 0 = frame-resident column-parallel kernel when a frame's plan fits in shared memory (<= 32 heads per
 *         frame), the large-frame kernel (edge-node chunks with staged head rows + head destinations over cp.async
 *         row rings) above 48 heads per frame and for batches of a few frames (fewer than SMs / 8: one CTA per frame
 *         would pay a single CTA's latency), else the warp-per-destination gather kernel; 1 = always the gather kernel,
 *         2 = the large-frame kernel where its plan fits, 3 = the frame-resident kernel (error if the plan does not fit);
 *   out[v,h,:] = sum_u softmax_u(LeakyReLU_alpha(a1[u,h] + a2[v,h])) * ft2[u,h,:]
 * Outputs (any may be null): raw_f32 [N_tot, heads*dim] (the layer output, gat2.py:68),
 *   planes act_hi/lo [N_tot, ld_planes] = LeakyReLU_{act_slope}(out) (GAT2.forward :141-142),
 *   scores [N_tot] = sigmoid(out[:,0]) (final_activation, :144-145; requires heads*dim == 1). */
int b200pose_gat_aggregate(int32_t n_frames, int32_t n_nodes_total, int32_t n_heads_total,
                           const int32_t* head_off, const int32_t* node_off,
                           const int32_t* row_ptr, const int32_t* col,
                           const float* z, int32_t ldz, int32_t heads, int32_t dim, int32_t layer0,
                           int32_t max_heads_per_frame, int32_t max_enodes_per_frame, float alpha, float act_slope,
                           float* raw_f32, uint16_t* act_hi, uint16_t* act_lo, int32_t ld_planes,
                           float* scores, int32_t impl, void* stream);
/* The same layer with a residual connection (GraphAttention2 built with residual=True and in_dim != out_dim,
 * gat2.py:43-48, 70-75): out[v] = res[v] + sum_u softmax * ft2[u], `res` [N, ld_res] fp32 = res_fc(h) computed by the caller
 * with b200pose_linear. Not the shipped configuration (train_skeleton_matching.py:50: residual = False); served by the
 * gather kernel. */
int b200pose_gat_aggregate_res(int32_t n_frames, int32_t n_nodes_total, int32_t n_heads_total,
                               const int32_t* head_off, const int32_t* node_off,
                               const int32_t* row_ptr, const int32_t* col,
                               const float* z, int32_t ldz, int32_t heads, int32_t dim,
                               int32_t max_heads_per_frame, int32_t max_enodes_per_frame, float alpha, float act_slope,
                               const float* res, int32_t ld_res,
                               float* raw_f32, uint16_t* act_hi, uint16_t* act_lo, int32_t ld_planes,
                               float* scores, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Stage 2b. Person proposals: get_person_proposal_from_network_output
 * (utils/skeleton_matching_utils.py:12-132) - threshold, score-ordered greedy camera-exclusive merge,
 * connected components - one warp per frame, bit-exact including the CPython-set iteration order the
 * reference's result depends on.
 *   scores [N_tot] fp32 (only edge-node entries are read), pairs/node_cam from b200pose_build_graph;
 *   threshold is compared as the reference does (python float(fp32 score) > threshold, strict);
 *   max_heads_per_frame / max_enodes_per_frame size the per-frame shared-memory plan
 * Outputs: person_heads [S_tot, v_sm] i32: rows head_off[b] .. head_off[b]+n_persons[b]-1 hold the persons
 *   of frame b in the reference's output order, frame-local head id per camera or -1 (None);
 *   n_persons [B] i32. */
int b200pose_cluster(int32_t n_frames, const int32_t* head_off, const int32_t* node_off,
                     const int32_t* pairs, const int32_t* node_cam, const float* scores,
                     int32_t v_sm, double threshold, int32_t min_views,
                     int32_t max_heads_per_frame, int32_t max_enodes_per_frame,
                     int32_t* person_heads, int32_t* n_persons, void* stream);

/* Stage 2b on graphs built by b200pose_build_graph_pairs (training-side topology, dgl.batch members): the same
 * function, with the first-seen head order of the reference's edge walk (skeleton_matching_utils.py:32-47) taken from
 * the explicit pair list instead of the closed form of the test-mode graph. */
int b200pose_cluster_pairs(int32_t n_graphs, const int32_t* head_off, const int32_t* node_off,
                           const int32_t* pairs, const int32_t* node_cam, const float* scores,
                           int32_t v_sm, double threshold, int32_t min_views,
                           int32_t max_heads_per_graph, int32_t max_enodes_per_graph,
                           int32_t* person_heads, int32_t* n_persons, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Stage 3a. MLP-input encoder: PoseEstimatorDataset.__init__ dict branch + get_3D_from_triangulation
 * (utils/pose_estimator_dataset_from_json.py:237-289, 63-101): fp64 undistortion (cv2.undistortPoints,
 * 5 iterations), back-projected rays, pairwise fp64 DLT (cv2.triangulatePoints) averaged over pairs.
 *   person_sk [P, C] i32: GLOBAL skeleton index (into sk_*) of the person in each camera, -1 = absent
 * Outputs: x_f32 [P, ld_f32] (may be null) and/or planes x_hi/x_lo [P, ld_planes]; row length 252*v_pe;
 *   valid [P] u8 = 1 iff sum|x| > 1 (the reference only keeps such rows, dataset.py:287). */
int b200pose_encode_persons(int32_t n_persons, const int32_t* person_sk,
                            const double* sk_xy, const float* sk_vp, const uint32_t* sk_mask,
                            const b200pose_cameras* cams_host,
                            float* x_f32, int32_t ld_f32, uint16_t* x_hi, uint16_t* x_lo, int32_t ld_planes,
                            uint8_t* valid, void* stream);
/* The same, launched for a CAPACITY of persons with the real count left on the device by the previous stage
 * (person_off[B] of b200pose_gather_persons): rows >= *n_persons_dev are not touched. Lets a whole step be enqueued
 * without the host reading the person count back (the reference has no counterpart: it is one frame at a time). */
int b200pose_encode_persons_n(int32_t capacity, const int32_t* n_persons_dev, const int32_t* person_sk,
                              const double* sk_xy, const float* sk_vp, const uint32_t* sk_mask,
                              const b200pose_cameras* cams_host,
                              float* x_f32, int32_t ld_f32, uint16_t* x_hi, uint16_t* x_lo, int32_t ld_planes,
                              uint8_t* valid, void* stream);

/* Stage 3b. Triangulation baseline: triangulate() (utils/pose_estimator_utils.py:52-75) fed as
 * test/metrics_from_triangulation.py:237-249 does (all present joints, camera order = camera index):
 * pairwise DLT, upper median on coordinate `median_axis`, keep pairs within 0.05 of it, mean.
 * Outputs: xyz [P,18,3] fp64, mask [P,18] u8 (joint seen by >= 2 cameras). */
int b200pose_triangulate(int32_t n_persons, const int32_t* person_sk,
                         const double* sk_xy, const uint32_t* sk_mask,
                         const b200pose_cameras* cams_host, int32_t median_axis,
                         double* xyz, uint8_t* mask, void* stream);

/* Helper for stage 2b -> 3a: flattens person_heads/n_persons into a dense person list.
 *   person_off [B+1] i32 (exclusive scan of n_persons, computed by the caller or by this call when
 *   scan != 0), person_sk [P_tot, C] i32 global skeleton ids, person_frame [P_tot] i32. */
int b200pose_gather_persons(int32_t n_frames, const int32_t* head_off, const int32_t* person_heads,
                            const int32_t* n_persons, int32_t* person_off, int32_t scan,
                            const int32_t* sk_cam, int32_t v_sm, const b200pose_cameras* cams_host,
                            int32_t* person_sk, int32_t* person_frame, void* stream);

/* Multi-GPU: one rank's results as the fixed-size int32 record of the final gather (SURVEY.md 8e: frames are sharded,
 * the only exchange is a gather of padded per-rank records; the reference has no counterpart - it is single-process).
 *   record = [ P | n_persons[frames_cap] | person_sk[persons_cap, C] (+head_base where >= 0) | joints[persons_cap, n_out] fp32 bits ]
 * P is read from person_off[n_frames] on the device, so the call needs no host-side person count. */
int b200pose_pack_record(int32_t n_frames, int32_t n_cameras, int32_t n_out,
                         const int32_t* n_persons, const int32_t* person_off, const int32_t* person_sk,
                         const float* joints, int32_t ld_joints, int32_t frames_cap, int32_t persons_cap,
                         int32_t head_base, int32_t* record, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Training side (SURVEY.md 8f-3, after the forward): the backward pass and the optimiser step of the skeleton-matching
 * loop, skeleton_matching/train_skeleton_matching.py:163-184. The reference has no hand-written backward - torch autograd
 * differentiates gat2.py:50-88, 137-149 - so these entry points replace `loss.backward()` / `optimizer.step()` for the GAT.
 * The projections' gradients (dW = G^T X, dX = G W) run on b200pose_linear with the transposed planes produced below.
 * Everything is deterministic (no atomics).
 * ------------------------------------------------------------------------------------------- */
/* Backward of b200pose_gat_aggregate (gat2.py:59-66, 78-88: attention logits, edge softmax, weighted sum) for one layer.
 *   z [N, ldz] = [ft2 | a1 | a2] of the forward, dout [N, ld_dout] = gradient of the layer output (before the inter-layer
 *   activation), attn_l / attn_r [heads*dim] fp32 (gat2.py:35-36), stats [N * heads * 3] fp32 scratch.
 *   dz [N, ld_dz] = [d ft2 (incl. the a1 / a2 paths through gat2.py:57-58) | d a1 | d a2].
 * The graph must be symmetric (v in row(u) <=> u in row(v)), which every graph of graph_generator.py:627-656 is. */
int b200pose_gat_aggregate_bwd(int32_t n_nodes, const int32_t* row_ptr, const int32_t* col,
                               const float* z, int32_t ldz, int32_t heads, int32_t dim, float alpha,
                               const float* dout, int32_t ld_dout, const float* attn_l, const float* attn_r,
                               float* stats, float* dz, int32_t ld_dz, void* stream);
/* x = g * (mask_hi ? LeakyReLU'_slope(mask) : 1) -> out_f32 (may alias g) and/or planes [rows, ld_p] and/or TRANSPOSED
 * planes [cols, ld_t] (padding columns up to the next multiple of 64 zero: the K padding of b200pose_linear). mask_hi = hi plane of the activated tensor (same sign as its input;
 * autograd: nn.LeakyReLU backward, gat2.py:54, 141-142). */
int b200pose_grad_planes(const float* g, int32_t rows, int32_t cols, int32_t ld_g,
                         const uint16_t* mask_hi, int32_t ld_mask, float slope,
                         float* out_f32, int32_t ld_out,
                         uint16_t* p_hi, uint16_t* p_lo, int32_t ld_p,
                         uint16_t* t_hi, uint16_t* t_lo, int32_t ld_t, void* stream);
/* planes [rows, ld] -> planes [cols, ld_t] of the transposed matrix (columns [rows, round_up(rows, 64)) zero) */
int b200pose_transpose_planes(const uint16_t* hi, const uint16_t* lo, int32_t rows, int32_t cols, int32_t ld,
                              uint16_t* t_hi, uint16_t* t_lo, int32_t ld_t, void* stream);
/* out[j] = sum_r x[r, j] * (w ? w[r, j / group] : 1): bias gradients; d attn[h, d] = sum_u d a[u, h] ft2[u, h, d] */
int b200pose_colsum(const float* x, int32_t rows, int32_t cols, int32_t ld, const float* w, int32_t ld_w, int32_t group,
                    float* out, void* stream);
/* A whole layer in one launch each. b200pose_gat_prepare_layer: every operand plane of a layer from its fp32 parameters (W1 and
 * W1^T planes, [W2 ; folds] planes + folded bias b2e, W2^T planes; ld_w1 = ld_w2 = round_up(din, 64)), where
 * [W2 ; folds] = [W2 ; sum_d attn_l[h,d] W2[h*dim+d, :] ; same with attn_r] and b2e likewise (gat2.py:55-58 as one projection;
 * the inference path does this fold once on the host, a training step after every parameter update).
 * b200pose_gat_attn_bias_grad: the three column sums behind b200pose_gat_aggregate_bwd (d attn_l, d attn_r, d fc2.bias) in one
 * pass over z and dz. */
int b200pose_gat_prepare_layer(const float* w1, const float* w2, int32_t ld_w, const float* b2, const float* attn_l,
                               const float* attn_r, int32_t heads, int32_t dim, int32_t din,
                               uint16_t* w1_hi, uint16_t* w1_lo, int32_t ld_w1, uint16_t* w1t_hi, uint16_t* w1t_lo, int32_t ld_w1t,
                               uint16_t* w2_hi, uint16_t* w2_lo, int32_t ld_w2, uint16_t* w2t_hi, uint16_t* w2t_lo, int32_t ld_w2t,
                               float* b2e, void* stream);
int b200pose_gat_attn_bias_grad(const float* z, int32_t ldz, const float* dz, int32_t ld_dz, int32_t rows, int32_t heads, int32_t dim,
                                float* g_attn_l, float* g_attn_r, float* g_b2, void* stream);
/* Backward of a residual connection (gat2.py:70-75): dx[r, c] += sum_{h < heads} src[r, h * cols + c]. heads = 1: src = the gradient
 * that came back through res_fc (computed with b200pose_linear); heads = H: the identity branch (resval = h.unsqueeze(1),
 * broadcast over the attention heads), src = the layer's output gradient. */
int b200pose_residual_bwd_add(float* dx, int32_t ld_dx, const float* src, int32_t ld_src, int32_t rows, int32_t cols, int32_t heads,
                              void* stream);
/* nn.MSELoss on scores[idx[i]] vs labels[i] (train_skeleton_matching.py:37, 174-178) and its gradient through the final
 * sigmoid: dlogit [n_nodes] (zero outside idx; idx entries distinct). loss / dlogit may be null. */
int b200pose_mse_sigmoid(const float* scores, int32_t n_nodes, const int32_t* idx, const float* labels, int32_t m,
                         float* loss, float* dlogit, void* stream);
/* dlogit = dscores * s * (1 - s): the final sigmoid when the loss is computed by the caller (autograd drop-in) */
int b200pose_sigmoid_bwd(const float* scores, const float* dscores, int32_t n, float* dlogit, void* stream);
/* torch.optim.Adam (train_skeleton_matching.py:150), single-tensor form, over one flat parameter buffer, with the step count
 * kept on the device: *step_dev is advanced by one and the bias corrections are computed there
 * (scalars_dev: 2 floats of scratch), so a whole optimisation step - forward, loss, backward, this - is replayable as a CUDA graph */
int b200pose_adam_step_dev(float* theta, const float* grad, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                           float eps, float weight_decay, int32_t* step_dev, float* scalars_dev, void* stream);

/* One linear layer of a flat parameter buffer for b200pose_mlp_adam_planes: the weight [n, k] at theta[offset], rows ld >= k
 * floats apart; its split-bf16 operand planes W [n, ld_w] (ld_w a multiple of 64, >= ld) and, unless wt_hi is null, W^T
 * [k, ld_wt] (ld_wt a multiple of 64, >= n). */
typedef struct {
    int64_t offset;
    int32_t n, k, ld;
    uint16_t *w_hi, *w_lo;
    int32_t ld_w;
    uint16_t *wt_hi, *wt_lo;
    int32_t ld_wt;
} b200pose_mlp_layer;
/* b200pose_adam_step_dev over theta[0, n_total) (bit-identical theta, m, v, *step_dev and scalars_dev) fused with the refresh of
 * every layer's operand planes from the updated weights, in one launch after the scalar kernel (PoseEstimatorMLP, utils/mlp.py:8-31,
 * trained with torch.optim.Adam). The weight slots come in increasing offset order, the first at 0; the floats between a weight
 * slot and the next one (or n_total) - the layer's bias - are updated too. Plane paddings (columns [k, ld_w) of W, columns
 * [n, round_up(n, 64)) of W^T) are written as zeros. grad == null: planes only, from theta as it is (theta, m, v, lr ... and the
 * step count are not touched; m, v, step_dev, scalars_dev may be null). At most 16 layers. */
int b200pose_mlp_adam_planes(float* theta, const float* grad, float* m, float* v, int64_t n_total,
                             const b200pose_mlp_layer* layers, int32_t n_layers, float lr, float beta1, float beta2,
                             float eps, float weight_decay, int32_t* step_dev, float* scalars_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Host-side frame packer (no GPU work): the reference's frame JSON - a list of frames
 * {camera: [json.dumps([skeleton, ...]), timestamp, ...]} as read by test/metrics_from_model.py:117-191, or one such
 * frame - parsed in parallel into the packed skeleton batch above. Replaces json.loads + the per-joint Python loops of
 * graph_generator.py:573-605. cam_names[i] -> cam_index[i] lists the cameras of used_cameras_skeleton_matching;
 * other cameras are skipped. Numbers are converted exactly like Python's float().
 *   b200pose_pack_json   : parses; *out_handle owns the result until b200pose_packed_free
 *   b200pose_packed_sizes: frame / head / node counts and the per-frame maxima the kernels are sized with
 *   b200pose_packed_copy : writes the arrays into caller-provided HOST buffers (pinned memory works best):
 *                          sk_xy [S,18,2] f64, sk_vp [S,18,2] f32, sk_mask [S] u32, sk_cam [S] i32, head_off/node_off [B+1] i32,
 *                          skeleton_index [S] i32 (position of the skeleton in its camera's list; may be null)
 * n_threads <= 0 uses every hardware thread.
 * ------------------------------------------------------------------------------------------- */
int b200pose_pack_json(const char* json_host, int64_t len, int32_t n_cams, const char* const* cam_names_host,
                       const int32_t* cam_index_host, int32_t n_threads, void** out_handle);
int b200pose_packed_sizes(const void* handle, int32_t* n_frames, int32_t* n_heads, int32_t* n_nodes,
                          int32_t* max_heads, int32_t* max_enodes);
int b200pose_packed_copy(const void* handle, double* sk_xy_host, float* sk_vp_host, uint32_t* sk_mask_host,
                         int32_t* sk_cam_host, int32_t* head_off_host, int32_t* node_off_host,
                         int32_t* skeleton_index_host, int32_t n_threads);
void b200pose_packed_free(void* handle);

#ifdef __cplusplus
}
#endif
#endif /* B200POSE_H */
