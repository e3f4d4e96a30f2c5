/*
 * p6d.h -- C ABI of libp6d.so, the B200 (sm_100a) pose-geometry library.
 *
 * The reference (SFR-Vision/6d-pose-estimation) is pure Python and has no FFI of its
 * own; the drop-in boundary is the Python call surface of models/add_loss.py,
 * models/pose_loss.py and utils/camera.py (SURVEY.md section 8b).  Each entry point below
 * names the reference code it replaces; the ctypes binding a maintainer would add is in
 * INTEGRATION.md and lives in 6d-pose-estimation_b200/_lib.py.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types in the signatures
 *     (`stream` is a cudaStream_t passed as void*, NULL = legacy default stream);
 *   - every function returns 0 on success and a negative P6D_E* code on failure;
 *     p6d_last_error() returns the thread-local message of the last failure;
 *   - unless the name ends in _host, data pointers are DEVICE pointers on the device the
 *     mesh table (or, for table-less calls, the `device` argument) belongs to, float32
 *     contiguous, quaternions scalar-last [x,y,z,w], translations in metres, K row-major
 *     3x3; the caller owns every buffer; [B,4] float rows and int32 boxes must be 16-byte aligned,
 *     [B,2] rows 8-byte aligned (vector loads; a misaligned pointer is refused with P6D_EINVAL);
 *   - there is no CPU fallback: without a CUDA device every compute entry fails with
 *     P6D_ECUDA;
 *   - threading: the table-less entries and p6d_add_eval / p6d_add_backward may be called
 *     from several host threads at once (launches on different streams of one table use
 *     separate scheduler counters, up to 256 in flight); the *_host entries and
 *     create/destroy own the table's staging buffers and must not run concurrently on
 *     the same table.  One launch takes at most 2^31 - 2^20 poses.
 */
#ifndef P6D_H_
#define P6D_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define P6D_VERSION 4

#define P6D_OK 0
#define P6D_EINVAL (-1)   /* bad argument */
#define P6D_ECUDA (-2)    /* CUDA runtime error (message has the CUDA string) */
#define P6D_ENOMEM (-3)   /* host or device allocation failed */
#define P6D_ETOOBIG (-4)  /* mesh does not fit the shared-memory budget of the kernel */

int p6d_version(void);
const char* p6d_last_error(void);

/* Device facts used by the host side to size grids / report rooflines. */
int p6d_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, int* sm_clock_khz,
                    int64_t* smem_per_block_optin);

/* ---------------------------------------------------------------------------------------
 * Mesh table: device-resident copy of ADDLoss.points / ADDLoss.diameters
 * (reference: models/add_loss.py:21-22, filled by _load_models :29-81).
 *   xyz        host, row-major [sum counts, 3] float32, objects back to back
 *   offsets    host [n_slots] first point of object id s
 *   counts     host [n_slots] point count, 0 = id not in self.points (poses with that id
 *              are skipped, add_loss.py:171-172)
 *   diameters  host [n_slots] metres, float64; threshold = 0.1 * diameter in float64 (:176)
 *   symmetric  host [n_slots] 1 for ids in SYMMETRIC_OBJECT_IDS (:10)
 * The table stores each mesh as a 16-byte aligned SoA block x[Np] y[Np] z[Np]
 * (Np = count rounded up to 4) so one TMA bulk copy stages it into shared memory.
 * ------------------------------------------------------------------------------------- */
typedef struct p6d_mesh_table p6d_mesh_table;

int p6d_mesh_table_create(const float* xyz, const int32_t* offsets, const int32_t* counts,
                          const double* diameters, const uint8_t* symmetric, int n_slots, int device,
                          p6d_mesh_table** out);
int p6d_mesh_table_destroy(p6d_mesh_table* table);
/* Largest mesh (points) the ADD-S kernel accepts on this device. */
int p6d_adds_max_points(int device, int* max_points);

/* The build's post-link pass (csrc/sass_sched.py) re-lays the scan loop of the ADD-S kernels (same
 * instructions, other order and stall counts; +4...9 % throughput).  Before a re-laid kernel is
 * used on a device, the library runs it and the ptxas-scheduled kernel of the same mesh-size class
 * on 592 seeded poses and compares every output byte; on any difference it prints one line to
 * stderr and uses the ptxas-scheduled kernel for the rest of the process.  The environment
 * variable P6D_ADDS_SCHEDULE=ptxas turns the re-laid kernels off altogether.
 *   p6d_adds_schedule()        1 if re-laid kernels are in the build and none has been rejected
 *   p6d_adds_schedule_state()  for the table's class: built_relaid 0/1; runtime_state 0 = not yet
 *                              checked, 1 = verified on this device, 2 = rejected
 *   p6d_adds_selfcheck()       runs the comparison now on n_poses seeded poses over the table's
 *                              meshes; mismatches = differing output bytes (0 when nothing is re-laid) */
int p6d_adds_schedule(void);
int p6d_adds_schedule_state(const p6d_mesh_table* table, int* built_relaid, int* runtime_state);
int p6d_adds_selfcheck(const p6d_mesh_table* table, int64_t n_poses, int64_t* mismatches);

/* All 2^32 float32 bit patterns through the packed square roots of kernel (a) (two-way and
 * four-way form) and through sqrt.rn.f32; mismatches must come back 0. */
int p6d_selftest_sqrt2(int device, int64_t* mismatches);

/* ---------------------------------------------------------------------------------------
 * Per-pose evaluation = the loop body of ADDLoss.eval_metrics (models/add_loss.py:168-195)
 * for B poses in one launch.
 *   pq,gq [B,4]  pt,gt [B,3]  obj [B] int64
 *   order        nullable [B] int32: processing order (e.g. argsort of obj so consecutive
 *                poses share a mesh); outputs are still written at the original index
 *   add  [B]     mean_i |pred_i - gt_i|                       (:181-183)
 *   adds [B]     mean_i min_j |pred_i - gt_j|, pred-major      (:185-190); NULL = skip the
 *                all-pairs part (ADD-only kernel, symmetric ids then decide on ADD)
 *   hit  [B]     (double)(symmetric ? adds : add) < 0.1*diameter  (:192-195)
 *   valid[B]     0 where the object id has no mesh (outputs 0 there)
 *   borderline   nullable [B]: 1 where the deciding distance lies within 4 float32 ulp of the
 *                threshold (SURVEY.md 7.3.1) -- the band in which a reference running on another
 *                BLAS / ATen build could round to the other side; callers that need certainty
 *                against such a build re-evaluate exactly these poses with it
 *   acc          nullable per-object accumulators updated with atomics (not zeroed here):
 *                hits[n_slots], valid[n_slots] int64; add_sum[n_slots], adds_sum[n_slots]
 *                float64 (any of the four pointers may be NULL)
 * Distances reproduce the reference's float32 arithmetic bit for bit, including the
 * summation order of Tensor.mean() on the CPU (see DESIGN.md).
 * ------------------------------------------------------------------------------------- */
typedef struct p6d_accumulators {
    int64_t* hits;
    int64_t* valid;
    double* add_sum;
    double* adds_sum;
} p6d_accumulators;

int p6d_add_eval(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                 const float* gt, const int64_t* obj, const int32_t* order, int64_t B, float* add,
                 float* adds, uint8_t* hit, uint8_t* valid, uint8_t* borderline,
                 const p6d_accumulators* acc, void* stream);

/* OPT-IN: the same outputs, bit for bit, from a kernel that skips gt points which provably cannot be a
 * nearest neighbour (exact block pruning: the mesh is cut into spatially compact 32-point blocks at table
 * creation; per pose a block pair is skipped when the distance of its bounding spheres exceeds the current
 * minima, with margins far above float32 error; anything that is not a number is evaluated).  Not the
 * all-pairs kernel the headline numbers are measured on, and never reported as a roofline fraction.
 *   p6d_add_eval_pruned          always this kernel; adds must not be NULL; a table whose largest mesh exceeds
 *                                ~4,700 points (shared memory) or 65,534 points answers P6D_ETOOBIG
 *   p6d_mesh_table_set_pruning   per-table switch (default off): p6d_add_eval, p6d_add_eval_host and p6d_sweep_run
 *                                then take this kernel where it pays -- largest mesh of the table >= 128 points
 *                                and within the shared-memory limit -- and the all-pairs kernel otherwise
 *                                (the loss form p6d_add_forward always takes the all-pairs kernel). */
int p6d_mesh_table_set_pruning(p6d_mesh_table* table, int enable);
int p6d_add_eval_pruned(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                        const float* gt, const int64_t* obj, const int32_t* order, int64_t B, float* add,
                        float* adds, uint8_t* hit, uint8_t* valid, uint8_t* borderline,
                        const p6d_accumulators* acc, void* stream);

/* OPT-IN: the same outputs, bit for bit, for meshes larger than shared memory.  The resident kernels stage the whole
 * mesh in shared memory and answer P6D_ETOOBIG beyond p6d_adds_max_points (ADD-S) or ~16,700 points (ADD only,
 * adds = NULL); this kernel streams the gt cloud through shared memory in tiles of 1,024 points (TMA bulk copies,
 * transformed by the gt pose per tile) and splits every pose into blocks of pred points, so it takes meshes of up to
 * 32,768 points.  Above that, torch's CPU Tensor.mean() sums a row on several threads and the reference's own result
 * depends on the caller's thread count: such tables answer P6D_ETOOBIG.  It allocates a workspace of 8 bytes per point
 * and pose (at most 64 MB; larger batches run in chunks) stream-ordered on `stream`; no host synchronisation.
 *   p6d_add_eval_streamed            always this kernel, for any mesh of 1 to 32,768 points; adds = NULL gives the
 *                                    ADD-only outputs (symmetric ids then decide on ADD)
 *   p6d_mesh_table_set_large_meshes  per-table switch (default off): p6d_add_eval, p6d_add_eval_host and p6d_sweep_run
 *                                    then take this kernel for a table whose largest mesh is beyond the resident
 *                                    kernel's limit, and the resident kernels otherwise (the loss form
 *                                    p6d_add_forward and p6d_add_backward keep their limit). */
int p6d_mesh_table_set_large_meshes(p6d_mesh_table* table, int enable);
int p6d_add_eval_streamed(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                          const float* gt, const int64_t* obj, const int32_t* order, int64_t B, float* add,
                          float* adds, uint8_t* hit, uint8_t* valid, uint8_t* borderline,
                          const p6d_accumulators* acc, void* stream);

/* Same computation with HOST buffers: stages inputs to the device, runs the kernels,
 * copies results back and synchronises (the end-to-end path of bench.py).  acc_* are
 * host arrays [n_slots] that receive (not accumulate) the per-object totals; nullable.
 * gpu_launches (nullable) receives the number of kernels this call launched. */
int p6d_add_eval_host(p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                      const float* gt, const int64_t* obj, int64_t B, int want_adds, float* add,
                      float* adds, uint8_t* hit, uint8_t* valid, uint8_t* borderline,
                      int64_t* acc_hits, int64_t* acc_valid, double* acc_add_sum, double* acc_adds_sum,
                      int* gpu_launches);

/* ---------------------------------------------------------------------------------------
 * Value of ADDLoss.forward (models/add_loss.py:101-150) in ONE launch and no host
 * synchronisation: per sample ADD (asymmetric ids) or ADD-S (symmetric ids) with the rounding
 * of the reference's batched torch.matmul, then -- by the last CTA to finish -- the reference's
 * grouping: objects in order of first appearance, per object the float32 sum of its samples
 * (ATen order), added to the running total; total / count.
 *   loss  [1] device float32 (0 when no sample has a mesh); count [1] device int32
 *   workspace: device buffer of p6d_add_forward_workspace_bytes(table, B) bytes, 16-byte aligned
 * Bit-exact against the reference for meshes of up to 44 points (ATen's naive bmm kernel) and
 * from 45 points on (MKL, fused chain), except group sizes for which MKL's batched sgemm takes
 * another path: 1e-5 there.  tests/test_loss_form.py measures where, on the machine it runs on,
 * over n = 1...3,000 points x g = 1...257 samples per group (24 x 17 points).  Measured: on an
 * 8-thread x86 CPU (torch 2.11.0, MKL) exactly 2 samples of a 97- or a 200-point mesh, ADD-S
 * only.  A point outside g = 2, n = 97...106 or 200 fails the test by name.
 * Groups of more than 32,768 samples are summed in the order of torch's CPU sum on ONE thread.
 * With more threads torch splits such a sum, so the reference's own value then depends on the
 * caller's thread count (measured: within 1e-5).  Such batches are accepted, not refused.
 * ------------------------------------------------------------------------------------- */
int64_t p6d_add_forward_workspace_bytes(const p6d_mesh_table* table, int64_t B);
int p6d_add_forward(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                    const float* gt, const int64_t* obj, int64_t B, float* loss, int32_t* count,
                    void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------
 * Gradient of ADDLoss.forward (models/add_loss.py:101-150) w.r.t. pred_r [B,4] and
 * pred_t [B,3]:  loss = (1/count) * sum over valid samples of ADD (asymmetric ids) or
 * ADD-S (symmetric ids).  grad_out: device pointer to the upstream scalar gradient;
 * count: device pointer to the number of valid samples (as written by p6d_add_forward), or
 * NULL to use the host value inv_count = 1 / count.  Skipped samples get zero gradient.
 * ------------------------------------------------------------------------------------- */
int p6d_add_backward(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                     const float* gt, const int64_t* obj, int64_t B, const float* grad_out,
                     const int32_t* count, float inv_count, float* grad_q, float* grad_t, void* stream);

/* Quaternion -> rotation matrix, ADDLoss._quat_to_mat (models/add_loss.py:203-215). */
int p6d_quat_to_mat(const float* q, int64_t B, float* R, int device, void* stream);

/* ---------------------------------------------------------------------------------------
 * PoseLoss.forward + gradients in one launch (models/pose_loss.py:19-61).
 *   mode 0 = 'geodesic' (:30-50), 1 = quaternion L1 (:52-61)
 *   out[0] = loss, out[1] = rotation term, out[2] = translation term (float32)
 *   grad_q [B,4], grad_t [B,3]: d loss / d pred for upstream gradient 1 (nullable)
 *   workspace: device buffer of p6d_pose_loss_workspace_bytes() bytes, zeroed by the
 *   caller before the first use only (the kernel leaves it zeroed).
 * ------------------------------------------------------------------------------------- */
int64_t p6d_pose_loss_workspace_bytes(void);
int p6d_pose_loss_fwd_bwd(const float* pq, const float* pt, const float* gq, const float* gt,
                          int64_t B, float rot_weight, float trans_weight, int mode, float* out,
                          float* grad_q, float* grad_t, void* workspace, int device, void* stream);

/* The RGB-Geometric training step in ONE launch: kernel (d1) fused into kernel (c).
 * pred_trans is computed in-kernel from (z [B], uv [B,2], K) exactly like p6d_pinhole_fwd
 * (models/pose_net_rgb_geometric.py:93-109) and the loss gradient is returned w.r.t. z
 * (grad_z [B], nullable) exactly like p6d_pinhole_bwd applied to d loss / d pred_trans.
 * trans_out [B,3] (nullable) receives the translation.  Other arguments as above. */
int p6d_pose_loss_pinhole_fwd_bwd(const float* pq, const float* z, const float* uv, const float* K, int k_batched,
                                  const float* gq, const float* gt, int64_t B, float rot_weight,
                                  float trans_weight, int mode, float* out, float* grad_q, float* grad_z,
                                  float* trans_out, void* workspace, int device, void* stream);

/* ---------------------------------------------------------------------------------------
 * Pinhole XY from bbox centre and predicted Z
 * (PoseNetRGBGeometric._compute_pinhole_translation, models/pose_net_rgb_geometric.py:93-109).
 *   z [B], uv [B,2], K [3,3] (k_batched = 0) or [B,3,3]; out [B,3] = (((u-cx)*z)/fx, ..., z)
 * Backward: grad_z [B] = gx*(u-cx)/fx + gy*(v-cy)/fy + gz for grad_out [B,3].
 * ------------------------------------------------------------------------------------- */
int p6d_pinhole_fwd(const float* z, const float* uv, const float* K, int k_batched, int64_t B,
                    float* out, int device, void* stream);
int p6d_pinhole_bwd(const float* grad_out, const float* uv, const float* K, int k_batched, int64_t B,
                    float* grad_z, int device, void* stream);

/* ---------------------------------------------------------------------------------------
 * Depth sample + back-projection
 * (PoseNetRGBDGeometric._compute_pinhole_translation, models/pose_net_rgbd_geometric.py:56-85).
 *   depth [B,H,W] metres; centre clamped to [0,clamp_hi] (reference: 223), truncated for
 *   the index; z <= 0.01 or NaN -> 0.5; clamp [0.1, 2.0]; pinhole XYZ.  out [B,3].
 * ------------------------------------------------------------------------------------- */
int p6d_depth_backproject(const float* depth, int H, int W, const float* uv, const float* K,
                          int k_batched, int64_t B, float clamp_hi, float* out, int device,
                          void* stream);

/* ---------------------------------------------------------------------------------------
 * Frame-level fusion of the crop pipeline with the depth back-projection (SURVEY.md N1):
 * LineMODDatasetRGBD.__getitem__ (data/dataset_rgbd.py:104-179: pad, square crop of
 * 1.2 x max(w,h), cv2.resize to img_size, centre and K remapped into crop coordinates)
 * followed by models/pose_net_rgbd_geometric.py:56-85, for B integer boxes (x,y,w,h) of ONE
 * uint16 depth frame [H,W] in millimetres and the frame's intrinsics K [3,3].
 *   xyz [B,3]; optional center [B,2] (crop-space bbox centre), kcrop [B,9], z_mm [B]
 *   (the resized crop's uint16 value under the centre).
 *   bilinear  which cv2.resize arithmetic for CV_16U to reproduce bit for bit:
 *             0 = the pip wheel's default (IPP's ippiResizeLinear_16u: the call the reference makes),
 *             1 = OpenCV's own C++ path (builds without IPP, cv2.ipp.setUseIPP(False)).
 * ------------------------------------------------------------------------------------- */
int p6d_depth_crop_backproject(const uint16_t* depth, int H, int W, const int32_t* boxes, int64_t B,
                               const float* K, int img_size, int bilinear, float* xyz, float* center,
                               float* kcrop, uint16_t* z_mm, int device, void* stream);

/* The same fusion for the INFERENCE script's per-detection crop code
 * (scripts/inference/inference_rgbd_geometric.py:109-170, then models/pose_net_rgbd_geometric.py:56-85):
 * B integer detector boxes (x1,y1,x2,y2) of ONE uint16 depth frame [H,W] in millimetres, K [3,3] in
 * FLOAT64 (the script passes utils.camera.DEFAULT_K, a float64 array, and computes centre and K_crop in
 * float64 before storing them as float32).  The crop is cast to float32 before cv2.resize there, so the
 * depth under the centre is the un-rounded float32 lerp of the pip wheel's default path
 * (ippiResizeLinear_32f), reproduced bit for bit; OpenCV's own C++ float path is not offered.
 *   xyz [B,3]; optional center [B,2], kcrop [B,9], z_m [B] (depth_meters under the centre, float32). */
int p6d_detection_backproject(const uint16_t* depth, int H, int W, const int32_t* boxes_xyxy, int64_t B,
                              const double* K, int img_size, float* xyz, float* center, float* kcrop,
                              float* z_m, int device, void* stream);

/* 3-D -> 2-D projection of N model points for B poses (SURVEY.md N4):
 * utils/visualization.project_points (utils/visualization.py:8-32) in float64 --
 * rotation [B,4] quaternions (normalised like scipy's Rotation.from_quat) or [B,3,3];
 * p = R x + t, z clipped to >= 0.001, u = x fx / z + cx, v = y fy / z + cy truncated to
 * integers; uv [B,N,2] int64. */
int p6d_project_points(const double* points, int N, const double* rotation, int rotation_is_quat,
                       const double* translation, const double* K, int64_t B, int64_t* uv, int device, void* stream);

/* ---------------------------------------------------------------------------------------
 * The compare_all_models sweep (scripts/visualization/compare_all_models.py:65-104 at the scale
 * of BASELINE config 5) for one rank, driven natively on two streams.
 *   p6d_synth_poses  seeded pose hypotheses generated on the device; a pure function of
 *                    (seed, obj_index, variant_index, first + i), so any sharding sees the same data.
 *                    kind 0: pred_t direct (RGB / RGBD heads) -> pt
 *                    kind 1: RGB-Geometric inputs z [n], uv [n,2] (bbox centre) for p6d_pinhole_fwd
 *                    kind 2: RGBD-Geometric inputs uv [n,2] (crop centre), kc [n,9], depth [n,8,8]
 *                            for p6d_depth_backproject(H = W = 8, clamp_hi = 7)
 *   p6d_sweep_run    for every (object, variant) block the hypotheses [lo, hi) of n_per_block, in
 *                    chunks: generate, translate (kernel d1 / d2 by variant kind), evaluate
 *                    (ADD + ADD-S + decision) into the variant's accumulator row.
 *                    acc_* : device [n_variants, n_slots], accumulated with atomics (not zeroed);
 *                    check_*: host arrays [n_obj * n_variants * min(check_n, hi - lo), ...] receiving
 *                    the first poses of every block as evaluated (inputs and outputs) so the caller
 *                    can re-evaluate them independently; nullable when check_n = 0.
 *                    Work is ordered after what is already queued on `stream`; the call returns
 *                    after the sweep has finished.
 * ------------------------------------------------------------------------------------- */
int p6d_synth_poses(uint64_t seed, int obj_index, int variant_index, int64_t first, int64_t n,
                    float rot_sigma, float trans_sigma, int kind, const float* K_host, int64_t oid,
                    float* pq, float* pt, float* gq, float* gt, int64_t* obj, float* z, float* uv,
                    float* kc, float* depth, int device, void* stream);
int p6d_sweep_run(p6d_mesh_table* table, const int32_t* obj_ids, int n_obj, const int32_t* variant_kinds,
                  int n_variants, int64_t n_per_block, int64_t lo, int64_t hi, int64_t chunk, uint64_t seed,
                  const float* K_host, float rot_sigma, float trans_sigma, int64_t* acc_hits,
                  int64_t* acc_valid, double* acc_add_sum, double* acc_adds_sum, int64_t check_n,
                  float* check_pq, float* check_pt, float* check_gq, float* check_gt, float* check_add,
                  float* check_adds, uint8_t* check_hit, int* gpu_launches, void* stream);

/* ---------------------------------------------------------------------------------------
 * OPT-IN EVIDENCE KERNEL, not used by any product path: ADD-S (models/add_loss.py:185-190) in GEMM
 * form, d^2 = |p|^2 + |g|^2 - 2 p.g, on the tcgen05 tensor cores (kind::tf32, FP32 accumulators in
 * TMEM); split_terms = 3: error-compensated 3xTF32 operands, 1: plain TF32.  BASELINE.json's
 * north_star excludes tensor cores from the ADD-S kernel "unless a 3xTF32 variant passes the stated
 * tolerance" (1e-5 relative); tests/test_tf32_variant.py measures this kernel against the oracle.
 *   adds [B] device float32: mean_i min_j |pred_i - gt_j| as this formulation computes it
 *   max_ctas: 0 = one CTA per SM.  Synchronises the stream before returning.
 * ------------------------------------------------------------------------------------- */
int p6d_adds_tf32_eval(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                       const float* gt, const int64_t* obj, int64_t B, int split_terms, float* adds,
                       int max_ctas, void* stream);

/* ---------------------------------------------------------------------------------------
 * Measurement helper (no reference counterpart): FP32 issue-rate microbenchmarks that give
 * the roofline its measured denominator.  kind 0 = FFMA only, 1 = packed FFMA2 only,
 * 2 = the ADD-S instruction mix (3 FADD2 + FMUL2 + 2 FFMA2 + FMNMX3 per 2 pairs).
 * Returns achieved TFLOP/s (2 FLOP per FMA lane-op; mix counted as 8 FLOP per pair) and
 * the kernel time in ms.
 * ------------------------------------------------------------------------------------- */
int p6d_fp32_microbench(int kind, int device, int iters, double* tflops, double* ms);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* P6D_H_ */
