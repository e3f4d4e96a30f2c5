/*
 * pose_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT.
 *
 * CPU restatement (plain C, scalar IEEE-754 binary32 arithmetic) of the pose-geometry
 * hot path of SFR-Vision/6d-pose-estimation.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this file's shared object;
 * the product path (6d-pose-estimation_b200/) never does.
 *
 * Parity status: PINNED.  The reference has no tests or golden vectors of its own
 * (SURVEY.md section 4), so the pin is the reference itself: oracle/gen_golden.py imports
 * the reference's Python modules from /root/reference in the build container, runs
 * them on seeded synthetic inputs and commits inputs+outputs under tests/golden/;
 * tests/test_oracle_golden.py checks this file against those vectors (bit-exact for
 * ADD / ADD-S / decisions / translations, 1e-5 relative for the transcendental loss).
 *
 * Every rounding step below is deliberate.  The reference runs PyTorch CPU eager ops;
 * the op-by-op float32 behaviour of those ops was measured in the build container
 * (torch 2.11.0, MKL 2024.2, AVX-512 host) and is restated here:
 *   - elementwise mul/add/sub: one rounding each, never contracted;
 *   - torch.mm([N,3] x [3,3]): k-sequential FMA chain  fma(p2,r2, fma(p1,r1, p0*r0));
 *   - torch.norm(v, dim=-1) over 3 components: sqrt(fma(z,z, fma(y,y, x*x))); over the 4
 *     components of a quaternion row: unfused sequential sum of squares;
 *   - Tensor.sum()/mean() over a contiguous float32 row: ATen's cascade_sum with
 *     256-bit vectors (8 lanes) x 4-way ILP x 4 cascade levels of 16 (see aten_sum);
 *   - the ADD-0.1d compare happens in float64 (Python floats).
 *
 * Build: gcc -O3 -mavx2 -mfma -fPIC -shared -ffp-contract=off -fno-fast-math -pthread (see Makefile).
 * -ffp-contract=off matters: GCC must not fuse a*b+c on its own.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <pthread.h>
#include <unistd.h>

#define P6O_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------
 * ATen cascade_sum, float32, contiguous row (reference: Tensor.mean()/.sum() called at
 * models/add_loss.py:139,142,144,182,189 and models/pose_loss.py:50,61; the kernel
 * itself is PyTorch's aten/src/ATen/native/cpu/SumKernel.cpp, torch==2.9.1 pinned in
 * requirements.txt:5, measured identical on 2.11.0).
 *
 * Shape of the computation, with V = 8 float lanes:
 *   row of n floats = nvec full vectors + (n % V) tail scalars;
 *   the nvec vectors are viewed as [nvec/4][4] -> four independent vector accumulators
 *   ("ILP"), each fed through a 4-level cascade that spills level l into level l+1 every
 *   16^(l+1) additions; left-over vectors go to ILP accumulator 0; the four ILP
 *   accumulators are then added 0+=1, 0+=2, 0+=3; finally a scalar starts at 0, takes
 *   the tail scalars in order, then the 8 lanes in order.
 *   Rows shorter than V use the same ILP/cascade scheme on scalars.
 * ---------------------------------------------------------------------------------- */
#define P6O_V 8
#define P6O_ILP 4
#define P6O_LEVELS 4

static int p6o_ceil_log2(int64_t x) {
    if (x <= 2) return 1;
    int r = 0;
    int64_t v = x - 1;
    while (v > 0) { v >>= 1; ++r; }
    return r;
}

/* Generic strided cascade over `size` steps; step i contributes, for each of the
 * `width` lanes w, the element base[i*step_stride + w].  acc_out[width] receives the
 * result.  width <= P6O_V * P6O_ILP. */
static void p6o_cascade_rows(const float* base, int64_t step_stride, int width, int64_t size,
                             float* acc_out) {
    float acc[P6O_LEVELS][P6O_V * P6O_ILP];
    int level_power = p6o_ceil_log2(size) / P6O_LEVELS;
    if (level_power < 4) level_power = 4;
    const int64_t level_step = (int64_t)1 << level_power;
    const int64_t level_mask = level_step - 1;
    for (int l = 0; l < P6O_LEVELS; ++l)
        for (int w = 0; w < width; ++w) acc[l][w] = 0.0f;

    int64_t i = 0;
    while (i + level_step <= size) {
        for (int64_t j = 0; j < level_step; ++j, ++i) {
            const float* p = base + i * step_stride;
            for (int w = 0; w < width; ++w) acc[0][w] = acc[0][w] + p[w];
        }
        for (int l = 1; l < P6O_LEVELS; ++l) {
            for (int w = 0; w < width; ++w) {
                acc[l][w] = acc[l][w] + acc[l - 1][w];
                acc[l - 1][w] = 0.0f;
            }
            const int64_t mask = level_mask << (l * level_power);
            if ((i & mask) != 0) break;
        }
    }
    for (; i < size; ++i) {
        const float* p = base + i * step_stride;
        for (int w = 0; w < width; ++w) acc[0][w] = acc[0][w] + p[w];
    }
    for (int l = 1; l < P6O_LEVELS; ++l)
        for (int w = 0; w < width; ++w) acc[0][w] = acc[0][w] + acc[l][w];
    for (int w = 0; w < width; ++w) acc_out[w] = acc[0][w];
}

/* row_sum over `size` items of `lanes` floats each (lanes = 8 for the vector part,
 * 1 for short rows).  out[lanes]. */
static void p6o_row_sum(const float* x, int lanes, int64_t size, float* out) {
    const int64_t size_ilp = size / P6O_ILP;
    float part[P6O_V * P6O_ILP];
    p6o_cascade_rows(x, (int64_t)lanes * P6O_ILP, lanes * P6O_ILP, size_ilp, part);
    for (int64_t i = size_ilp * P6O_ILP; i < size; ++i)
        for (int w = 0; w < lanes; ++w) part[w] = part[w] + x[i * lanes + w];
    for (int k = 1; k < P6O_ILP; ++k)
        for (int w = 0; w < lanes; ++w) part[w] = part[w] + part[k * lanes + w];
    for (int w = 0; w < lanes; ++w) out[w] = part[w];
}

P6O_API float p6o_aten_sum_f32(const float* x, int64_t n) {
    if (n <= 0) return 0.0f;
    if (n < P6O_V) {
        float r;
        p6o_row_sum(x, 1, n, &r);
        return 0.0f + r;
    }
    const int64_t nvec = n / P6O_V;
    float lanes[P6O_V];
    p6o_row_sum(x, P6O_V, nvec, lanes);
    float acc = 0.0f;
    for (int64_t k = nvec * P6O_V; k < n; ++k) acc = acc + x[k];
    for (int k = 0; k < P6O_V; ++k) acc = acc + lanes[k];
    return 0.0f + acc;
}

P6O_API float p6o_aten_mean_f32(const float* x, int64_t n) {
    return p6o_aten_sum_f32(x, n) / (float)n;
}

/* ------------------------------------------------------------------------------------
 * Quaternion [x,y,z,w] -> row-major 3x3, no normalisation.
 * Restates ADDLoss._quat_to_mat, models/add_loss.py:203-215: products first, then
 * "1 - 2*a - 2*b" evaluated left to right, every op rounded on its own.
 * ---------------------------------------------------------------------------------- */
P6O_API void p6o_quat_to_mat(const float* q, float* R) {
    const float x = q[0], y = q[1], z = q[2], w = q[3];
    const float x2 = x * x, y2 = y * y, z2 = z * z;
    const float xy = x * y, xz = x * z, yz = y * z;
    const float wx = w * x, wy = w * y, wz = w * z;
    R[0] = (1.0f - 2.0f * y2) - 2.0f * z2;
    R[1] = 2.0f * xy - 2.0f * wz;
    R[2] = 2.0f * xz + 2.0f * wy;
    R[3] = 2.0f * xy + 2.0f * wz;
    R[4] = (1.0f - 2.0f * x2) - 2.0f * z2;
    R[5] = 2.0f * yz - 2.0f * wx;
    R[6] = 2.0f * xz - 2.0f * wy;
    R[7] = 2.0f * yz + 2.0f * wx;
    R[8] = (1.0f - 2.0f * x2) - 2.0f * y2;
}

/* cloud[i] = mesh[i] . R^T + t  (models/add_loss.py:178-179 and :132-133).
 * torch.mm's float32 rounding depends on the row count n of the [n,3] x [3,3] product
 * (measured, torch 2.11.0 + MKL 2024.2): n >= 11 takes the k-sequential FMA chain;
 * tiny products take unfused kernels: n == 1 -> (p1*r1 + p2*r2) + p0*r0,
 * 2 <= n <= 10 -> (p0*r0 + p2*r2) + p1*r1.
 * The loss form (models/add_loss.py:132-133) goes through torch.matmul on a [1,n,3] x [B,3,3]
 * batch instead (measured, same build): ATen's naive bmm kernel for 3*n*3 < 400, i.e. n <= 44,
 * which accumulates left to right without fusing, and the FMA chain above that (except where MKL's
 * batched sgemm takes another path: observed for exactly 2 samples of a 97..106- or 200-point mesh).
 * Callers select that rule by passing n = P6O_BMM(n). */
#define P6O_BMM(n) ((n) <= 44 ? (int64_t)-1 : (int64_t)11)
static inline void p6o_xform_point(const float* m, const float* R, const float* t, int64_t n,
                                   float* o) {
    for (int c = 0; c < 3; ++c) {
        const float* r = R + 3 * c;
        float v;
        if (n >= 11) {
            v = m[0] * r[0];
            v = fmaf(m[1], r[1], v);
            v = fmaf(m[2], r[2], v);
        } else if (n < 0) {
            v = (m[0] * r[0] + m[1] * r[1]) + m[2] * r[2];
        } else if (n == 1) {
            v = (m[1] * r[1] + m[2] * r[2]) + m[0] * r[0];
        } else {
            v = (m[0] * r[0] + m[2] * r[2]) + m[1] * r[1];
        }
        o[c] = v + t[c];
    }
}

P6O_API void p6o_transform(const float* mesh, int64_t n, const float* q, const float* t, float* out) {
    float R[9];
    p6o_quat_to_mat(q, R);
    for (int64_t i = 0; i < n; ++i) p6o_xform_point(mesh + 3 * i, R, t, n, out + 3 * i);
}

static inline float p6o_sq3(float dx, float dy, float dz) {
    float s = dx * dx;
    s = fmaf(dy, dy, s);
    s = fmaf(dz, dz, s);
    return s;
}

/* NaN-propagating minimum, like torch.min. */
static inline float p6o_min_nan(float a, float b) {
    if (a != a) return a;
    if (b != b) return b;
    return b < a ? b : a;
}

/* ------------------------------------------------------------------------------------
 * One pose: ADD (models/add_loss.py:181-183), ADD-S (:185-190, pred-major: for each
 * *pred* point the nearest *gt* point).  scratch: 3 arrays of n floats x2 + n.
 * ---------------------------------------------------------------------------------- */
static void p6o_pose_distances(const float* mesh, int64_t n, const float* pq, const float* pt,
                               const float* gq, const float* gt, int want_adds, float* add_out,
                               float* adds_out, float* scratch, int bmm) {
    const int64_t rule = bmm ? P6O_BMM(n) : n;
    float Rp[9], Rg[9];
    p6o_quat_to_mat(pq, Rp);
    p6o_quat_to_mat(gq, Rg);
    float* px = scratch;          float* py = px + n; float* pz = py + n;
    float* gx = pz + n;           float* gy = gx + n; float* gz = gy + n;
    float* d = gz + n;
    for (int64_t i = 0; i < n; ++i) {
        float p[3], g[3];
        p6o_xform_point(mesh + 3 * i, Rp, pt, rule, p);
        p6o_xform_point(mesh + 3 * i, Rg, gt, rule, g);
        px[i] = p[0]; py[i] = p[1]; pz[i] = p[2];
        gx[i] = g[0]; gy[i] = g[1]; gz[i] = g[2];
        d[i] = sqrtf(p6o_sq3(p[0] - g[0], p[1] - g[1], p[2] - g[2]));
    }
    *add_out = p6o_aten_mean_f32(d, n);
    if (!want_adds) return;
    for (int64_t i = 0; i < n; ++i) {
        const float x = px[i], y = py[i], z = pz[i];
        float m = INFINITY;
        int saw_nan = 0;
        /* min over squared distances; sqrt is monotone and correctly rounded, so
         * sqrt(min s) == min sqrt(s) bit for bit. */
        for (int64_t j = 0; j < n; ++j) {
            const float s = p6o_sq3(x - gx[j], y - gy[j], z - gz[j]);
            saw_nan |= (s != s);
            m = s < m ? s : m;
        }
        d[i] = saw_nan ? NAN : sqrtf(m);
    }
    *adds_out = p6o_aten_mean_f32(d, n);
}

/* ------------------------------------------------------------------------------------
 * Batched evaluation = the loop body of ADDLoss.eval_metrics, models/add_loss.py:168-195.
 *   mesh_xyz   : all object meshes concatenated, row-major [sum N, 3]
 *   offsets/counts[n_slots] : first point / point count of object id s (count 0 = the
 *                id is not in self.points -> the pose is skipped, add_loss.py:171-172)
 *   diameters[n_slots] (metres, float64); threshold = 0.1 * diameter in float64 (:176)
 *   symmetric[n_slots] : 1 for ids in SYMMETRIC_OBJECT_IDS (:10,:193-194)
 * Outputs per pose: add, adds (float32, 0 when skipped), hit, valid (uint8).
 * want_adds bit 0 clear skips the N^2 part (adds untouched; symmetric ids then decide on ADD,
 * which the reference never does -- only used by the ADD-only kernel's tests); bit 1 set
 * transforms with torch.matmul's rounding (the loss form, ADDLoss.forward).
 * ---------------------------------------------------------------------------------- */
typedef struct {
    const float* mesh_xyz; const int32_t* offsets; const int32_t* counts;
    const double* diameters; const uint8_t* symmetric; int n_slots;
    const float* pq; const float* pt; const float* gq; const float* gt; const int64_t* obj;
    int64_t B; int want_adds; float* add; float* adds; uint8_t* hit; uint8_t* valid;
    int64_t max_n; int64_t* next; int failed;
} p6o_eval_job;

static void* p6o_eval_worker(void* arg) {
    p6o_eval_job* J = (p6o_eval_job*)arg;
    float* scratch = (float*)malloc(sizeof(float) * (size_t)(7 * (J->max_n > 0 ? J->max_n : 1)));
    if (!scratch) { J->failed = 1; return NULL; }
    for (;;) {
        /* dynamic schedule, one pose at a time (poses differ in N) */
        const int64_t b = __atomic_fetch_add(J->next, 1, __ATOMIC_RELAXED);
        if (b >= J->B) break;
        const int64_t oid = J->obj[b];
        if (oid < 0 || oid >= J->n_slots || J->counts[oid] <= 0) {
            J->add[b] = 0.0f;
            if (J->adds) J->adds[b] = 0.0f;
            J->hit[b] = 0;
            J->valid[b] = 0;
            continue;
        }
        const int do_s = (J->want_adds & 1) && J->adds != NULL;
        float a = 0.0f, as = 0.0f;
        p6o_pose_distances(J->mesh_xyz + 3 * (int64_t)J->offsets[oid], J->counts[oid], J->pq + 4 * b,
                           J->pt + 3 * b, J->gq + 4 * b, J->gt + 3 * b, do_s, &a, &as, scratch,
                           (J->want_adds & 2) != 0);
        J->add[b] = a;
        if (do_s) J->adds[b] = as;
        const double thr = 0.1 * J->diameters[oid];
        const float eff = (J->symmetric[oid] && do_s) ? as : a;
        J->hit[b] = ((double)eff < thr) ? 1 : 0;
        J->valid[b] = 1;
    }
    free(scratch);
    return NULL;
}

P6O_API int p6o_add_eval(const float* mesh_xyz, const int32_t* offsets, const int32_t* counts,
                         const double* diameters, const uint8_t* symmetric, int n_slots,
                         const float* pq, const float* pt, const float* gq, const float* gt,
                         const int64_t* obj, int64_t B, int want_adds, float* add, float* adds,
                         uint8_t* hit, uint8_t* valid, int n_threads) {
    int64_t max_n = 0;
    for (int s = 0; s < n_slots; ++s) if (counts[s] > max_n) max_n = counts[s];
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    if ((int64_t)n_threads > B) n_threads = B > 0 ? (int)B : 1;
    int64_t next = 0;
    p6o_eval_job jobs[256];
    pthread_t tid[256];
    for (int t = 0; t < n_threads; ++t) {
        p6o_eval_job J = {mesh_xyz, offsets, counts, diameters, symmetric, n_slots, pq, pt, gq, gt,
                          obj, B, want_adds, add, adds, hit, valid, max_n, &next, 0};
        jobs[t] = J;
    }
    int spawned = 0;
    for (int t = 1; t < n_threads; ++t) {
        if (pthread_create(&tid[t], NULL, p6o_eval_worker, &jobs[t]) != 0) break;
        spawned = t;
    }
    p6o_eval_worker(&jobs[0]);
    int failed = jobs[0].failed;
    for (int t = 1; t <= spawned; ++t) { pthread_join(tid[t], NULL); failed |= jobs[t].failed; }
    return failed ? -1 : 0;
}

/* ------------------------------------------------------------------------------------
 * Gradient of ADDLoss.forward (models/add_loss.py:101-150) w.r.t. pred_r / pred_t, i.e.
 * what autograd derives through matmul, norm, min and mean:
 *   loss = (1/count) sum_b mean_i d_bi,  dL/dp_i = (1/(count*N)) (p_i - g*) / d  (0 if d == 0)
 *   dL/dt = sum_i dL/dp_i,  dL/dR = sum_i dL/dp_i m_i^T,  dL/dq = J(_quat_to_mat)^T dL/dR.
 * Forward quantities in float32 (same rounding as the loss), accumulation in float64.
 * ---------------------------------------------------------------------------------- */
P6O_API int p6o_add_backward(const float* mesh_xyz, const int32_t* offsets, const int32_t* counts,
                             const uint8_t* symmetric, int n_slots, const float* pq, const float* pt,
                             const float* gq, const float* gt, const int64_t* obj, int64_t B,
                             double grad_out, float* grad_q, float* grad_t) {
    int64_t count = 0, max_n = 1;
    for (int64_t b = 0; b < B; ++b)
        if (obj[b] >= 0 && obj[b] < n_slots && counts[obj[b]] > 0) ++count;
    for (int s = 0; s < n_slots; ++s) if (counts[s] > max_n) max_n = counts[s];
    float* g = (float*)malloc(sizeof(float) * 3 * (size_t)max_n);
    if (!g) return -1;
    for (int64_t b = 0; b < B; ++b) {
        for (int k = 0; k < 4; ++k) grad_q[4 * b + k] = 0.0f;
        for (int k = 0; k < 3; ++k) grad_t[3 * b + k] = 0.0f;
        const int64_t oid = obj[b];
        if (oid < 0 || oid >= n_slots || counts[oid] <= 0) continue;
        const int64_t n = counts[oid];
        const float* mesh = mesh_xyz + 3 * (int64_t)offsets[oid];
        float Rp[9], Rg[9];
        p6o_quat_to_mat(pq + 4 * b, Rp);
        p6o_quat_to_mat(gq + 4 * b, Rg);
        for (int64_t i = 0; i < n; ++i) p6o_xform_point(mesh + 3 * i, Rg, gt + 3 * b, P6O_BMM(n), g + 3 * i);
        double T[3] = {0, 0, 0}, R[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int64_t i = 0; i < n; ++i) {
            float p[3];
            p6o_xform_point(mesh + 3 * i, Rp, pt + 3 * b, P6O_BMM(n), p);
            int64_t js = i;
            if (symmetric[oid]) {
                /* torch.norm(...).min(dim=2): the first j with the smallest ROOTED distance.  Two
                 * different squares can have the same sqrtf; the earlier point wins then.  best_r
                 * is always sqrtf(best), so the root is only taken when the square improves. */
                float best = INFINITY, best_r = INFINITY;
                js = 0;
                for (int64_t j = 0; j < n; ++j) {
                    const float sv = p6o_sq3(p[0] - g[3 * j], p[1] - g[3 * j + 1], p[2] - g[3 * j + 2]);
                    if (sv != sv) { js = j; break; }
                    if (sv < best) {
                        best = sv;
                        const float r = sqrtf(sv);
                        if (r < best_r) { best_r = r; js = j; }
                    }
                }
            }
            const float d3[3] = {p[0] - g[3 * js], p[1] - g[3 * js + 1], p[2] - g[3 * js + 2]};
            const float d = sqrtf(p6o_sq3(d3[0], d3[1], d3[2]));
            if (d == 0.0f) continue;
            for (int r = 0; r < 3; ++r) {
                const double G = (double)(d3[r] / d);
                T[r] += G;
                for (int c = 0; c < 3; ++c) R[3 * r + c] += G * (double)mesh[3 * i + c];
            }
        }
        const double scale = grad_out / (double)count / (double)n;
        const double x = pq[4 * b], y = pq[4 * b + 1], z = pq[4 * b + 2], w = pq[4 * b + 3];
        const double gx = 2*y*R[1] + 2*z*R[2] + 2*y*R[3] - 4*x*R[4] - 2*w*R[5] + 2*z*R[6] + 2*w*R[7] - 4*x*R[8];
        const double gy = -4*y*R[0] + 2*x*R[1] + 2*w*R[2] + 2*x*R[3] + 2*z*R[5] - 2*w*R[6] + 2*z*R[7] - 4*y*R[8];
        const double gz = -4*z*R[0] - 2*w*R[1] + 2*x*R[2] + 2*w*R[3] - 4*z*R[4] + 2*y*R[5] + 2*x*R[6] + 2*y*R[7];
        const double gw = -2*z*R[1] + 2*y*R[2] + 2*z*R[3] - 2*x*R[5] - 2*y*R[6] + 2*x*R[7];
        grad_q[4 * b + 0] = (float)(scale * gx);
        grad_q[4 * b + 1] = (float)(scale * gy);
        grad_q[4 * b + 2] = (float)(scale * gz);
        grad_q[4 * b + 3] = (float)(scale * gw);
        for (int k = 0; k < 3; ++k) grad_t[3 * b + k] = (float)(scale * T[k]);
    }
    free(g);
    return 0;
}

/* ------------------------------------------------------------------------------------
 * PoseLoss (models/pose_loss.py:19-61).  mode 0 = 'geodesic', 1 = quaternion L1.
 * Forward mirrors the float32 op order; per-row terms are returned so the caller can
 * check them independently of the mean.  Gradients (w.r.t. pred_rot, pred_trans, for
 * upstream grad 1) are the analytic derivatives of that graph with PyTorch's
 * sub-gradient conventions: norm'(0) = 0, clamp_min passes grad when x >= min,
 * sign(0) = 0, minimum() splits ties in halves, where() routes no grad to its mask.
 * They are evaluated in float64 from the float32 forward intermediates and rounded once.
 * ---------------------------------------------------------------------------------- */
/* torch.norm / F.normalize over a [B,4] row: measured to be the UNFUSED sequential sum
 * ((x0^2 + x1^2) + x2^2) + x3^2 (unlike the 3-component rows, which take the FMA chain). */
static inline float p6o_norm4(const float* v) {
    float s = v[0] * v[0];
    s = s + v[1] * v[1];
    s = s + v[2] * v[2];
    s = s + v[3] * v[3];
    return sqrtf(s);
}

P6O_API int p6o_pose_loss(const float* pq, const float* pt, const float* gq, const float* gt,
                          int64_t B, float rot_weight, float trans_weight, int mode,
                          float* loss_out, float* rot_out, float* trans_out,
                          float* row_rot /* [B] nullable */, float* grad_q /* [B,4] nullable */,
                          float* grad_t /* [B,3] nullable */) {
    if (B <= 0) return -1;
    float* rows = (float*)malloc(sizeof(float) * (size_t)B);
    float* absd = (float*)malloc(sizeof(float) * (size_t)(3 * B));
    if (!rows || !absd) { free(rows); free(absd); return -1; }
    const double inv_b = 1.0 / (double)B;
    for (int64_t b = 0; b < B; ++b) {
        const float* a = pq + 4 * b;
        const float* c = gq + 4 * b;
        const float na_raw = p6o_norm4(a), nc_raw = p6o_norm4(c);
        const float na = na_raw > 1e-12f ? na_raw : 1e-12f; /* clamp_min(eps) */
        const float nc = nc_raw > 1e-12f ? nc_raw : 1e-12f;
        float u[4], v[4];
        for (int k = 0; k < 4; ++k) { u[k] = a[k] / na; v[k] = c[k] / nc; }
        double gu[4] = {0, 0, 0, 0};
        if (mode == 0) {
            /* torch.sum(q1*q2, dim=1): sequential over 4 products, each product rounded */
            float dot = u[0] * v[0];
            dot = dot + u[1] * v[1];
            dot = dot + u[2] * v[2];
            dot = dot + u[3] * v[3];
            if (dot < 0.0f) for (int k = 0; k < 4; ++k) v[k] = -v[k];
            float d[4], s[4];
            for (int k = 0; k < 4; ++k) { d[k] = u[k] - v[k]; s[k] = u[k] + v[k]; }
            const float dn = p6o_norm4(d), sn = p6o_norm4(s);
            rows[b] = 2.0f * atan2f(dn, sn);
            const double den = (double)dn * dn + (double)sn * sn;
            const double dA_ddn = den > 0 ? 2.0 * sn / den : 0.0;
            const double dA_dsn = den > 0 ? -2.0 * dn / den : 0.0;
            for (int k = 0; k < 4; ++k) {
                double g = 0.0;
                if (dn > 0.0f) g += dA_ddn * (double)d[k] / dn;
                if (sn > 0.0f) g += dA_dsn * (double)s[k] / sn;
                gu[k] = g;
            }
        } else {
            float dp = 0.0f, dm = 0.0f;
            float ap[4], am[4];
            for (int k = 0; k < 4; ++k) { ap[k] = u[k] - v[k]; am[k] = u[k] + v[k]; }
            dp = fabsf(ap[0]); dp = dp + fabsf(ap[1]); dp = dp + fabsf(ap[2]); dp = dp + fabsf(ap[3]);
            dm = fabsf(am[0]); dm = dm + fabsf(am[1]); dm = dm + fabsf(am[2]); dm = dm + fabsf(am[3]);
            rows[b] = dp < dm ? dp : dm;
            if (dp != dp || dm != dm) rows[b] = NAN;
            const double wp = dp < dm ? 1.0 : (dp == dm ? 0.5 : 0.0);
            const double wm = dm < dp ? 1.0 : (dp == dm ? 0.5 : 0.0);
            for (int k = 0; k < 4; ++k) {
                const double sp = (ap[k] > 0) - (ap[k] < 0);
                const double sm = (am[k] > 0) - (am[k] < 0);
                gu[k] = wp * sp + wm * sm;
            }
        }
        if (row_rot) row_rot[b] = rows[b];
        if (grad_q) {
            double gdotu = 0.0;
            for (int k = 0; k < 4; ++k) gdotu += gu[k] * (double)u[k];
            for (int k = 0; k < 4; ++k) {
                double g;
                if (na_raw >= 1e-12f && na_raw > 0.0f) g = (gu[k] - (double)u[k] * gdotu) / (double)na;
                else g = gu[k] / (double)na;
                grad_q[4 * b + k] = (float)((double)rot_weight * inv_b * g);
            }
        }
        for (int k = 0; k < 3; ++k) {
            const float df = pt[3 * b + k] - gt[3 * b + k];
            absd[3 * b + k] = fabsf(df);
            if (grad_t) {
                /* ATen's mean backward: float32(weight) / float32(numel), then times sign */
                const float sg = (float)((df > 0) - (df < 0));
                grad_t[3 * b + k] = sg * (trans_weight / (float)(3 * B));
            }
        }
    }
    const float rot = p6o_aten_mean_f32(rows, B);
    const float tr = p6o_aten_mean_f32(absd, 3 * B);
    if (rot_out) *rot_out = rot;
    if (trans_out) *trans_out = tr;
    *loss_out = rot_weight * rot + trans_weight * tr;
    free(rows);
    free(absd);
    return 0;
}

/* ------------------------------------------------------------------------------------
 * Pinhole XY from bbox centre + predicted Z
 * (PoseNetRGBGeometric._compute_pinhole_translation, models/pose_net_rgb_geometric.py:93-109).
 * K row-major 3x3, shared (k_batched = 0) or per row.  out [B,3].
 * grad_z (nullable) = d(sum(out * grad_out))/dz for a given grad_out [B,3].
 * ---------------------------------------------------------------------------------- */
P6O_API void p6o_pinhole(const float* z, const float* uv, const float* K, int k_batched, int64_t B,
                         float* out, const float* grad_out, float* grad_z) {
    for (int64_t b = 0; b < B; ++b) {
        const float* k = K + (k_batched ? 9 * b : 0);
        const float fx = k[0], fy = k[4], cx = k[2], cy = k[5];
        const float du = uv[2 * b] - cx, dv = uv[2 * b + 1] - cy;
        if (out) {
            out[3 * b + 0] = (du * z[b]) / fx;
            out[3 * b + 1] = (dv * z[b]) / fy;
            out[3 * b + 2] = z[b];
        }
        if (grad_out && grad_z) {
            /* autograd order: d/dz [(du*z)/fx] = (g/fx)*du */
            const float gx = grad_out[3 * b] / fx, gy = grad_out[3 * b + 1] / fy;
            grad_z[b] = (gx * du + gy * dv) + grad_out[3 * b + 2];
        }
    }
}

/* ------------------------------------------------------------------------------------
 * Depth sample + back-projection
 * (PoseNetRGBDGeometric._compute_pinhole_translation, models/pose_net_rgbd_geometric.py:56-85).
 * depth [B,H,W] metres; the centre is clamped to [0, clamp_hi] as float (the reference
 * hard-codes 223), truncated toward zero for the index, index clamped again; NaN centre
 * -> clamp keeps NaN in torch, .long() of NaN is INT64_MIN on x86 -> index 0.
 * ---------------------------------------------------------------------------------- */
static inline float p6o_clampf(float x, float lo, float hi) {
    /* torch.clamp: NaN stays NaN; min(max(x,lo),hi) */
    if (x != x) return x;
    return x < lo ? lo : (x > hi ? hi : x);
}

P6O_API void p6o_depth_backproject(const float* depth, int H, int W, const float* uv, const float* K,
                                   int k_batched, int64_t B, float clamp_hi, float* out) {
    for (int64_t b = 0; b < B; ++b) {
        const float* k = K + (k_batched ? 9 * b : 0);
        const float fx = k[0], fy = k[4], cx = k[2], cy = k[5];
        const float u = p6o_clampf(uv[2 * b], 0.0f, clamp_hi);
        const float v = p6o_clampf(uv[2 * b + 1], 0.0f, clamp_hi);
        int64_t ui = (u != u) ? INT64_MIN : (int64_t)u;
        int64_t vi = (v != v) ? INT64_MIN : (int64_t)v;
        const int64_t hi = (int64_t)clamp_hi;
        ui = ui < 0 ? 0 : (ui > hi ? hi : ui);
        vi = vi < 0 ? 0 : (vi > hi ? hi : vi);
        float z = depth[((int64_t)b * H + vi) * W + ui];
        z = (z > 0.01f) ? z : 0.5f;
        z = p6o_clampf(z, 0.1f, 2.0f);
        out[3 * b + 0] = ((u - cx) * z) / fx;
        out[3 * b + 1] = ((v - cy) * z) / fy;
        out[3 * b + 2] = z;
    }
}

P6O_API int p6o_max_threads(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}

P6O_API int p6o_version(void) { return 1; }
