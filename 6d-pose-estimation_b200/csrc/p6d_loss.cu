// p6d_loss.cu -- PoseLoss forward + backward in one launch (sm_100a).
//
// Replaces ~20 forward + ~20 autograd-backward eager launches of
// PoseLoss.forward (reference models/pose_loss.py:19-61) on ~2 KB of data.
// Per row: normalise both quaternions (x / max(|x|, 1e-12), F.normalize), resolve the
// double cover, 2*atan2(|q1-q2|, |q1+q2|) or the quaternion-L1 distance, |t_p - t_g|;
// gradients w.r.t. the prediction are emitted by the same threads (PyTorch's
// sub-gradient conventions, see oracle/pose_oracle.c p6o_pose_loss).
//
// Two shapes of the same kernel:
//   B <= SMALL_B : one CTA; per-row terms go to shared memory and one warp reduces them
//                  in ATen's summation order, so the L1 rotation term and the translation
//                  term equal the CPU reference bit for bit (atan2f differs by <= 2 ulp);
//   B >  SMALL_B : grid-stride rows, float64 block partials + atomics, last block
//                  finalises (HBM-bound shape used for the GB/s measurement).  The sum order is
//                  not ATen's there, so nothing is bit-exact by construction (bar: 1e-5); the
//                  geodesic mode therefore runs the FAST row: reciprocal square roots and
//                  multiplications (MUFU.RSQ / MUFU.RCP, <= 2 ulp each) instead of 4 IEEE square
//                  roots and 13 IEEE divisions per row, which halves the instruction count and
//                  lets the loads of the next rows overlap the arithmetic.
#include "p6d_common.cuh"

namespace p6d {

constexpr int LOSS_T = 256;
constexpr int SMALL_B = 2048;

struct Workspace {
    double rot_sum;
    double trans_sum;
    unsigned long long blocks_done;
    unsigned long long pad;
};

struct RowOut {
    float rot;     // per-row rotation term
    float ad[3];   // |t_p - t_g|
};

// torch.norm over a [B,4] row is the unfused sequential sum of squares (oracle: p6o_norm4)
__device__ __forceinline__ float norm4(const float* v) {
    float s = __fmul_rn(v[0], v[0]);
    s = __fadd_rn(s, __fmul_rn(v[1], v[1]));
    s = __fadd_rn(s, __fmul_rn(v[2], v[2]));
    s = __fadd_rn(s, __fmul_rn(v[3], v[3]));
    return __fsqrt_rn(s);
}

__device__ __forceinline__ float sumsq4(const float* v) {
    return fmaf(v[3], v[3], fmaf(v[2], v[2], fmaf(v[1], v[1], v[0] * v[0])));
}

// pt_row / gt_row / grad_t_row point at the 3 floats of row b.
// FAST (large batches, geodesic mode only): see the header comment.
template <bool FAST>
__device__ __forceinline__ RowOut loss_row(const float4 a4, const float* pt_row, const float4 c4, const float* gt_row,
                                           int64_t B, float wr, float wt, int mode,
                                           float* __restrict__ grad_q_row, float* grad_t_row) {
    RowOut o;
    const float a[4] = {a4.x, a4.y, a4.z, a4.w};
    const float c[4] = {c4.x, c4.y, c4.z, c4.w};
    float u[4], v[4];
    float na = 1.0f, inv_na = 1.0f;      // max(|a|, 1e-12) (exact row) or its reciprocal (FAST row)
    bool a_has_norm_grad;
    if (FAST) {
        const float sa = sumsq4(a), sc = sumsq4(c);
        // |x| >= 1e-12  <=>  |x|^2 >= 1e-24 (a normal float32)
        inv_na = sa >= 1e-24f ? rsqrtf(sa) : 1e12f;
        const float inv_nc = sc >= 1e-24f ? rsqrtf(sc) : 1e12f;
        a_has_norm_grad = sa >= 1e-24f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            u[k] = a[k] * inv_na;
            v[k] = c[k] * inv_nc;
        }
    } else {
        const float na_raw = norm4(a), nc_raw = norm4(c);
        na = na_raw > 1e-12f ? na_raw : 1e-12f;
        const float nc = nc_raw > 1e-12f ? nc_raw : 1e-12f;
        // clamp_min passes the gradient of the norm only when |a| >= eps; norm'(0) = 0
        a_has_norm_grad = na_raw >= 1e-12f && na_raw > 0.0f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            u[k] = __fdiv_rn(a[k], na);
            v[k] = __fdiv_rn(c[k], nc);
        }
    }
    // Gradient math runs in float32: the two terms of gu are orthogonal (u-v is
    // perpendicular to u+v) and gu is already tangent to the unit sphere, so nothing cancels;
    // measured error vs the float64 oracle ~1e-7 of the row maximum (bar: 1e-5).
    float gu[4];
    if (mode == 0) {
        float dot = __fmul_rn(u[0], v[0]);
        dot = __fadd_rn(dot, __fmul_rn(u[1], v[1]));
        dot = __fadd_rn(dot, __fmul_rn(u[2], v[2]));
        dot = __fadd_rn(dot, __fmul_rn(u[3], v[3]));
        if (dot < 0.0f) {
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = -v[k];
        }
        float d[4], s[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            d[k] = __fsub_rn(u[k], v[k]);
            s[k] = __fadd_rn(u[k], v[k]);
        }
        float dn, sn, cd, cs;
        if (FAST) {
            const float sd = sumsq4(d), ss = sumsq4(s);
            // Two decisions of the exact row are discontinuous in u and v: the sign of dot (it negates
            // the gradient) and dn == 0 (zero gradient instead of a unit vector along rounding noise).
            // A FAST u or v differs from the exact one by <= ~10 ulp per component (RSQ 2 ulp, sums and
            // products), so the FAST dot is within ~28 * 2^-24 < 2^-19 of the exact dot, and a FAST
            // |d|^2 is below (20 * 2^-24)^2 < 2^-39 where the exact d is 0.  Near either edge (margins
            // >= 8x) the row is recomputed exactly; uniformly random pairs land there with probability ~1e-5.
            if (fabsf(dot) < 0x1p-16f || sd < 0x1p-30f)
                return loss_row<false>(a4, pt_row, c4, gt_row, B, wr, wt, mode, grad_q_row, grad_t_row);
            const float rd = sd > 0.0f ? rsqrtf(sd) : 0.0f, rs = ss > 0.0f ? rsqrtf(ss) : 0.0f;
            dn = sd * rd;
            sn = ss * rs;
            const float den = sd + ss;
            const float inv_den = den > 0.0f ? __fdividef(2.0f, den) : 0.0f;
            cd = sn * inv_den * rd;
            cs = -(dn * inv_den * rs);
        } else {
            dn = norm4(d);
            sn = norm4(s);
            const float den = fmaf(dn, dn, sn * sn);
            const float inv_den = den > 0.0f ? __fdiv_rn(2.0f, den) : 0.0f;
            // d(angle)/d(dn) * 1/dn  and  d(angle)/d(sn) * 1/sn  (norm'(0) = 0)
            cd = dn > 0.0f ? __fdiv_rn(sn * inv_den, dn) : 0.0f;
            cs = sn > 0.0f ? -__fdiv_rn(dn * inv_den, sn) : 0.0f;
        }
        o.rot = __fmul_rn(2.0f, atan2f(dn, sn));
#pragma unroll
        for (int k = 0; k < 4; ++k) gu[k] = fmaf(cd, d[k], cs * s[k]);
    } else {
        float ap[4], am[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            ap[k] = __fsub_rn(u[k], v[k]);
            am[k] = __fadd_rn(u[k], v[k]);
        }
        float dp = fabsf(ap[0]), dm = fabsf(am[0]);
#pragma unroll
        for (int k = 1; k < 4; ++k) {
            dp = __fadd_rn(dp, fabsf(ap[k]));
            dm = __fadd_rn(dm, fabsf(am[k]));
        }
        o.rot = min_nan(dp, dm);
        const float wp = dp < dm ? 1.0f : (dp == dm ? 0.5f : 0.0f);
        const float wm = dm < dp ? 1.0f : (dp == dm ? 0.5f : 0.0f);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float sp = (float)((ap[k] > 0.0f) - (ap[k] < 0.0f));
            const float sm = (float)((am[k] > 0.0f) - (am[k] < 0.0f));
            gu[k] = wp * sp + wm * sm;
        }
    }
    if (grad_q_row) {
        float gdotu = 0.0f;
#pragma unroll
        for (int k = 0; k < 4; ++k) gdotu = fmaf(gu[k], u[k], gdotu);
        const float proj = a_has_norm_grad ? gdotu : 0.0f;
        const float scale = FAST ? __fdiv_rn(wr, (float)B) * inv_na : __fdiv_rn(__fdiv_rn(wr, (float)B), na);
        float4 g4;
        float* gp = reinterpret_cast<float*>(&g4);
#pragma unroll
        for (int k = 0; k < 4; ++k) gp[k] = scale * fmaf(-u[k], proj, gu[k]);
        *reinterpret_cast<float4*>(grad_q_row) = g4;
    }
    // ATen's mean backward divides in float32 by float32(numel), which is inexact once 3B > 2^24
    const float tscale = __fdiv_rn(wt, (float)(3 * B));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float df = __fsub_rn(pt_row[k], gt_row[k]);
        o.ad[k] = fabsf(df);
        if (grad_t_row) grad_t_row[k] = df > 0.0f ? tscale : (df < 0.0f ? -tscale : 0.0f);
    }
    return o;
}

// Optional fused geometric translation (kernel d1 inside kernel c): pred_trans is not read
// from memory but computed from (z, bbox centre, K) exactly like p6d_pinhole_fwd, and the
// gradient w.r.t. z is produced exactly like p6d_pinhole_bwd applied to grad_trans.
struct Geo {
    const float* z;      // [B]   (nullptr = plain PoseLoss on pred_trans)
    const float* uv;     // [B,2]
    const float* K;      // [3,3] or [B,3,3]
    int k_batched;
    float* grad_z;       // [B] nullable
    float* trans_out;    // [B,3] nullable: the translation the reference's model would return
};

template <bool FAST, bool GEO>
__device__ __forceinline__ RowOut loss_row_any(const float* __restrict__ pq, const float* __restrict__ pt,
                                               const float* __restrict__ gq, const float* __restrict__ gt,
                                               int64_t b, int64_t B, float wr, float wt, int mode,
                                               float* __restrict__ grad_q, float* __restrict__ grad_t,
                                               const Geo& geo) {
    const float4 a4 = *reinterpret_cast<const float4*>(pq + 4 * b);
    const float4 c4 = *reinterpret_cast<const float4*>(gq + 4 * b);
    float* gq_row = grad_q ? grad_q + 4 * b : nullptr;
    if (!GEO) return loss_row<FAST>(a4, pt + 3 * b, c4, gt + 3 * b, B, wr, wt, mode, gq_row,
                                    grad_t ? grad_t + 3 * b : nullptr);
    const float* k = geo.K + (geo.k_batched ? 9 * b : 0);
    const float fx = __ldg(k + 0), cx = __ldg(k + 2), fy = __ldg(k + 4), cy = __ldg(k + 5);
    const float2 c = *reinterpret_cast<const float2*>(geo.uv + 2 * b);
    const float zz = geo.z[b];
    const float du = __fsub_rn(c.x, cx), dv = __fsub_rn(c.y, cy);
    float t3[3] = {__fdiv_rn(__fmul_rn(du, zz), fx), __fdiv_rn(__fmul_rn(dv, zz), fy), zz};
    float g3[3] = {0.0f, 0.0f, 0.0f};
    const RowOut o = loss_row<FAST>(a4, t3, c4, gt + 3 * b, B, wr, wt, mode, gq_row, geo.grad_z ? g3 : nullptr);
    if (geo.trans_out) {
        geo.trans_out[3 * b + 0] = t3[0];
        geo.trans_out[3 * b + 1] = t3[1];
        geo.trans_out[3 * b + 2] = t3[2];
    }
    if (geo.grad_z) {
        const float gx = __fmul_rn(__fdiv_rn(g3[0], fx), du);
        const float gy = __fmul_rn(__fdiv_rn(g3[1], fy), dv);
        geo.grad_z[b] = __fadd_rn(__fadd_rn(gx, gy), g3[2]);
    }
    return o;
}

__device__ __forceinline__ void finish(float rot, float tr, float wr, float wt, float* out) {
    out[0] = __fadd_rn(__fmul_rn(wr, rot), __fmul_rn(wt, tr));
    out[1] = rot;
    out[2] = tr;
}

// B <= SMALL_B: single CTA, ATen-ordered means
template <bool GEO>
__global__ void __launch_bounds__(LOSS_T) pose_loss_small_kernel(const float* pq, const float* pt, const float* gq,
                                                                 const float* gt, int B, float wr, float wt,
                                                                 int mode, float* out, float* grad_q,
                                                                 float* grad_t, Geo geo) {
    __shared__ float s_rot[SMALL_B];
    __shared__ float s_ad[3 * SMALL_B];
    for (int b = threadIdx.x; b < B; b += LOSS_T) {
        const RowOut o = loss_row_any<false, GEO>(pq, pt, gq, gt, b, B, wr, wt, mode, grad_q, grad_t, geo);
        s_rot[b] = o.rot;
        s_ad[3 * b] = o.ad[0];
        s_ad[3 * b + 1] = o.ad[1];
        s_ad[3 * b + 2] = o.ad[2];
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        const float rot = aten_mean_warp([&](int e) { return s_rot[e]; }, B, lane);
        const float tr = aten_mean_warp([&](int e) { return s_ad[e]; }, 3 * B, lane);
        if (lane == 0) finish(rot, tr, wr, wt, out);
    }
}

// B > SMALL_B: grid-stride, float64 partial sums, last block finalises.
// Measured alternatives at 4 M rows (all slower than this shape, 91-94 us): prefetch.global.L1 of the
// thread's next row (101 us), two rows per thread and trip (120 us, 80 registers), 6 CTAs per SM at
// 40 registers (102 us, spills), shared-memory tile staging of the [B,3] rows (100 us).
#ifndef P6D_LOSS_MINB
#define P6D_LOSS_MINB 4     // CTAs per SM the register budget is sized for
#endif
template <bool FAST, bool GEO>
__global__ void __launch_bounds__(LOSS_T, P6D_LOSS_MINB) pose_loss_large_kernel(const float* pq, const float* pt, const float* gq,
                                                                 const float* gt, int64_t B, float wr, float wt,
                                                                 int mode, float* out, float* grad_q,
                                                                 float* grad_t, Workspace* ws, Geo geo) {
    double rs = 0.0, ts = 0.0;
    // (prefetching the next row of the thread with prefetch.global.L1 was tried: 10 % slower)
    for (int64_t b = (int64_t)blockIdx.x * LOSS_T + threadIdx.x; b < B; b += (int64_t)gridDim.x * LOSS_T) {
        const RowOut o = loss_row_any<FAST, GEO>(pq, pt, gq, gt, b, B, wr, wt, mode, grad_q, grad_t, geo);
        rs += (double)o.rot;
        ts += ((double)o.ad[0] + (double)o.ad[1]) + (double)o.ad[2];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        rs += __shfl_xor_sync(0xffffffffu, rs, o);
        ts += __shfl_xor_sync(0xffffffffu, ts, o);
    }
    __shared__ double s_r[LOSS_T / 32], s_t[LOSS_T / 32];
    __shared__ bool s_last;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_r[w] = rs; s_t[w] = ts; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0, t = 0.0;
        for (int i = 0; i < LOSS_T / 32; ++i) { r += s_r[i]; t += s_t[i]; }
        atomicAdd(&ws->rot_sum, r);
        atomicAdd(&ws->trans_sum, t);
        __threadfence();
        const unsigned long long done = atomicAdd(&ws->blocks_done, 1ull);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        const double r = atomicAdd(&ws->rot_sum, 0.0), t = atomicAdd(&ws->trans_sum, 0.0);
        finish((float)(r / (double)B), (float)(t / (3.0 * (double)B)), wr, wt, out);
        ws->rot_sum = 0.0;  // leave the workspace zeroed for the next call
        ws->trans_sum = 0.0;
        ws->blocks_done = 0ull;
    }
}

// B > SMALL_B, plain PoseLoss, 16-byte aligned inputs: the same rows STREAMED through shared memory.
// The grid-stride kernel above has at most one row per thread in flight (56 B x 1,024 threads = 57 KB
// per SM), which is less than HBM latency x bandwidth asks for (ncu: stall "long scoreboard" 10 warps
// per issue cycle, DRAM 54 % busy).  Here one thread per CTA issues TMA bulk copies
// (cp.async.bulk, SASS UBLKCP) of whole 256-row tiles -- [256,4] + [256,4] + [256,3] + [256,3] floats =
// 14 KB -- into a ring of STREAM_STAGES stages, each with its own mbarrier, so STAGES x 14 KB x CTAs/SM
// are in flight independent of what the warps are doing; the warps read their row out of shared memory
// (float4 / stride-3 scalars: conflict-free), hand the stage back with one __syncthreads and compute.
constexpr int STREAM_STAGES = 3;
constexpr int STREAM_TILE = LOSS_T;                                  // rows per tile = threads
constexpr int STREAM_STAGE_FLOATS = STREAM_TILE * (4 + 4 + 3 + 3);   // pq | gq | pt | gt
constexpr int STREAM_CTAS_PER_SM = 4;

template <bool FAST>
__global__ void __launch_bounds__(LOSS_T, STREAM_CTAS_PER_SM) pose_loss_stream_kernel(
    const float* __restrict__ pq, const float* __restrict__ pt, const float* __restrict__ gq,
    const float* __restrict__ gt, int64_t B, float wr, float wt, int mode, float* out, float* __restrict__ grad_q,
    float* __restrict__ grad_t, Workspace* ws) {
    extern __shared__ __align__(128) float s_ring[];
    __shared__ uint64_t s_full[STREAM_STAGES];
    const int tid = threadIdx.x;
    const int64_t n_tiles = B / STREAM_TILE;          // full tiles; the ragged tail is read directly
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STREAM_STAGES; ++s) mbar_init(&s_full[s], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](int64_t tile, int stage) {      // thread 0 only
        float* dst = s_ring + stage * STREAM_STAGE_FLOATS;
        const int64_t r0 = tile * STREAM_TILE;
        mbar_arrive_expect_tx(&s_full[stage], STREAM_STAGE_FLOATS * sizeof(float));
        tma_bulk_g2s(dst, pq + 4 * r0, STREAM_TILE * 16, &s_full[stage]);
        tma_bulk_g2s(dst + STREAM_TILE * 4, gq + 4 * r0, STREAM_TILE * 16, &s_full[stage]);
        tma_bulk_g2s(dst + STREAM_TILE * 8, pt + 3 * r0, STREAM_TILE * 12, &s_full[stage]);
        tma_bulk_g2s(dst + STREAM_TILE * 11, gt + 3 * r0, STREAM_TILE * 12, &s_full[stage]);
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STREAM_STAGES; ++s) {
            const int64_t tile = blockIdx.x + static_cast<int64_t>(s) * gridDim.x;
            if (tile < n_tiles) issue(tile, s);
        }
    }
    double rs = 0.0, ts = 0.0;
    int k = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
        const int stage = k % STREAM_STAGES;
        mbar_wait(&s_full[stage], (k / STREAM_STAGES) & 1);
        const float* src = s_ring + stage * STREAM_STAGE_FLOATS;
        const float4 a4 = reinterpret_cast<const float4*>(src)[tid];
        const float4 c4 = reinterpret_cast<const float4*>(src + STREAM_TILE * 4)[tid];
        float t3[3], g3[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            t3[c] = src[STREAM_TILE * 8 + 3 * tid + c];
            g3[c] = src[STREAM_TILE * 11 + 3 * tid + c];
        }
        __syncthreads();                              // every thread holds its row: the stage is free
        if (tid == 0) {
            const int64_t next = tile + static_cast<int64_t>(STREAM_STAGES) * gridDim.x;
            if (next < n_tiles) {
                fence_proxy_async();
                issue(next, stage);
            }
        }
        const int64_t b = tile * STREAM_TILE + tid;
        const RowOut o = loss_row<FAST>(a4, t3, c4, g3, B, wr, wt, mode, grad_q ? grad_q + 4 * b : nullptr,
                                        grad_t ? grad_t + 3 * b : nullptr);
        rs += (double)o.rot;
        ts += ((double)o.ad[0] + (double)o.ad[1]) + (double)o.ad[2];
    }
    // ragged tail (< 256 rows): CTA 0, straight from global memory
    if (blockIdx.x == 0) {
        const int64_t b = n_tiles * STREAM_TILE + tid;
        if (b < B) {
            Geo none{};
            const RowOut o = loss_row_any<FAST, false>(pq, pt, gq, gt, b, B, wr, wt, mode, grad_q, grad_t, none);
            rs += (double)o.rot;
            ts += ((double)o.ad[0] + (double)o.ad[1]) + (double)o.ad[2];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        rs += __shfl_xor_sync(0xffffffffu, rs, o);
        ts += __shfl_xor_sync(0xffffffffu, ts, o);
    }
    __shared__ double s_r[LOSS_T / 32], s_t[LOSS_T / 32];
    __shared__ bool s_last;
    const int w = tid >> 5, lane = tid & 31;
    if (lane == 0) { s_r[w] = rs; s_t[w] = ts; }
    __syncthreads();
    if (tid == 0) {
        double r = 0.0, t = 0.0;
        for (int i = 0; i < LOSS_T / 32; ++i) { r += s_r[i]; t += s_t[i]; }
        atomicAdd(&ws->rot_sum, r);
        atomicAdd(&ws->trans_sum, t);
        __threadfence();
        const unsigned long long done = atomicAdd(&ws->blocks_done, 1ull);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last && tid == 0) {
        __threadfence();
        const double r = atomicAdd(&ws->rot_sum, 0.0), t = atomicAdd(&ws->trans_sum, 0.0);
        finish((float)(r / (double)B), (float)(t / (3.0 * (double)B)), wr, wt, out);
        ws->rot_sum = 0.0;
        ws->trans_sum = 0.0;
        ws->blocks_done = 0ull;
    }
}

}  // namespace p6d

using namespace p6d;

extern "C" {

int64_t p6d_pose_loss_workspace_bytes(void) { return (int64_t)sizeof(Workspace); }

static int launch_pose_loss(const float* pq, const float* pt, const float* gq, const float* gt, int64_t B,
                            float rot_weight, float trans_weight, int mode, float* out, float* grad_q,
                            float* grad_t, void* workspace, int device, void* stream, const Geo& geo) {
    DeviceGuard guard(device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool g = geo.z != nullptr;
    if (B <= SMALL_B) {
        auto k = g ? pose_loss_small_kernel<true> : pose_loss_small_kernel<false>;
        k<<<1, LOSS_T, 0, st>>>(pq, pt, gq, gt, (int)B, rot_weight, trans_weight, mode, out, grad_q, grad_t, geo);
    } else {
        if (!workspace) { set_error("pose loss: workspace required for B > %d", SMALL_B); return P6D_EINVAL; }
        int sms = 0;
        P6D_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        int64_t blocks = (B + LOSS_T - 1) / LOSS_T;
        const int64_t cap = (int64_t)sms * 8;
        if (blocks > cap) blocks = cap;
        // geodesic: FAST row (nothing is bit-exact at this size anyway); quaternion-L1: exact row, because
        // its sub-gradient is a sign pattern that a 1-ulp change of u - v could flip
        const bool aligned = ((reinterpret_cast<uintptr_t>(pq) | reinterpret_cast<uintptr_t>(gq) |
                               reinterpret_cast<uintptr_t>(pt) | reinterpret_cast<uintptr_t>(gt)) & 15u) == 0;
        if (!g && aligned) {
            const size_t smem = static_cast<size_t>(STREAM_STAGES) * STREAM_STAGE_FLOATS * sizeof(float);
            auto k = mode == 0 ? pose_loss_stream_kernel<true> : pose_loss_stream_kernel<false>;
            static_assert(STREAM_STAGES * STREAM_STAGE_FLOATS * sizeof(float) + 512 <= 48 * 1024,
                          "the ring must fit the default dynamic shared memory limit (no opt-in attribute is set)");
            int64_t grid = static_cast<int64_t>(sms) * STREAM_CTAS_PER_SM;
            const int64_t n_tiles = B / STREAM_TILE;
            if (grid > n_tiles) grid = n_tiles > 0 ? n_tiles : 1;
            k<<<(unsigned)grid, LOSS_T, smem, st>>>(pq, pt, gq, gt, B, rot_weight, trans_weight, mode, out, grad_q, grad_t,
                                                    static_cast<Workspace*>(workspace));
        } else {
            auto k = mode == 0 ? (g ? pose_loss_large_kernel<true, true> : pose_loss_large_kernel<true, false>)
                               : (g ? pose_loss_large_kernel<false, true> : pose_loss_large_kernel<false, false>);
            k<<<(unsigned)blocks, LOSS_T, 0, st>>>(pq, pt, gq, gt, B, rot_weight, trans_weight, mode, out, grad_q, grad_t,
                                                   static_cast<Workspace*>(workspace), geo);
        }
    }
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

int p6d_pose_loss_fwd_bwd(const float* pq, const float* pt, const float* gq, const float* gt, int64_t B,
                          float rot_weight, float trans_weight, int mode, float* out, float* grad_q,
                          float* grad_t, void* workspace, int device, void* stream) {
    if (B <= 0 || !pq || !pt || !gq || !gt || !out || (mode != 0 && mode != 1)) {
        set_error("p6d_pose_loss_fwd_bwd: bad arguments (B=%lld, mode=%d)", (long long)B, mode);
        return P6D_EINVAL;
    }
    if (((reinterpret_cast<uintptr_t>(pq) | reinterpret_cast<uintptr_t>(gq) | reinterpret_cast<uintptr_t>(grad_q)) & 15u) != 0) {
        set_error("p6d_pose_loss_fwd_bwd: pred_rot, gt_rot and grad_q must be 16-byte aligned (float4 rows)");
        return P6D_EINVAL;
    }
    Geo geo{};
    return launch_pose_loss(pq, pt, gq, gt, B, rot_weight, trans_weight, mode, out, grad_q, grad_t, workspace,
                            device, stream, geo);
}

int p6d_pose_loss_pinhole_fwd_bwd(const float* pq, const float* z, const float* uv, const float* K, int k_batched,
                                  const float* gq, const float* gt, int64_t B, float rot_weight,
                                  float trans_weight, int mode, float* out, float* grad_q, float* grad_z,
                                  float* trans_out, void* workspace, int device, void* stream) {
    if (B <= 0 || !pq || !z || !uv || !K || !gq || !gt || !out || (mode != 0 && mode != 1)) {
        set_error("p6d_pose_loss_pinhole_fwd_bwd: bad arguments (B=%lld, mode=%d)", (long long)B, mode);
        return P6D_EINVAL;
    }
    if (((reinterpret_cast<uintptr_t>(pq) | reinterpret_cast<uintptr_t>(gq) | reinterpret_cast<uintptr_t>(grad_q)) & 15u) != 0 ||
        (reinterpret_cast<uintptr_t>(uv) & 7u) != 0) {
        set_error("p6d_pose_loss_pinhole_fwd_bwd: pred_rot, gt_rot, grad_q must be 16-byte and bbox_center 8-byte aligned");
        return P6D_EINVAL;
    }
    Geo geo{z, uv, K, k_batched, grad_z, trans_out};
    return launch_pose_loss(pq, nullptr, gq, gt, B, rot_weight, trans_weight, mode, out, grad_q, nullptr, workspace,
                            device, stream, geo);
}

}  // extern "C"
