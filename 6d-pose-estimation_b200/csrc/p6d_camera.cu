// p6d_camera.cu -- geometric-translation kernels (sm_100a).
//
//   pinhole_fwd / pinhole_bwd : PoseNetRGBGeometric._compute_pinhole_translation
//                               (reference models/pose_net_rgb_geometric.py:93-109)
//   depth_backproject         : PoseNetRGBDGeometric._compute_pinhole_translation
//                               (reference models/pose_net_rgbd_geometric.py:56-85)
//
// Elementwise, HBM/latency-bound: one thread per row, K read as scalars (4 of the 9
// entries), everything else coalesced.  Operation order is the reference's:
// ((u - cx) * z) / fx with an IEEE division.

#include "p6d_common.cuh"

namespace p6d {

constexpr int CAM_T = 256;

__device__ __forceinline__ void load_k(const float* __restrict__ K, int k_batched, int64_t b, float& fx,
                                       float& fy, float& cx, float& cy) {
    const float* k = K + (k_batched ? 9 * b : 0);
    fx = __ldg(k + 0);
    cx = __ldg(k + 2);
    fy = __ldg(k + 4);
    cy = __ldg(k + 5);
}

__global__ void __launch_bounds__(CAM_T) pinhole_fwd_kernel(const float* __restrict__ z, const float* __restrict__ uv,
                                                            const float* __restrict__ K, int k_batched, int64_t B,
                                                            float* __restrict__ out) {
    for (int64_t b = (int64_t)blockIdx.x * CAM_T + threadIdx.x; b < B; b += (int64_t)gridDim.x * CAM_T) {
        float fx, fy, cx, cy;
        load_k(K, k_batched, b, fx, fy, cx, cy);
        const float2 c = *reinterpret_cast<const float2*>(uv + 2 * b);
        const float zz = z[b];
        out[3 * b + 0] = __fdiv_rn(__fmul_rn(__fsub_rn(c.x, cx), zz), fx);
        out[3 * b + 1] = __fdiv_rn(__fmul_rn(__fsub_rn(c.y, cy), zz), fy);
        out[3 * b + 2] = zz;
    }
}

// Shared [3,3] K (the reference's common case): 24 B per row, nothing but z, the centre and the
// output.  One row per thread writes its three floats with stride-12 scalar stores -- three store
// instructions that each touch every sector of the warp's 384 bytes (measured 3.9 TB/s = 60 % of HBM).
// Four rows per thread: z as one float4, the centres as two, the output as three 16-byte vectors (72 %).
// The three vectors of a lane are 48 bytes apart, so each store instruction still fills only half of every
// 32-byte sector it touches; the warp therefore passes its 1,536 output bytes through shared memory (12-word
// lane stride: conflict-free for 128-bit accesses) and stores them as three fully coalesced 512-byte rows.
// Same arithmetic per row.
__global__ void __launch_bounds__(CAM_T) pinhole_fwd_shared4_kernel(const float4* __restrict__ z4,
                                                                    const float4* __restrict__ uv4,
                                                                    const float* __restrict__ K, int64_t B4,
                                                                    float4* __restrict__ out4) {
    __shared__ float4 s_out[CAM_T / 32][96];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4* so = s_out[warp];
    const float fx = __ldg(K + 0), cx = __ldg(K + 2), fy = __ldg(K + 4), cy = __ldg(K + 5);
    // whole warps only: the loop bound is per warp so that every lane reaches the __syncwarp()s
    const int64_t stride = (int64_t)gridDim.x * CAM_T;
    for (int64_t q0 = (int64_t)blockIdx.x * CAM_T + warp * 32; q0 < B4; q0 += stride) {
        const int64_t q = q0 + lane;
        const bool live = q < B4;
        if (live) {
            const float4 zz = z4[q];
            const float4 c0 = uv4[2 * q], c1 = uv4[2 * q + 1];          // (u0,v0,u1,v1), (u2,v2,u3,v3)
            const float x0 = __fdiv_rn(__fmul_rn(__fsub_rn(c0.x, cx), zz.x), fx), y0 = __fdiv_rn(__fmul_rn(__fsub_rn(c0.y, cy), zz.x), fy);
            const float x1 = __fdiv_rn(__fmul_rn(__fsub_rn(c0.z, cx), zz.y), fx), y1 = __fdiv_rn(__fmul_rn(__fsub_rn(c0.w, cy), zz.y), fy);
            const float x2 = __fdiv_rn(__fmul_rn(__fsub_rn(c1.x, cx), zz.z), fx), y2 = __fdiv_rn(__fmul_rn(__fsub_rn(c1.y, cy), zz.z), fy);
            const float x3 = __fdiv_rn(__fmul_rn(__fsub_rn(c1.z, cx), zz.w), fx), y3 = __fdiv_rn(__fmul_rn(__fsub_rn(c1.w, cy), zz.w), fy);
            so[3 * lane + 0] = make_float4(x0, y0, zz.x, x1);
            so[3 * lane + 1] = make_float4(y1, zz.y, x2, y2);
            so[3 * lane + 2] = make_float4(zz.z, x3, y3, zz.w);
        }
        __syncwarp();
        const int64_t left = B4 - q0;                                  // rows-of-four of this warp that exist
        const int vecs = left >= 32 ? 96 : (int)(3 * left);
#pragma unroll
        for (int k = 0; k < 3; ++k)
            if (32 * k + lane < vecs) out4[3 * q0 + 32 * k + lane] = so[32 * k + lane];
        __syncwarp();
    }
}

__global__ void __launch_bounds__(CAM_T) pinhole_bwd_kernel(const float* __restrict__ go, const float* __restrict__ uv,
                                                            const float* __restrict__ K, int k_batched, int64_t B,
                                                            float* __restrict__ gz) {
    for (int64_t b = (int64_t)blockIdx.x * CAM_T + threadIdx.x; b < B; b += (int64_t)gridDim.x * CAM_T) {
        float fx, fy, cx, cy;
        load_k(K, k_batched, b, fx, fy, cx, cy);
        const float2 c = *reinterpret_cast<const float2*>(uv + 2 * b);
        // autograd order: d/dz[((u-cx)*z)/fx] = (g/fx)*(u-cx)
        const float gx = __fmul_rn(__fdiv_rn(go[3 * b + 0], fx), __fsub_rn(c.x, cx));
        const float gy = __fmul_rn(__fdiv_rn(go[3 * b + 1], fy), __fsub_rn(c.y, cy));
        gz[b] = __fadd_rn(__fadd_rn(gx, gy), go[3 * b + 2]);
    }
}

__device__ __forceinline__ float clamp_keep_nan(float x, float lo, float hi) {
    // torch.clamp: NaN stays NaN
    if (x != x) return x;
    return x < lo ? lo : (x > hi ? hi : x);
}

__global__ void __launch_bounds__(CAM_T) depth_backproject_kernel(const float* __restrict__ depth, int H, int W,
                                                                  const float* __restrict__ uv,
                                                                  const float* __restrict__ K, int k_batched,
                                                                  int64_t B, float clamp_hi,
                                                                  float* __restrict__ out) {
    const long long hi = (long long)clamp_hi;
    for (int64_t b = (int64_t)blockIdx.x * CAM_T + threadIdx.x; b < B; b += (int64_t)gridDim.x * CAM_T) {
        float fx, fy, cx, cy;
        load_k(K, k_batched, b, fx, fy, cx, cy);
        const float2 c = *reinterpret_cast<const float2*>(uv + 2 * b);
        const float u = clamp_keep_nan(c.x, 0.0f, clamp_hi);
        const float v = clamp_keep_nan(c.y, 0.0f, clamp_hi);
        // .long(): truncation toward zero; NaN converts to INT64_MIN on the reference's x86 host
        long long ui = (u != u) ? LLONG_MIN : (long long)u;
        long long vi = (v != v) ? LLONG_MIN : (long long)v;
        ui = ui < 0 ? 0 : (ui > hi ? hi : ui);
        vi = vi < 0 ? 0 : (vi > hi ? hi : vi);
        // one pixel per crop: ask L2 for the smallest fetch it offers (64 B; the default promotes a
        // miss to 128 B, which was 2/3 of this kernel's DRAM traffic) and keep the line out of L1
        float zz;
        asm("ld.global.nc.L1::no_allocate.L2::64B.f32 %0, [%1];" : "=f"(zz) : "l"(depth + ((int64_t)b * H + vi) * W + ui));
        zz = (zz > 0.01f) ? zz : 0.5f;  // false for NaN -> 0.5
        zz = clamp_keep_nan(zz, 0.1f, 2.0f);
        out[3 * b + 0] = __fdiv_rn(__fmul_rn(__fsub_rn(u, cx), zz), fx);
        out[3 * b + 1] = __fdiv_rn(__fmul_rn(__fsub_rn(v, cy), zz), fy);
        out[3 * b + 2] = zz;
    }
}

// ---------------------------------------------------------------------------------
// N1: frame-level fusion of the reference's crop pipeline with (d2).
// The reference (data/dataset_rgbd.py:104-179) pads the uint16 depth frame, cuts a square
// crop of 1.2 x max(w,h), resizes it to 224^2 with cv2.resize(INTER_LINEAR) -- ~200 KB of
// traffic per box -- and the network then reads ONE pixel of the result
// (models/pose_net_rgbd_geometric.py:69-75).  Here one thread per box computes the crop
// geometry (Python int / float64 semantics), the remapped centre and K_crop (NumPy
// float32 semantics), evaluates cv2's bilinear formula at that single pixel from 4 texels of the
// original frame (zero outside the frame = the constant border), and back-projects.
// cv2.resize on CV_16U has two arithmetics (oracle.resize_linear_u16, tests/test_live_pins.py):
//   bilinear 0  the pip wheel's default, i.e. what the reference's call computes: IPP's
//               ippiResizeLinear_16u -- float64 source coordinate, float32 weight, horizontal then
//               vertical lerp as one fma(b - a, w, a) each, round half to even;
//   bilinear 1  OpenCV's own C++ path (no IPP): float32 coordinate, a*(1-w) + b*w with separate
//               roundings, and INTER_AREA ((a+b+c+d+2) >> 2) when the crop is exactly 2x the output.
__device__ __forceinline__ void resize_axis_ipp(int d, long long cs, int img, int& s0, int& s1, float& w) {
    const double c = __dsub_rn(__dmul_rn((double)d + 0.5, (double)cs / (double)img), 0.5);
    const double fl = floor(c);
    const long long s = (long long)fl;
    w = s < 0 ? 0.0f : (float)__dsub_rn(c, fl);
    s0 = (int)(s < 0 ? 0 : (s > cs - 1 ? cs - 1 : s));
    s1 = (int)(s + 1 < 0 ? 0 : (s + 1 > cs - 1 ? cs - 1 : s + 1));
}

__device__ __forceinline__ void resize_axis(int d, long long cs, int img, int& s0, int& s1, float& w0, float& w1) {
    const double scale = 1.0 / ((double)img / (double)cs);
    const float v = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
    int s = (int)floorf(v);
    float w = __fsub_rn(v, (float)s);
    if (s < 0) { s = 0; w = 0.0f; }
    if (s >= cs - 1) { s = (int)cs - 1; w = 0.0f; }
    s0 = s;
    s1 = s + 1 < cs ? s + 1 : (int)cs - 1;
    w0 = __fsub_rn(1.0f, w);
    w1 = w;
}

__global__ void __launch_bounds__(CAM_T) depth_crop_backproject_kernel(
    const unsigned short* __restrict__ depth, int H, int W, const int* __restrict__ boxes, int64_t B,
    const float* __restrict__ K, int img, int bilinear, float* __restrict__ xyz, float* __restrict__ center_out,
    float* __restrict__ kcrop_out, unsigned short* __restrict__ zmm_out) {
    const float fx = __ldg(K + 0), cx = __ldg(K + 2), fy = __ldg(K + 4), cy = __ldg(K + 5);
    for (int64_t b = (int64_t)blockIdx.x * CAM_T + threadIdx.x; b < B; b += (int64_t)gridDim.x * CAM_T) {
        const int4 bb = *reinterpret_cast<const int4*>(boxes + 4 * b);
        const int x = bb.x, y = bb.y, w = bb.z, h = bb.w;
        // Python scalars: float64 and int() truncation toward zero
        const double c_x = (double)x + (double)w / 2.0, c_y = (double)y + (double)h / 2.0;
        const double size = (double)(w > h ? w : h) * 1.2;
        long long x1 = (long long)__dsub_rn(c_x, size / 2.0), y1 = (long long)__dsub_rn(c_y, size / 2.0);
        const long long cs = (long long)size;
        if (cs < 1) {  // degenerate box: the reference would fail in cv2.resize; emit the fallback depth
            xyz[3 * b] = 0.0f; xyz[3 * b + 1] = 0.0f; xyz[3 * b + 2] = 0.5f;
            if (center_out) { center_out[2 * b] = 0.0f; center_out[2 * b + 1] = 0.0f; }
            if (kcrop_out) for (int k = 0; k < 9; ++k) kcrop_out[9 * b + k] = 0.0f;
            if (zmm_out) zmm_out[b] = 0;
            continue;
        }
        const long long pad_l = x1 < 0 ? -x1 : 0, pad_t = y1 < 0 ? -y1 : 0;
        x1 += pad_l;
        y1 += pad_t;
        // NumPy float32 arithmetic
        const float scale32 = (float)((double)img / (double)cs);
        const float hi = (float)(img - 1);
        const float ccx = __fsub_rn(__fadd_rn((float)c_x, (float)pad_l), (float)x1);
        const float ccy = __fsub_rn(__fadd_rn((float)c_y, (float)pad_t), (float)y1);
        float u = __fmul_rn(ccx, scale32), v = __fmul_rn(ccy, scale32);
        u = u < 0.0f ? 0.0f : (u > hi ? hi : u);   // np.clip(center_resized, 0, img-1)
        v = v < 0.0f ? 0.0f : (v > hi ? hi : v);
        const float fxc = __fmul_rn(fx, scale32), fyc = __fmul_rn(fy, scale32);
        const float cxc = __fmul_rn(__fsub_rn(__fadd_rn(cx, (float)pad_l), (float)x1), scale32);
        const float cyc = __fmul_rn(__fsub_rn(__fadd_rn(cy, (float)pad_t), (float)y1), scale32);
        int ui = (int)u, vi = (int)v;              // .long(): truncation, then clamp
        ui = ui < 0 ? 0 : (ui > img - 1 ? img - 1 : ui);
        vi = vi < 0 ? 0 : (vi > img - 1 ? img - 1 : vi);
        auto texel = [&](int yy, int xx) -> float {
            const long long fy_ = y1 + yy - pad_t, fx_ = x1 + xx - pad_l;
            if (fy_ < 0 || fy_ >= H || fx_ < 0 || fx_ >= W) return 0.0f;   // cv2.copyMakeBorder(..., value=0)
            return (float)__ldg(depth + fy_ * W + fx_);
        };
        int sx0, sx1, sy0, sy1;
        float val;
        if (bilinear == 0) {                        // IPP (the reference's default cv2.resize)
            float wx, wy;
            resize_axis_ipp(ui, cs, img, sx0, sx1, wx);
            resize_axis_ipp(vi, cs, img, sy0, sy1, wy);
            const float t00 = texel(sy0, sx0), t01 = texel(sy0, sx1), t10 = texel(sy1, sx0), t11 = texel(sy1, sx1);
            const float h0 = __fmaf_rn(__fsub_rn(t01, t00), wx, t00);
            const float h1 = __fmaf_rn(__fsub_rn(t11, t10), wx, t10);
            val = __fmaf_rn(__fsub_rn(h1, h0), wy, h0);
        } else if (cs == 2ll * img) {               // OpenCV C++ path, exact 2x: INTER_AREA, rounds half up
            const int q = (int)texel(2 * vi, 2 * ui) + (int)texel(2 * vi, 2 * ui + 1) + (int)texel(2 * vi + 1, 2 * ui) +
                          (int)texel(2 * vi + 1, 2 * ui + 1);
            val = (float)((q + 2) >> 2);
        } else {                                    // OpenCV C++ path
            float a0, a1, b0, b1;
            resize_axis(ui, cs, img, sx0, sx1, a0, a1);
            resize_axis(vi, cs, img, sy0, sy1, b0, b1);
            const float h0 = __fadd_rn(__fmul_rn(texel(sy0, sx0), a0), __fmul_rn(texel(sy0, sx1), a1));
            const float h1 = __fadd_rn(__fmul_rn(texel(sy1, sx0), a0), __fmul_rn(texel(sy1, sx1), a1));
            val = __fadd_rn(__fmul_rn(h0, b0), __fmul_rn(h1, b1));
        }
        int zi = __float2int_rn(val);              // saturate_cast<ushort>(cvRound)
        zi = zi < 0 ? 0 : (zi > 65535 ? 65535 : zi);
        float z = __fdiv_rn((float)zi, 1000.0f);
        z = (z > 0.01f) ? z : 0.5f;
        z = z < 0.1f ? 0.1f : (z > 2.0f ? 2.0f : z);
        xyz[3 * b + 0] = __fdiv_rn(__fmul_rn(__fsub_rn(u, cxc), z), fxc);
        xyz[3 * b + 1] = __fdiv_rn(__fmul_rn(__fsub_rn(v, cyc), z), fyc);
        xyz[3 * b + 2] = z;
        if (center_out) { center_out[2 * b] = u; center_out[2 * b + 1] = v; }
        if (kcrop_out) {
            float* k = kcrop_out + 9 * b;
            k[0] = fxc; k[1] = 0.0f; k[2] = cxc; k[3] = 0.0f; k[4] = fyc; k[5] = cyc; k[6] = 0.0f; k[7] = 0.0f; k[8] = 1.0f;
        }
        if (zmm_out) zmm_out[b] = (unsigned short)zi;
    }
}

// ---------------------------------------------------------------------------------
// N1, inference form: the per-detection crop code of scripts/inference/inference_rgbd_geometric.py:109-170
// fused with (d2).  Differs from the dataset form above in three places, each of which moves a rounding:
// detector boxes are integer (x1, y1, x2, y2); the crop is cast to float32 BEFORE cv2.resize, so the
// resized depth is the un-rounded float32 lerp (IPP's ippiResizeLinear_32f: the same float64 coordinate /
// float32 weight / one fma per lerp as its 16-bit form); centre and K_crop are computed in float64 (Python
// floats, the float64 DEFAULT_K) and only the results are stored as float32.
__global__ void __launch_bounds__(CAM_T) detection_backproject_kernel(
    const unsigned short* __restrict__ depth, int H, int W, const int* __restrict__ boxes, int64_t B,
    const double* __restrict__ K, int img, float* __restrict__ xyz, float* __restrict__ center_out,
    float* __restrict__ kcrop_out, float* __restrict__ zm_out) {
    const double fx = K[0], cx = K[2], fy = K[4], cy = K[5];
    for (int64_t b = (int64_t)blockIdx.x * CAM_T + threadIdx.x; b < B; b += (int64_t)gridDim.x * CAM_T) {
        const int4 bb = *reinterpret_cast<const int4*>(boxes + 4 * b);
        // Python scalars: float64 and int() truncation toward zero
        const double c_x = ((double)bb.x + (double)bb.z) / 2.0, c_y = ((double)bb.y + (double)bb.w) / 2.0;
        const long long w = (long long)bb.z - bb.x, h = (long long)bb.w - bb.y;
        const double size = (double)(w > h ? w : h) * 1.2;
        const long long crop_x1 = (long long)__dsub_rn(c_x, size / 2.0), crop_y1 = (long long)__dsub_rn(c_y, size / 2.0);
        const long long cs = (long long)size;
        if (cs < 1) {  // degenerate box: the reference would fail in cv2.resize; emit the fallback depth
            xyz[3 * b] = 0.0f; xyz[3 * b + 1] = 0.0f; xyz[3 * b + 2] = 0.5f;
            if (center_out) { center_out[2 * b] = 0.0f; center_out[2 * b + 1] = 0.0f; }
            if (kcrop_out) for (int k = 0; k < 9; ++k) kcrop_out[9 * b + k] = 0.0f;
            if (zm_out) zm_out[b] = 0.0f;
            continue;
        }
        const long long pad_l = crop_x1 < 0 ? -crop_x1 : 0, pad_t = crop_y1 < 0 ? -crop_y1 : 0;
        const long long adj_x1 = crop_x1 + pad_l, adj_y1 = crop_y1 + pad_t;
        const double scale = (double)img / (double)cs;
        const float hi = (float)(img - 1);
        // float64 products, stored as float32 (np.array(..., dtype=np.float32)), then np.clip in float32
        float u = (float)__dmul_rn(__dsub_rn(__dadd_rn(c_x, (double)pad_l), (double)adj_x1), scale);
        float v = (float)__dmul_rn(__dsub_rn(__dadd_rn(c_y, (double)pad_t), (double)adj_y1), scale);
        u = u < 0.0f ? 0.0f : (u > hi ? hi : u);
        v = v < 0.0f ? 0.0f : (v > hi ? hi : v);
        const float fxc = (float)__dmul_rn(fx, scale), fyc = (float)__dmul_rn(fy, scale);
        const float cxc = (float)__dmul_rn(__dsub_rn(__dadd_rn(cx, (double)pad_l), (double)crop_x1), scale);
        const float cyc = (float)__dmul_rn(__dsub_rn(__dadd_rn(cy, (double)pad_t), (double)crop_y1), scale);
        int ui = (int)u, vi = (int)v;              // .long(): truncation, then clamp
        ui = ui < 0 ? 0 : (ui > img - 1 ? img - 1 : ui);
        vi = vi < 0 ? 0 : (vi > img - 1 ? img - 1 : vi);
        auto texel = [&](int yy, int xx) -> float {
            const long long fy_ = adj_y1 + yy - pad_t, fx_ = adj_x1 + xx - pad_l;
            if (fy_ < 0 || fy_ >= H || fx_ < 0 || fx_ >= W) return 0.0f;   // cv2.copyMakeBorder(..., value=0)
            return (float)__ldg(depth + fy_ * W + fx_);
        };
        int sx0, sx1, sy0, sy1;
        float wx, wy;
        resize_axis_ipp(ui, cs, img, sx0, sx1, wx);
        resize_axis_ipp(vi, cs, img, sy0, sy1, wy);
        const float t00 = texel(sy0, sx0), t01 = texel(sy0, sx1), t10 = texel(sy1, sx0), t11 = texel(sy1, sx1);
        const float h0 = __fmaf_rn(__fsub_rn(t01, t00), wx, t00);
        const float h1 = __fmaf_rn(__fsub_rn(t11, t10), wx, t10);
        const float val = __fmaf_rn(__fsub_rn(h1, h0), wy, h0);
        const float zm = __fdiv_rn(val, 1000.0f);  // crop_depth_resized / 1000.0 (float32 array / Python float)
        float z = (zm > 0.01f) ? zm : 0.5f;
        z = z < 0.1f ? 0.1f : (z > 2.0f ? 2.0f : z);
        xyz[3 * b + 0] = __fdiv_rn(__fmul_rn(__fsub_rn(u, cxc), z), fxc);
        xyz[3 * b + 1] = __fdiv_rn(__fmul_rn(__fsub_rn(v, cyc), z), fyc);
        xyz[3 * b + 2] = z;
        if (center_out) { center_out[2 * b] = u; center_out[2 * b + 1] = v; }
        if (kcrop_out) {
            float* k = kcrop_out + 9 * b;
            k[0] = fxc; k[1] = 0.0f; k[2] = cxc; k[3] = 0.0f; k[4] = fyc; k[5] = cyc; k[6] = 0.0f; k[7] = 0.0f; k[8] = 1.0f;
        }
        if (zm_out) zm_out[b] = zm;
    }
}

// ---------------------------------------------------------------------------------
// N4: utils/visualization.project_points for B poses (float64 like the reference's NumPy).
__global__ void __launch_bounds__(CAM_T) project_points_kernel(const double* __restrict__ pts, int N,
                                                               const double* __restrict__ rot, int is_quat,
                                                               const double* __restrict__ tr,
                                                               const double* __restrict__ K, int64_t B,
                                                               long long* __restrict__ uv) {
    const double fx = K[0], cx = K[2], fy = K[4], cy = K[5];
    const int64_t total = B * N;
    for (int64_t i = (int64_t)blockIdx.x * CAM_T + threadIdx.x; i < total; i += (int64_t)gridDim.x * CAM_T) {
        const int64_t b = i / N;
        const int n = (int)(i - b * N);
        double R[9];
        if (is_quat) {
            // scipy Rotation.from_quat: normalise, then the homogeneous formula
            double x = rot[4 * b], y = rot[4 * b + 1], z = rot[4 * b + 2], w = rot[4 * b + 3];
            const double nrm = sqrt(x * x + y * y + z * z + w * w);
            x /= nrm; y /= nrm; z /= nrm; w /= nrm;
            R[0] = x * x - y * y - z * z + w * w; R[1] = 2 * (x * y - z * w); R[2] = 2 * (x * z + y * w);
            R[3] = 2 * (x * y + z * w); R[4] = -x * x + y * y - z * z + w * w; R[5] = 2 * (y * z - x * w);
            R[6] = 2 * (x * z - y * w); R[7] = 2 * (y * z + x * w); R[8] = -x * x - y * y + z * z + w * w;
        } else {
#pragma unroll
            for (int k = 0; k < 9; ++k) R[k] = rot[9 * b + k];
        }
        const double px = pts[3 * n], py = pts[3 * n + 1], pz = pts[3 * n + 2];
        const double X = R[0] * px + R[1] * py + R[2] * pz + tr[3 * b];
        const double Y = R[3] * px + R[4] * py + R[5] * pz + tr[3 * b + 1];
        double Z = R[6] * px + R[7] * py + R[8] * pz + tr[3 * b + 2];
        Z = Z < 0.001 ? 0.001 : Z;                    // np.clip(z, 0.001, None)
        uv[2 * i] = (long long)(X * fx / Z + cx);     // .astype(int): truncation toward zero
        uv[2 * i + 1] = (long long)(Y * fy / Z + cy);
    }
}

// Grid of a grid-stride kernel: one thread per row up to what is RESIDENT at once.  Every block of a grid-stride
// loop runs the same number of trips, so blocks beyond the resident set form a second, thinly occupied wave that
// takes as long as the first (the 40-register shared-K pinhole kernel fits 6 blocks per SM: a fixed cap of 8 per
// SM ran 1.33 waves and reached 72 % of HBM).
template <class Kernel>
static int grid_for(Kernel kernel, int64_t B, int device, unsigned* grid) {
    int per_sm = 0;
    int rc = ctas_per_sm(reinterpret_cast<const void*>(kernel), CAM_T, device, 0, &per_sm);
    if (rc) return rc;
    int sms = 0;
    P6D_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    int64_t blocks = (B + CAM_T - 1) / CAM_T;
    const int64_t cap = (int64_t)sms * per_sm;
    *grid = (unsigned)(blocks > cap ? cap : blocks);
    return P6D_OK;
}

}  // namespace p6d

using namespace p6d;

extern "C" {

int p6d_pinhole_fwd(const float* z, const float* uv, const float* K, int k_batched, int64_t B, float* out,
                    int device, void* stream) {
    if (B < 0 || (B > 0 && (!z || !uv || !K || !out))) { set_error("p6d_pinhole_fwd: bad arguments"); return P6D_EINVAL; }
    if (reinterpret_cast<uintptr_t>(uv) & 7u) { set_error("p6d_pinhole_fwd: bbox_center must be 8-byte aligned (float2 rows)"); return P6D_EINVAL; }
    if (B == 0) return P6D_OK;
    DeviceGuard guard(device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    unsigned grid;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = !k_batched && B >= 1024 &&
                     ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(uv) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
    if (vec) {       // four rows per thread, 16-byte accesses; the last B % 4 rows go through the scalar kernel
        const int64_t B4 = B / 4, done = 4 * B4;
        int rc = grid_for(pinhole_fwd_shared4_kernel, B4, device, &grid);
        if (rc) return rc;
        pinhole_fwd_shared4_kernel<<<grid, CAM_T, 0, st>>>(reinterpret_cast<const float4*>(z), reinterpret_cast<const float4*>(uv),
                                                         K, B4, reinterpret_cast<float4*>(out));
        P6D_CUDA(cudaGetLastError());
        if (done < B) {
            pinhole_fwd_kernel<<<1, CAM_T, 0, st>>>(z + done, uv + 2 * done, K, 0, B - done, out + 3 * done);
            P6D_CUDA(cudaGetLastError());
        }
        return P6D_OK;
    }
    int rc = grid_for(pinhole_fwd_kernel, B, device, &grid);
    if (rc) return rc;
    pinhole_fwd_kernel<<<grid, CAM_T, 0, st>>>(z, uv, K, k_batched, B, out);
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

int p6d_pinhole_bwd(const float* grad_out, const float* uv, const float* K, int k_batched, int64_t B,
                    float* grad_z, int device, void* stream) {
    if (B < 0 || (B > 0 && (!grad_out || !uv || !K || !grad_z))) { set_error("p6d_pinhole_bwd: bad arguments"); return P6D_EINVAL; }
    if (reinterpret_cast<uintptr_t>(uv) & 7u) { set_error("p6d_pinhole_bwd: bbox_center must be 8-byte aligned (float2 rows)"); return P6D_EINVAL; }
    if (B == 0) return P6D_OK;
    DeviceGuard guard(device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    unsigned grid;
    int rc = grid_for(pinhole_bwd_kernel, B, device, &grid);
    if (rc) return rc;
    pinhole_bwd_kernel<<<grid, CAM_T, 0, static_cast<cudaStream_t>(stream)>>>(grad_out, uv, K, k_batched, B, grad_z);
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

int p6d_depth_backproject(const float* depth, int H, int W, const float* uv, const float* K, int k_batched,
                          int64_t B, float clamp_hi, float* out, int device, void* stream) {
    if (B < 0 || H < 1 || W < 1 || (B > 0 && (!depth || !uv || !K || !out))) {
        set_error("p6d_depth_backproject: bad arguments");
        return P6D_EINVAL;
    }
    if (!(clamp_hi >= 0.0f) || clamp_hi > (float)(H - 1) || clamp_hi > (float)(W - 1)) {
        set_error("p6d_depth_backproject: clamp_hi=%g outside the %dx%d depth map", (double)clamp_hi, H, W);
        return P6D_EINVAL;
    }
    if (reinterpret_cast<uintptr_t>(uv) & 7u) {
        set_error("p6d_depth_backproject: bbox_center must be 8-byte aligned (float2 rows)");
        return P6D_EINVAL;
    }
    if (B == 0) return P6D_OK;
    DeviceGuard guard(device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    unsigned grid;
    int rc = grid_for(depth_backproject_kernel, B, device, &grid);
    if (rc) return rc;
    depth_backproject_kernel<<<grid, CAM_T, 0, static_cast<cudaStream_t>(stream)>>>(depth, H, W, uv, K, k_batched, B,
                                                                                    clamp_hi, out);
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

int p6d_depth_crop_backproject(const uint16_t* depth, int H, int W, const int32_t* boxes, int64_t B,
                               const float* K, int img_size, int bilinear, float* xyz, float* center, float* kcrop,
                               uint16_t* z_mm, int device, void* stream) {
    if (B < 0 || H < 1 || W < 1 || img_size < 1 || (bilinear != 0 && bilinear != 1) ||
        (B > 0 && (!depth || !boxes || !K || !xyz))) {
        set_error("p6d_depth_crop_backproject: bad arguments");
        return P6D_EINVAL;
    }
    if (reinterpret_cast<uintptr_t>(boxes) & 15u) {
        set_error("p6d_depth_crop_backproject: boxes must be 16-byte aligned (int4 rows)");
        return P6D_EINVAL;
    }
    if (B == 0) return P6D_OK;
    DeviceGuard guard(device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    unsigned grid;
    int rc = grid_for(depth_crop_backproject_kernel, B, device, &grid);
    if (rc) return rc;
    depth_crop_backproject_kernel<<<grid, CAM_T, 0, static_cast<cudaStream_t>(stream)>>>(
        depth, H, W, boxes, B, K, img_size, bilinear, xyz, center, kcrop, z_mm);
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

int p6d_detection_backproject(const uint16_t* depth, int H, int W, const int32_t* boxes_xyxy, int64_t B,
                              const double* K, int img_size, float* xyz, float* center, float* kcrop, float* z_m,
                              int device, void* stream) {
    if (B < 0 || H < 1 || W < 1 || img_size < 1 || (B > 0 && (!depth || !boxes_xyxy || !K || !xyz))) {
        set_error("p6d_detection_backproject: bad arguments");
        return P6D_EINVAL;
    }
    if (reinterpret_cast<uintptr_t>(boxes_xyxy) & 15u) {
        set_error("p6d_detection_backproject: boxes must be 16-byte aligned (int4 rows)");
        return P6D_EINVAL;
    }
    if (B == 0) return P6D_OK;
    DeviceGuard guard(device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    unsigned grid;
    int rc = grid_for(detection_backproject_kernel, B, device, &grid);
    if (rc) return rc;
    detection_backproject_kernel<<<grid, CAM_T, 0, static_cast<cudaStream_t>(stream)>>>(
        depth, H, W, boxes_xyxy, B, K, img_size, xyz, center, kcrop, z_m);
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

int p6d_project_points(const double* points, int N, const double* rotation, int rotation_is_quat,
                       const double* translation, const double* K, int64_t B, int64_t* uv, int device, void* stream) {
    if (B < 0 || N < 0 || ((B > 0 && N > 0) && (!points || !rotation || !translation || !K || !uv))) {
        set_error("p6d_project_points: bad arguments");
        return P6D_EINVAL;
    }
    if (B == 0 || N == 0) return P6D_OK;
    DeviceGuard guard(device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    unsigned grid;
    int rc = grid_for(project_points_kernel, B * N, device, &grid);
    if (rc) return rc;
    project_points_kernel<<<grid, CAM_T, 0, static_cast<cudaStream_t>(stream)>>>(
        points, N, rotation, rotation_is_quat, translation, K, B, reinterpret_cast<long long*>(uv));
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

}  // extern "C"
