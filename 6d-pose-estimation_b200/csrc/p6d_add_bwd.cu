// p6d_add_bwd.cu -- gradient of ADDLoss.forward w.r.t. the predicted pose (SURVEY.md N3).
//
// The reference gets this from autograd through matmul / norm / min / mean
// (models/add_loss.py:101-150), materialising [n,N,N,3] for symmetric objects (1.6 GB at
// n=32, N=2048).  Here: one CTA per pose, the gt cloud in shared memory, each thread owns
// pred points, finds the nearest gt point (the first index whose ROOTED distance is minimal,
// like torch.norm(...).min: equal roots of different squares tie) with a value+index scan, and
// accumulates dL/dt (3) and dL/dR (9) in float64; thread 0 applies
// the quaternion Jacobian of _quat_to_mat (add_loss.py:203-215, no normalisation).
//   loss = (1/count) * sum_b mean_i d_bi ,  d = |p_i - g_i| (ADD) or min_j |p_i - g_j| (ADD-S)
//   dL/dp_i = scale * (p_i - g*) / d   (0 where d == 0, PyTorch's norm sub-gradient)
// Training-size problem (B = 32, N = 500): latency matters, throughput does not.
#include <mutex>

#include "p6d_common.cuh"

namespace p6d {

constexpr int BWD_T = 256;

struct BwdArgs {
    const float* soa;
    const SlotInfo* slots;
    int n_slots;
    const float* pq;
    const float* pt;
    const float* gq;
    const float* gt;
    const int64_t* obj;
    int64_t B;
    const float* grad_out;  // device scalar (upstream gradient of the 0-d loss)
    const int32_t* count;   // device: number of valid samples (nullable -> inv_count)
    float inv_count;        // 1 / number of valid samples
    float* grad_q;          // [B,4]
    float* grad_t;          // [B,3]
};

__global__ void __launch_bounds__(BWD_T) add_backward_kernel(BwdArgs a, int nmax) {
    extern __shared__ float s_g[];  // gt cloud SoA: x[nmax] y[nmax] z[nmax]
    __shared__ double s_red[BWD_T / 32][12];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int64_t b = blockIdx.x; b < a.B; b += gridDim.x) {
        const int64_t oid = a.obj[b];
        const bool known = oid >= 0 && oid < a.n_slots && a.slots[oid].count > 0;
        if (!known) {  // skipped sample: no gradient (add_loss.py:113)
            if (tid < 4) a.grad_q[4 * b + tid] = 0.0f;
            if (tid < 3) a.grad_t[3 * b + tid] = 0.0f;
            continue;
        }
        const SlotInfo s = a.slots[oid];
        const int n = s.count;
        const float* mx = a.soa + s.soa_offset;
        const float* my = mx + s.padded;
        const float* mz = my + s.padded;
        float q[4], Rp[9], Rg[9], tp[3], tg[3];
#pragma unroll
        for (int k = 0; k < 4; ++k) q[k] = __ldg(a.gq + 4 * b + k);
        quat_to_mat(q, Rg);
#pragma unroll
        for (int k = 0; k < 4; ++k) q[k] = __ldg(a.pq + 4 * b + k);
        quat_to_mat(q, Rp);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            tp[k] = __ldg(a.pt + 3 * b + k);
            tg[k] = __ldg(a.gt + 3 * b + k);
        }
        float* gx = s_g;
        float* gy = s_g + nmax;
        float* gz = s_g + 2 * nmax;
        __syncthreads();  // previous pose's scan is done with s_g / s_red
        for (int i = tid; i < n; i += BWD_T) {
            float x, y, z;
            xform_point(s.xform_bmm, __ldg(mx + i), __ldg(my + i), __ldg(mz + i), Rg, tg, x, y, z);
            gx[i] = x; gy[i] = y; gz[i] = z;
        }
        __syncthreads();
        double acc[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) acc[k] = 0.0;
        for (int i = tid; i < n; i += BWD_T) {
            const float m0 = __ldg(mx + i), m1 = __ldg(my + i), m2 = __ldg(mz + i);
            float px, py, pz;
            xform_point(s.xform_bmm, m0, m1, m2, Rp, tp, px, py, pz);
            int js = i;
            if (s.symmetric) {
                float best = __int_as_float(0x7f800000), prev = best;  // prev: the minimum before best
                js = 0;
                bool nan_seen = false;
                for (int j = 0; j < n; ++j) {
                    const float sv = sq3(__fsub_rn(px, gx[j]), __fsub_rn(py, gy[j]), __fsub_rn(pz, gz[j]));
                    if (sv != sv && !nan_seen) { nan_seen = true; js = j; best = sv; }
                    if (!nan_seen && sv < best) { prev = best; best = sv; js = j; }
                }
                // torch.min runs on the ROOTED distances: an earlier point whose square is larger but
                // whose sqrt equals sqrt(best) is the nearest one.  Its square is >= prev (the running
                // minimum before js), so there is none unless sqrt(prev) == sqrt(best); only then
                // (rare) rescan [0, js).
                if (!nan_seen && js > 0 && __fsqrt_rn(prev) == __fsqrt_rn(best)) {
                    const float r = __fsqrt_rn(best);
                    for (int j = 0; j < js; ++j) {
                        if (__fsqrt_rn(sq3(__fsub_rn(px, gx[j]), __fsub_rn(py, gy[j]), __fsub_rn(pz, gz[j]))) == r) {
                            js = j;
                            break;
                        }
                    }
                }
            }
            const float dx = __fsub_rn(px, gx[js]), dy = __fsub_rn(py, gy[js]), dz = __fsub_rn(pz, gz[js]);
            const float d = __fsqrt_rn(sq3(dx, dy, dz));
            float G[3] = {0.0f, 0.0f, 0.0f};
            if (d != 0.0f) { G[0] = __fdiv_rn(dx, d); G[1] = __fdiv_rn(dy, d); G[2] = __fdiv_rn(dz, d); }
            const float m[3] = {m0, m1, m2};
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                acc[r] += (double)G[r];
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[3 + 3 * r + c] += (double)G[r] * (double)m[c];  // dL/dR[r][c]
            }
        }
#pragma unroll
        for (int k = 0; k < 12; ++k) {
            double v = acc[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) s_red[warp][k] = v;
        }
        __syncthreads();
        if (tid == 0) {
            double t[12];
            for (int k = 0; k < 12; ++k) {
                double v = 0.0;
                for (int w = 0; w < BWD_T / 32; ++w) v += s_red[w][k];
                t[k] = v;
            }
            const double inv_count = a.count ? (__ldg(a.count) > 0 ? 1.0 / (double)__ldg(a.count) : 0.0) : (double)a.inv_count;
            const double scale = (double)__ldg(a.grad_out) * inv_count / (double)n;
            const double x = q[0], y = q[1], z = q[2], w = q[3];
            const double* R = t + 3;  // dL/dR row-major (unscaled)
            const double gxq = 2 * y * R[1] + 2 * z * R[2] + 2 * y * R[3] - 4 * x * R[4] - 2 * w * R[5] + 2 * z * R[6] +
                               2 * w * R[7] - 4 * x * R[8];
            const double gyq = -4 * y * R[0] + 2 * x * R[1] + 2 * w * R[2] + 2 * x * R[3] + 2 * z * R[5] - 2 * w * R[6] +
                               2 * z * R[7] - 4 * y * R[8];
            const double gzq = -4 * z * R[0] - 2 * w * R[1] + 2 * x * R[2] + 2 * w * R[3] - 4 * z * R[4] + 2 * y * R[5] +
                               2 * x * R[6] + 2 * y * R[7];
            const double gwq = -2 * z * R[1] + 2 * y * R[2] + 2 * z * R[3] - 2 * x * R[5] - 2 * y * R[6] + 2 * x * R[7];
            a.grad_q[4 * b + 0] = (float)(scale * gxq);
            a.grad_q[4 * b + 1] = (float)(scale * gyq);
            a.grad_q[4 * b + 2] = (float)(scale * gzq);
            a.grad_q[4 * b + 3] = (float)(scale * gwq);
            a.grad_t[3 * b + 0] = (float)(scale * t[0]);
            a.grad_t[3 * b + 1] = (float)(scale * t[1]);
            a.grad_t[3 * b + 2] = (float)(scale * t[2]);
        }
    }
}

}  // namespace p6d

using namespace p6d;

extern "C" int p6d_add_backward(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                                const float* gt, const int64_t* obj, int64_t B, const float* grad_out,
                                const int32_t* count, float inv_count, float* grad_q, float* grad_t, void* stream) {
    if (!table || B < 0 || (B > 0 && (!pq || !pt || !gq || !gt || !obj || !grad_out || !grad_q || !grad_t))) {
        set_error("p6d_add_backward: bad arguments");
        return P6D_EINVAL;
    }
    if (B == 0) return P6D_OK;
    DeviceGuard guard(table->device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    const int nmax = table->max_count > 0 ? table->max_count : 1;
    const size_t smem = sizeof(float) * 3 * (size_t)nmax;
    int limit = 0;
    P6D_CUDA(cudaDeviceGetAttribute(&limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, table->device));
    if (smem + 1024 > (size_t)limit) {
        set_error("p6d_add_backward: mesh of %d points does not fit shared memory", nmax);
        return P6D_ETOOBIG;
    }
    {
        // the attribute is a per-device maximum shared by every table and thread: only ever raise it
        static std::mutex mu;
        static size_t raised[64];
        std::lock_guard<std::mutex> lock(mu);
        size_t& cur = raised[table->device & 63];
        if (smem > cur) {
            P6D_CUDA(cudaFuncSetAttribute(add_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            cur = smem;
        }
    }
    BwdArgs a{table->d_soa, table->d_slots, table->n_slots, pq, pt, gq, gt, obj, B, grad_out, count, inv_count, grad_q, grad_t};
    int64_t grid = B < (int64_t)table->sm_count * 4 ? B : (int64_t)table->sm_count * 4;
    add_backward_kernel<<<(unsigned)grid, BWD_T, smem, static_cast<cudaStream_t>(stream)>>>(a, nmax);
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}
