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
//
// Meshes beyond its shared memory (opt-in, p6d_mesh_table_set_large_mesh_loss): add_backward_streamed_kernel splits
// every pose into items of P pred points (a persistent grid claims them through an atomic counter); symmetric
// samples stream the gt cloud in 1,024-point tiles through the TMA / mbarrier ring of the streamed evaluation kernel
// and carry the nearest-point state (best, prev, js, NaN) across tiles, so every pred point picks the index the
// resident kernel picks.  Each item stores its 12 float64 partials; the pose's last item sums them in item order
// (deterministic) and applies the same tail (bwd_pose_tail) as the resident kernel.

#include <algorithm>

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

// dL/dt and dL/dq of pose b from the unscaled sums t = (sum G, sum G m^T) over its n points: scale by
// grad_out / (count * n), then the Jacobian of _quat_to_mat at the pred quaternion q (add_loss.py:203-215).
__device__ __forceinline__ void bwd_pose_tail(const BwdArgs& a, int64_t b, const float* q, int n, const double* t) {
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

__global__ void __launch_bounds__(BWD_T) add_backward_kernel(BwdArgs a, int nmax) {
    extern __shared__ float s_g[];  // gt cloud SoA: x[nmax] y[nmax] z[nmax]
    __shared__ double s_red[BWD_T / 32][12];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int64_t b = blockIdx.x; b < a.B; b += gridDim.x) {
        const int64_t oid = a.obj[b];
        if (!slot_known(oid, a.n_slots, a.slots)) {  // skipped sample: no gradient (add_loss.py:113)
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
            bwd_pose_tail(a, b, q, n, t);
        }
    }
}


// ---------------------------------------------------------------- streamed backward
constexpr int SB_G = 1024;                 // gt points per tile (the streamed evaluation kernel's tile)
constexpr int SB_STAGES = 2;               // TMA ring depth
constexpr size_t SB_WS_BYTES = size_t(64) << 20;

struct BwdStreamArgs {
    int64_t first;      // first pose of the chunk
    int nposes;         // poses in the chunk
    int nblk;           // items per pose of the table's largest mesh
    int* counter;       // work counter (zeroed before the launch)
    int* tickets;       // [nposes] finished items per pose (zeroed before the launch)
    double* part;       // [nposes][nblk][12] per-item partial sums
};

template <int K, int MINB>
__global__ void __launch_bounds__(BWD_T, MINB) add_backward_streamed_kernel(BwdArgs a, BwdStreamArgs sa) {
    constexpr int P = BWD_T * K;
    __shared__ __align__(128) float s_raw[SB_STAGES][3 * SB_G];   // TMA destination: x | y | z of one tile
    __shared__ __align__(16) float s_g[3 * SB_G];                  // transformed tile: x | y | z
    __shared__ __align__(8) uint64_t s_bar[SB_STAGES];
    __shared__ double s_red[BWD_T / 32][12];
    __shared__ float s_rg[12];
    __shared__ int s_item, s_last;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < SB_STAGES; ++s) mbar_init(&s_bar[s], 1);
        fence_mbar_init();
    }
    uint32_t phases = 0;
    const int64_t total = static_cast<int64_t>(sa.nposes) * sa.nblk;

    for (;;) {
        if (tid == 0) s_item = atomicAdd(sa.counter, 1);
        __syncthreads();  // (A) also: the previous item's readers of shared memory are done
        const int64_t it = s_item;
        __syncthreads();  // every thread has read s_item
        if (it >= total) break;
        const int pi = static_cast<int>(it / sa.nblk), j = static_cast<int>(it % sa.nblk);
        const int64_t b = sa.first + pi;
        const int64_t oid = a.obj[b];
        if (!slot_known(oid, a.n_slots, a.slots)) {  // skipped sample: no gradient; CTA-uniform
            if (j == 0 && tid < 4) a.grad_q[4 * b + tid] = 0.0f;
            if (j == 0 && tid < 3) a.grad_t[3 * b + tid] = 0.0f;
            continue;
        }
        const SlotInfo s = a.slots[oid];
        const int n = s.count, np = s.padded, mode = s.xform_bmm;
        if (j * P >= n) continue;  // beyond this pose's mesh: not counted in its ticket
        const int items = (n + P - 1) / P;
        const float* mx = a.soa + s.soa_offset;
        const float* my = mx + np;
        const float* mz = my + np;
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

        // the item's pred points; nearest gt index per point (ADD: the same index)
        float px[K], py[K], pz[K], best[K], prev[K];
        int js[K];
        bool nan_seen[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int i = j * P + k * BWD_T + tid;
            const int ii = i < n ? i : 0;
            xform_point(mode, __ldg(mx + ii), __ldg(my + ii), __ldg(mz + ii), Rp, tp, px[k], py[k], pz[k]);
            best[k] = __int_as_float(0x7f800000);
            prev[k] = best[k];
            js[k] = s.symmetric ? 0 : ii;
            nan_seen[k] = false;
        }
        if (s.symmetric) {   // CTA-uniform
            if (tid == 0) {
#pragma unroll
                for (int k = 0; k < 9; ++k) s_rg[k] = Rg[k];
#pragma unroll
                for (int k = 0; k < 3; ++k) s_rg[9 + k] = tg[k];
            }
            const int ntiles = (n + SB_G - 1) / SB_G;
            auto issue = [&](int t) {  // one elected thread: tile t into its ring slot
                const int st = t % SB_STAGES;
                const int c = min(SB_G, np - t * SB_G);  // multiple of 4 floats: 16-byte segments
                const uint32_t bytes = static_cast<uint32_t>(c) * sizeof(float);
                mbar_arrive_expect_tx(&s_bar[st], 3 * bytes);
                tma_bulk_g2s(s_raw[st], mx + t * SB_G, bytes, &s_bar[st]);
                tma_bulk_g2s(s_raw[st] + SB_G, my + t * SB_G, bytes, &s_bar[st]);
                tma_bulk_g2s(s_raw[st] + 2 * SB_G, mz + t * SB_G, bytes, &s_bar[st]);
            };
            if (tid == 0) {
                fence_proxy_async();
                for (int t = 0; t < SB_STAGES && t < ntiles; ++t) issue(t);
            }
            for (int t = 0; t < ntiles; ++t) {
                const int st = t % SB_STAGES;
                mbar_wait(&s_bar[st], (phases >> st) & 1u);
                phases ^= 1u << st;
                __syncthreads();  // (T1) the previous tile's scan is done with s_g; s_rg is visible
                const int tn = min(SB_G, n - t * SB_G);
                for (int i = tid; i < tn; i += BWD_T)
                    xform_point(mode, s_raw[st][i], s_raw[st][SB_G + i], s_raw[st][2 * SB_G + i], s_rg, s_rg + 9,
                                s_g[i], s_g[SB_G + i], s_g[2 * SB_G + i]);
                __syncthreads();  // (T2) s_g is complete and s_raw[st] is consumed
                if (tid == 0 && t + SB_STAGES < ntiles) {
                    fence_proxy_async();
                    issue(t + SB_STAGES);
                }
                // add_backward_kernel's scan, continued: the first index with the smallest square, the minimum
                // before it in prev, and the first NaN, which ends the search
                const int j0 = t * SB_G;
#pragma unroll 1
                for (int jj = 0; jj < tn; ++jj) {
                    const float gx = s_g[jj], gy = s_g[SB_G + jj], gz = s_g[2 * SB_G + jj];
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        const float sv = sq3(__fsub_rn(px[k], gx), __fsub_rn(py[k], gy), __fsub_rn(pz[k], gz));
                        if (sv != sv && !nan_seen[k]) { nan_seen[k] = true; js[k] = j0 + jj; best[k] = sv; }
                        if (!nan_seen[k] && sv < best[k]) { prev[k] = best[k]; best[k] = sv; js[k] = j0 + jj; }
                    }
                }
            }
            // the rooted tie rule of add_backward_kernel: an earlier point whose square is larger but whose sqrt
            // equals sqrt(best) is the nearest one; there is none unless sqrt(prev) == sqrt(best).  The earlier
            // tiles are gone, so the (rare) rescan of [0, js) re-transforms the gt points from the mesh.
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (!nan_seen[k] && js[k] > 0 && __fsqrt_rn(prev[k]) == __fsqrt_rn(best[k])) {
                    const float r = __fsqrt_rn(best[k]);
                    for (int jj = 0; jj < js[k]; ++jj) {
                        float gx, gy, gz;
                        xform_point(mode, __ldg(mx + jj), __ldg(my + jj), __ldg(mz + jj), Rg, tg, gx, gy, gz);
                        if (__fsqrt_rn(sq3(__fsub_rn(px[k], gx), __fsub_rn(py[k], gy), __fsub_rn(pz[k], gz))) == r) {
                            js[k] = jj;
                            break;
                        }
                    }
                }
            }
        }

        double acc[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) acc[k] = 0.0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int i = j * P + k * BWD_T + tid;
            if (i < n) {
                // the gt point of index js[k], with the rounding of the tiles (add_backward_kernel's G and sums)
                float gx, gy, gz;
                xform_point(mode, __ldg(mx + js[k]), __ldg(my + js[k]), __ldg(mz + js[k]), Rg, tg, gx, gy, gz);
                const float dx = __fsub_rn(px[k], gx), dy = __fsub_rn(py[k], gy), dz = __fsub_rn(pz[k], gz);
                const float d = __fsqrt_rn(sq3(dx, dy, dz));
                float G[3] = {0.0f, 0.0f, 0.0f};
                if (d != 0.0f) { G[0] = __fdiv_rn(dx, d); G[1] = __fdiv_rn(dy, d); G[2] = __fdiv_rn(dz, d); }
                const float m[3] = {__ldg(mx + i), __ldg(my + i), __ldg(mz + i)};
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    acc[r] += (double)G[r];
#pragma unroll
                    for (int c = 0; c < 3; ++c) acc[3 + 3 * r + c] += (double)G[r] * (double)m[c];  // dL/dR[r][c]
                }
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
        double* part = sa.part + (static_cast<size_t>(pi) * sa.nblk + j) * 12;
        if (tid < 12) {
            double v = 0.0;
            for (int w = 0; w < BWD_T / 32; ++w) v += s_red[w][tid];
            part[tid] = v;
        }
        // the last item of the pose sums the items' partials in item order
        __threadfence();
        __syncthreads();
        if (tid == 0) s_last = atomicAdd(sa.tickets + pi, 1) == items - 1;
        __syncthreads();
        if (s_last && tid == 0) {
            __threadfence();
            const double* p0 = sa.part + static_cast<size_t>(pi) * sa.nblk * 12;
            double t[12];
            for (int k = 0; k < 12; ++k) t[k] = 0.0;
            for (int e = 0; e < items; ++e)
                for (int k = 0; k < 12; ++k) t[k] += __ldcg(p0 + 12 * e + k);
            bwd_pose_tail(a, b, q, n, t);
        }
    }
}

struct SbShape {
    const void* fn;
    int k;
};
static const SbShape kSbShapes[3] = {   // widest first
    {(const void*)add_backward_streamed_kernel<4, 2>, 4},
    {(const void*)add_backward_streamed_kernel<2, 3>, 2},
    {(const void*)add_backward_streamed_kernel<1, 3>, 1},
};

static int launch_backward_streamed(const p6d_mesh_table* t, const BwdArgs& args, cudaStream_t st) {
    const int nmax = t->max_count > 0 ? t->max_count : 1;
    // the widest shape whose items fill the device at least twice; the narrowest otherwise
    int pick = 2, per_sm_pick = 1;
    for (int si = 0; si < 3; ++si) {
        int per_sm = 0;
        int rc = ctas_per_sm(kSbShapes[si].fn, BWD_T, t->device, 0, &per_sm);
        if (rc) return rc;
        const int P = BWD_T * kSbShapes[si].k;
        if (args.B * ((nmax + P - 1) / P) >= 2 * static_cast<int64_t>(t->sm_count) * per_sm || si == 2) {
            pick = si;
            per_sm_pick = per_sm;
            break;
        }
    }
    const SbShape& shape = kSbShapes[pick];
    const int P = BWD_T * shape.k;
    const int nblk = (nmax + P - 1) / P;
    const size_t per_pose = sizeof(double) * 12 * static_cast<size_t>(nblk) + sizeof(int);
    const int64_t bc = std::max<int64_t>(1, std::min<int64_t>(args.B, static_cast<int64_t>(SB_WS_BYTES / per_pose)));
    const size_t head = 16 + (sizeof(int) * static_cast<size_t>(bc) + 15) / 16 * 16;
    const size_t ws_bytes = head + sizeof(double) * 12 * static_cast<size_t>(nblk) * static_cast<size_t>(bc);

    char* ws = nullptr;
    P6D_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), ws_bytes, st));
    int rc = P6D_OK;
    for (int64_t c0 = 0; c0 < args.B && rc == P6D_OK; c0 += bc) {
        const int64_t nc = std::min<int64_t>(bc, args.B - c0);
        BwdStreamArgs sa;
        sa.first = c0;
        sa.nposes = static_cast<int>(nc);
        sa.nblk = nblk;
        sa.counter = reinterpret_cast<int*>(ws);
        sa.tickets = reinterpret_cast<int*>(ws + 16);
        sa.part = reinterpret_cast<double*>(ws + head);
        cudaError_t e = cudaMemsetAsync(ws, 0, 16 + sizeof(int) * static_cast<size_t>(nc), st);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemsetAsync(streamed backward workspace)"); break; }
        const int64_t grid = std::min<int64_t>(nc * nblk, static_cast<int64_t>(t->sm_count) * per_sm_pick);
        BwdArgs a = args;
        void* kargs[] = {&a, &sa};
        e = cudaLaunchKernel(shape.fn, dim3(static_cast<unsigned>(grid)), dim3(BWD_T), kargs, 0, st);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaLaunchKernel(add_backward_streamed_kernel)");
    }
    const cudaError_t ef = cudaFreeAsync(ws, st);
    if (rc == P6D_OK && ef != cudaSuccess) rc = cuda_fail(ef, "cudaFreeAsync(streamed backward workspace)");
    return rc;
}

// Every backward call picks its kernel here: the streamed kernel when forced, or when the table's large-mesh loss
// switch is on and the largest mesh is beyond the resident kernel's shared memory; the resident kernel otherwise.
static int launch_backward(const p6d_mesh_table* t, const BwdArgs& a, bool force_streamed, cudaStream_t st) {
    const int nmax = t->max_count > 0 ? t->max_count : 1;
    const size_t smem = sizeof(float) * 3 * (size_t)nmax;
    int limit = 0;
    int rc = max_optin_smem(t->device, &limit);
    if (rc) return rc;
    const bool fits = smem + 1024 <= (size_t)limit;
    if (force_streamed || (!fits && t->large_mesh_loss.load(std::memory_order_relaxed))) {
        if ((rc = check_streamed_size(t))) return rc;
        return launch_backward_streamed(t, a, st);
    }
    if (!fits) {
        set_error("p6d_add_backward: mesh of %d points does not fit shared memory", nmax);
        return P6D_ETOOBIG;
    }
    if ((rc = raise_dyn_smem((const void*)add_backward_kernel, t->device, smem))) return rc;
    int64_t grid = a.B < (int64_t)t->sm_count * 4 ? a.B : (int64_t)t->sm_count * 4;
    add_backward_kernel<<<(unsigned)grid, BWD_T, smem, st>>>(a, nmax);
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

}  // namespace p6d

using namespace p6d;

static int backward_entry(bool streamed, const p6d_mesh_table* table, const float* pq, const float* pt,
                          const float* gq, const float* gt, const int64_t* obj, int64_t B, const float* grad_out,
                          const int32_t* count, float inv_count, float* grad_q, float* grad_t, void* stream) {
    if (!table || B < 0 || (B > 0 && (!pq || !pt || !gq || !gt || !obj || !grad_out || !grad_q || !grad_t))) {
        set_error("%s: bad arguments", streamed ? "p6d_add_backward_streamed" : "p6d_add_backward");
        return P6D_EINVAL;
    }
    if (B == 0) return P6D_OK;
    DeviceGuard guard(table->device);
    if (!guard.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice");
    BwdArgs a{table->d_soa, table->d_slots, table->n_slots, pq, pt, gq, gt, obj, B, grad_out, count, inv_count, grad_q, grad_t};
    return launch_backward(table, a, streamed, static_cast<cudaStream_t>(stream));
}

extern "C" int p6d_add_backward(const p6d_mesh_table* table, const float* pq, const float* pt, const float* gq,
                                const float* gt, const int64_t* obj, int64_t B, const float* grad_out,
                                const int32_t* count, float inv_count, float* grad_q, float* grad_t, void* stream) {
    return backward_entry(false, table, pq, pt, gq, gt, obj, B, grad_out, count, inv_count, grad_q, grad_t, stream);
}

extern "C" int p6d_add_backward_streamed(const p6d_mesh_table* table, const float* pq, const float* pt,
                                         const float* gq, const float* gt, const int64_t* obj, int64_t B,
                                         const float* grad_out, const int32_t* count, float inv_count, float* grad_q,
                                         float* grad_t, void* stream) {
    return backward_entry(true, table, pq, pt, gq, gt, obj, B, grad_out, count, inv_count, grad_q, grad_t, stream);
}
