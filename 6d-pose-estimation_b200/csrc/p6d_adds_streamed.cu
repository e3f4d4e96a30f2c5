// p6d_adds_streamed.cu -- kernel (b''): ADD / ADD-S for meshes larger than shared memory (opt-in), sm_100a.
//
// The resident kernels (b) and (a) stage the whole mesh in shared memory and refuse a table whose largest mesh
// does not fit (about 7,150 points for ADD-S, 16,700 for ADD only).  This kernel streams the gt cloud through
// shared memory in tiles instead, so the mesh size is bounded by the arithmetic contract, not by a buffer:
//
//   work item  = (pose, block of P = 256 * K pred points); items of one pose are consecutive and claimed through
//                an atomic counter by a persistent grid.  K = 8 (the register shape of the large-mesh resident
//                variant) when a launch has enough items to fill the device, K = 4 or 2 for small batches;
//   pred side  = the item's P mesh points, transformed by the pred pose into registers (quat_to_mat, xform_point
//                with the slot's torch.mm rounding), plus the gt point of the same index for the ADD distance;
//   gt side    = tiles of G = 1,024 mesh points arrive by TMA bulk copies (x, y, z segments of the table's SoA
//                block) in a two-stage mbarrier ring, are transformed by the gt pose into the quad layout of
//                kernel (b) (padded with GT_SENTINEL) and scanned with its packed step (3 FADD2 + FMUL2 + 2 FFMA2 +
//                FMNMX3.NAN per two pairs).  The gt cloud is re-transformed per item: 18 FLOP per gt point against
//                8 * P per gt point of scan, so nothing per pose goes through global memory;
//   finish     = sqrt of each row minimum (sqrt is monotone and correctly rounded, and min is exact and
//                NaN-propagating, so neither the tiling nor the split into items changes a bit), both per-point
//                rows to a workspace; the last item of a pose (per-pose ticket after __threadfence) computes the
//                two ATen-ordered means, the float64 decision, `near_threshold` and the accumulators exactly as
//                phase D of adds_cta_kernel.
// The workspace (8 bytes per point and pose, plus tickets) is allocated stream-ordered on the caller's stream and
// the batch is launched in chunks that keep it within 64 MB, so two streams never share a buffer.
#include <algorithm>

#include "p6d_common.cuh"

namespace p6d {

constexpr int ST_T = 256;                  // threads per CTA
constexpr int ST_G = 1024;                 // gt points per tile (multiple of 8)
constexpr int ST_STAGES = 2;               // TMA ring depth
constexpr int ST_MAX_POINTS = 32768;       // see the refusal message in launch_eval_streamed
constexpr size_t ST_WS_BYTES = size_t(64) << 20;

struct StreamArgs {
    int64_t first;      // first pose of the chunk in processing order
    int nposes;         // poses in the chunk
    int nblk;           // items per pose of the table's largest mesh (poses of smaller meshes use fewer)
    int stride;         // floats per per-point row in the workspace
    int* counter;       // work counter (zeroed before the launch)
    int* tickets;       // [nposes] finished items per pose (zeroed before the launch)
    float* rows;        // [nposes][2][stride]: ADD row, ADD-S row
};

template <int K, int MINB, bool ADDS>
__global__ void __launch_bounds__(ST_T, MINB) adds_streamed_kernel(EvalArgs a, StreamArgs sa) {
    constexpr int P = ST_T * K;
    __shared__ __align__(128) float s_raw[ST_STAGES][3 * ST_G];   // TMA destination: x | y | z of one tile
    __shared__ __align__(128) float s_quad[3 * ST_G];              // transformed tile as quads (48 B per 4 points)
    __shared__ __align__(8) uint64_t s_bar[ST_STAGES];
    __shared__ float s_pose[14];
    __shared__ float s_rg[12];                                    // gt rotation and translation of the item's pose
    __shared__ float s_mean[2];
    __shared__ long long s_oid;
    __shared__ int s_item, s_last;

    const int tid = threadIdx.x, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < ST_STAGES; ++s) mbar_init(&s_bar[s], 1);
        fence_mbar_init();
    }
    uint32_t phases = 0;
    const int64_t total = static_cast<int64_t>(sa.nposes) * sa.nblk;

    for (;;) {
        if (tid == 0) s_item = atomicAdd(sa.counter, 1);
        __syncthreads();  // (A) also: the previous item's readers of shared memory are done
        const int64_t it = s_item;
        if (it >= total) break;
        const int pi = static_cast<int>(it / sa.nblk), j = static_cast<int>(it % sa.nblk);
        const int64_t idx = sa.first + pi;
        const int64_t b = a.order ? a.order[idx] : idx;
        load_pose(a, b, tid, s_pose, &s_oid);
        __syncthreads();  // (B) also: every thread has read s_item
        const long long oid = s_oid;
        if (!slot_known(oid, a.n_slots, a.slots)) {  // CTA-uniform; the first item of the pose writes its outputs
            if (tid == 0 && j == 0) write_skipped(a, b, ADDS);
            continue;
        }
        const SlotInfo s = a.slots[oid];
        const int n = s.count, np = s.padded, mode = s.xform_mode;
        if (j * P >= n) continue;  // beyond this pose's mesh: not counted in its ticket
        const int items = (n + P - 1) / P;
        const float* msh = a.soa + s.soa_offset;
        float* row_add = sa.rows + static_cast<size_t>(pi) * 2 * sa.stride;
        float* row_adds = row_add + sa.stride;

        // pred points of the item into registers; ADD distances of the same indices
        float px[K], py[K], pz[K], m[K];
        {
            float Rp[9], Rg[9], tp[3], tg[3];
            quat_to_mat(s_pose, Rp);
            quat_to_mat(s_pose + 4, Rg);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                tp[k] = s_pose[8 + k];
                tg[k] = s_pose[11 + k];
            }
            if (ADDS && tid == 0) {
#pragma unroll
                for (int k = 0; k < 9; ++k) s_rg[k] = Rg[k];
#pragma unroll
                for (int k = 0; k < 3; ++k) s_rg[9 + k] = tg[k];
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int i = j * P + k * ST_T + tid;
                const int ii = i < n ? i : 0;
                const float x = __ldg(msh + ii), y = __ldg(msh + np + ii), z = __ldg(msh + 2 * np + ii);
                xform_point(mode, x, y, z, Rp, tp, px[k], py[k], pz[k]);
                if (i < n) {
                    float qx, qy, qz;
                    xform_point(mode, x, y, z, Rg, tg, qx, qy, qz);
                    row_add[i] = __fsqrt_rn(sq3(__fsub_rn(px[k], qx), __fsub_rn(py[k], qy), __fsub_rn(pz[k], qz)));
                }
                m[k] = __int_as_float(0x7f800000);  // +inf
            }
        }

        if (ADDS) {
            const int ntiles = (n + ST_G - 1) / ST_G;
            auto issue = [&](int t) {  // one elected thread: tile t into its ring slot
                const int st = t % ST_STAGES;
                const int c = min(ST_G, np - t * ST_G);  // multiple of 4 floats: 16-byte segments
                const uint32_t bytes = static_cast<uint32_t>(c) * sizeof(float);
                mbar_arrive_expect_tx(&s_bar[st], 3 * bytes);
                tma_bulk_g2s(s_raw[st], msh + t * ST_G, bytes, &s_bar[st]);
                tma_bulk_g2s(s_raw[st] + ST_G, msh + np + t * ST_G, bytes, &s_bar[st]);
                tma_bulk_g2s(s_raw[st] + 2 * ST_G, msh + 2 * np + t * ST_G, bytes, &s_bar[st]);
            };
            if (tid == 0) {
                fence_proxy_async();
                for (int t = 0; t < ST_STAGES && t < ntiles; ++t) issue(t);
            }
            for (int t = 0; t < ntiles; ++t) {
                const int st = t % ST_STAGES;
                mbar_wait(&s_bar[st], (phases >> st) & 1u);
                phases ^= 1u << st;
                __syncthreads();  // (T1) the previous tile's scan is done with s_quad; s_rg is visible
                const int tn = min(ST_G, n - t * ST_G);
                const int tq = (tn + 7) & ~7;  // two quads per scan trip
                for (int i = tid; i < tq; i += ST_T) {
                    float* gq = s_quad + (i >> 2) * 12 + (i & 3);
                    if (i < tn) {
                        float qx, qy, qz;
                        xform_point(mode, s_raw[st][i], s_raw[st][ST_G + i], s_raw[st][2 * ST_G + i], s_rg, s_rg + 9,
                                    qx, qy, qz);
                        gq[0] = qx;
                        gq[4] = qy;
                        gq[8] = qz;
                    } else {
                        gq[0] = GT_SENTINEL;
                        gq[4] = GT_SENTINEL;
                        gq[8] = GT_SENTINEL;
                    }
                }
                __syncthreads();  // (T2) s_quad is complete and s_raw[st] is consumed
                if (tid == 0 && t + ST_STAGES < ntiles) {
                    fence_proxy_async();
                    issue(t + ST_STAGES);
                }
                const float4* p = reinterpret_cast<const float4*>(s_quad);
                const float4* const pend = p + 3 * (tq >> 2);
#pragma unroll 1
                for (; p < pend; p += 6) {
                    const float4 X0 = p[0], Y0 = p[1], Z0 = p[2], X1 = p[3], Y1 = p[4], Z1 = p[5];
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        pair_tile(px[k], py[k], pz[k], make_float2(X0.x, X0.y), make_float2(Y0.x, Y0.y),
                                  make_float2(Z0.x, Z0.y), m[k]);
                        pair_tile(px[k], py[k], pz[k], make_float2(X0.z, X0.w), make_float2(Y0.z, Y0.w),
                                  make_float2(Z0.z, Z0.w), m[k]);
                        pair_tile(px[k], py[k], pz[k], make_float2(X1.x, X1.y), make_float2(Y1.x, Y1.y),
                                  make_float2(Z1.x, Z1.y), m[k]);
                        pair_tile(px[k], py[k], pz[k], make_float2(X1.z, X1.w), make_float2(Y1.z, Y1.w),
                                  make_float2(Z1.z, Z1.w), m[k]);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int i = j * P + k * ST_T + tid;
                // sqrt is monotone and correctly rounded: sqrt(min s) == min sqrt(s)
                if (i < n) row_adds[i] = __fsqrt_rn(m[k]);
            }
        }

        // the last item of the pose to finish computes the means
        __threadfence();
        __syncthreads();
        if (tid == 0) s_last = atomicAdd(sa.tickets + pi, 1) == items - 1;
        __syncthreads();
        if (!s_last) continue;
        __threadfence();
        if (tid < (ADDS ? 64 : 32)) {
            ordered_means(row_add, row_adds, n, tid, lane, ADDS, s_mean, [](const float* p) { return __ldcg(p); });
            if (tid == 0) write_pose(a, b, oid, s, s_mean[0], ADDS ? s_mean[1] : 0.0f, ADDS);
        }
    }
}

struct StShape {
    const void* fn;
    int k;
};
// per ADD-S flag, widest first
static const StShape kStShapes[2][3] = {
    {{(const void*)adds_streamed_kernel<8, 2, false>, 8},
     {(const void*)adds_streamed_kernel<4, 4, false>, 4},
     {(const void*)adds_streamed_kernel<2, 4, false>, 2}},
    {{(const void*)adds_streamed_kernel<8, 2, true>, 8},
     {(const void*)adds_streamed_kernel<4, 4, true>, 4},
     {(const void*)adds_streamed_kernel<2, 4, true>, 2}},
};

int launch_eval_streamed(const p6d_mesh_table* t, const EvalArgs& args, bool want_adds, cudaStream_t st) {
    if (t->max_count > ST_MAX_POINTS) {
        set_error("largest mesh has %d points; the streamed ADD/ADD-S kernel accepts at most %d points: above that, "
                  "torch's CPU Tensor.mean() splits a row across threads, so the reference's own result depends on "
                  "the caller's thread count and there is no single result to reproduce",
                  t->max_count, ST_MAX_POINTS);
        return P6D_ETOOBIG;
    }
    if (args.B == 0) return P6D_OK;
    const int nmax = t->max_count > 0 ? t->max_count : 1;
    const int stride = (nmax + 3) / 4 * 4;
    const size_t per_pose = 2 * sizeof(float) * static_cast<size_t>(stride) + sizeof(int);
    const int64_t bc = std::max<int64_t>(1, std::min<int64_t>(args.B, static_cast<int64_t>(ST_WS_BYTES / per_pose)));
    const size_t tickets_bytes = (sizeof(int) * static_cast<size_t>(bc) + 15) / 16 * 16;
    const size_t head = 16 + tickets_bytes;
    const size_t ws_bytes = head + 2 * sizeof(float) * static_cast<size_t>(stride) * static_cast<size_t>(bc);

    // the widest shape whose items fill the device at least twice; the narrowest otherwise
    const int ai = want_adds ? 1 : 0;
    int pick = 2, per_sm_pick = 1;
    for (int si = 0; si < 3; ++si) {
        int per_sm = 0;
        int rc = ctas_per_sm(kStShapes[ai][si].fn, ST_T, t->device, 0, &per_sm);
        if (rc) return rc;
        const int P = ST_T * kStShapes[ai][si].k;
        const int64_t items = bc * ((nmax + P - 1) / P);
        if (items >= 2 * static_cast<int64_t>(t->sm_count) * per_sm || si == 2) {
            pick = si;
            per_sm_pick = per_sm;
            break;
        }
    }
    const StShape& shape = kStShapes[ai][pick];
    const int P = ST_T * shape.k;
    const int nblk = (nmax + P - 1) / P;

    char* ws = nullptr;
    P6D_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), ws_bytes, st));
    int rc = P6D_OK;
    for (int64_t c0 = 0; c0 < args.B && rc == P6D_OK; c0 += bc) {
        const int64_t nc = std::min<int64_t>(bc, args.B - c0);
        StreamArgs sa;
        sa.first = c0;
        sa.nposes = static_cast<int>(nc);
        sa.nblk = nblk;
        sa.stride = stride;
        sa.counter = reinterpret_cast<int*>(ws);
        sa.tickets = reinterpret_cast<int*>(ws + 16);
        sa.rows = reinterpret_cast<float*>(ws + head);
        cudaError_t e = cudaMemsetAsync(ws, 0, 16 + sizeof(int) * static_cast<size_t>(nc), st);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemsetAsync(streamed workspace)"); break; }
        const int64_t items = nc * nblk;
        const int64_t grid = std::min<int64_t>(items, static_cast<int64_t>(t->sm_count) * per_sm_pick);
        EvalArgs a = args;
        void* kargs[] = {&a, &sa};
        e = cudaLaunchKernel(shape.fn, dim3(static_cast<unsigned>(grid)), dim3(ST_T), kargs, 0, st);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaLaunchKernel(adds_streamed_kernel)");
    }
    const cudaError_t ef = cudaFreeAsync(ws, st);
    if (rc == P6D_OK && ef != cudaSuccess) rc = cuda_fail(ef, "cudaFreeAsync(streamed workspace)");
    return rc;
}

}  // namespace p6d
