// p6d_adds_pruned.cu -- kernel (b'): ADD + ADD-S with EXACT block pruning (opt-in), sm_100a.
//
// Same outputs, bit for bit, as the all-pairs kernel (b) of p6d_add.cu -- the kernel BASELINE's north-star names
// and the one every headline number is measured on.  This one skips gt points that provably cannot be the
// nearest neighbour and is reported separately (bench.py "pruned"), never as a roofline fraction: it does less
// work, it does not do the same work faster.
//
// ADD-S = mean_i min_j |pred_i - gt_j| (reference models/add_loss.py:185-190).  Only the minimum of every row has
// to be exact; any pair that is provably not below the current minimum may be skipped.  Both clouds are the SAME
// mesh under two rigid (or at least linear) maps, so the mesh is cut ONCE, at table creation, into spatially
// compact blocks of 32 points, each made of four compact sub-blocks of 8 (k-d median splits, points stored
// block-sorted with the permutation back to the original index).  A pred block is the 32 points of a warp; the
// gt cloud is skipped in sub-blocks of 8 (two quads): the pair work left over goes with (rA + rB + d)^2, so the
// smaller gt spheres save ~40 % of it against 32-point gt blocks.  Per pose:
//   B'  one warp per block: lane l transforms point l of the block by both poses (the very xform_point calls of
//       kernel (b): same coordinates, bit for bit), writes the gt cloud (quads) and the pred cloud to shared
//       memory, the ADD distance at the ORIGINAL index, and the bounding spheres -- of the pred block and of the
//       four gt sub-blocks: centre = the transformed model-space centroid, radius = the largest distance of an
//       actual transformed point to it (no assumption about R being orthonormal -- _quat_to_mat does not normalise);
//   C'  one warp per pred block A, one pred point per lane: the same-index gt block first (for a prediction
//       anywhere near the truth that is where the neighbours are), then every lane tests one other gt sub-block B,
//       |cA - cB| >= sqrt(max_i m_i) + rA + rB   (with margins far above the float32 error of either side:
//       1e-4 relative against < 1e-6), and the warp evaluates the blocks that are left.  A skipped block holds no
//       pair with  s_ij < m_i  for any lane, and m_i only decreases, so the final minimum is the all-pairs minimum.
//       Anything that is not a number fails the test and is evaluated: NaN propagates exactly as in kernel (b);
//   D   ordered means (ATen order), decision, outputs: as in kernel (b).
// The squared distance of a pair is computed by the same packed instructions in the same order as kernel (b)
// (3 FADD2, FMUL2, 2 FFMA2, FMNMX3.NAN), so every surviving value has the same bits.
#include <algorithm>
#include <memory>
#include <vector>

#include "p6d_common.cuh"

namespace p6d {

constexpr int PR_BLOCK = 32;              // points per block = lanes per warp
constexpr int PR_SUB = 8;                 // points per gt sub-block (two quads)

// per-object description of the block-sorted copy of the mesh (device + host)
struct PrunedSlot {
    int64_t offset;     // first float of the object's block in the sorted buffer
    int32_t nb;         // blocks
    int32_t floats;     // size of the block (multiple of 4)
};
// layout of one object's block (floats), Np = 32 * nb, nbp = nb rounded up to 4:
//   x[Np] y[Np] z[Np]   block-sorted coordinates (padding of the last block repeats its first point)
//   cx[nbp] cy[nbp] cz[nbp]   model-space centroid of every block
//   sx[4 nb] sy[4 nb] sz[4 nb]   model-space centroid of every sub-block
//   perm[Np] as uint16  original index of sorted position p (0xffff = padding)
__host__ __device__ inline int pr_floats(int nb) {
    const int np = PR_BLOCK * nb, nbp = (nb + 3) / 4 * 4;
    return 3 * np + 3 * nbp + 12 * nb + np / 2;
}

struct PrunedTable {
    float* d_sorted = nullptr;
    PrunedSlot* d_slots = nullptr;
    std::vector<PrunedSlot> h_slots;
    int max_nb = 0;
    int max_count = 0;
};

// k-d median splits: idx[lo, hi) -> blocks of 32 consecutive entries made of sub-blocks of 8, each spatially compact
static void kd_split(const float* xyz, std::vector<int>& idx, int lo, int hi) {
    if (hi - lo <= PR_SUB) return;
    const int unit = hi - lo > PR_BLOCK ? PR_BLOCK : PR_SUB;
    float mn[3] = {1e30f, 1e30f, 1e30f}, mx[3] = {-1e30f, -1e30f, -1e30f};
    for (int i = lo; i < hi; ++i)
        for (int c = 0; c < 3; ++c) {
            const float v = xyz[3 * idx[i] + c];
            if (v < mn[c]) mn[c] = v;
            if (v > mx[c]) mx[c] = v;
        }
    int axis = 0;
    for (int c = 1; c < 3; ++c)
        if (mx[c] - mn[c] > mx[axis] - mn[axis]) axis = c;
    const int blocks = (hi - lo + unit - 1) / unit;
    const int mid = lo + (blocks + 1) / 2 * unit;         // a multiple of 32 (8) from lo: (sub-)blocks never straddle a split
    auto key = [&](int i) { const float v = xyz[3 * i + axis]; return v == v ? v : 3.0e38f; };   // NaN sorts last
    std::nth_element(idx.begin() + lo, idx.begin() + mid, idx.begin() + hi, [&](int a, int b) {
        const float va = key(a), vb = key(b);
        return va < vb || (va == vb && a < b);
    });
    kd_split(xyz, idx, lo, mid);
    kd_split(xyz, idx, mid, hi);
}

static PrunedTable* build_blocks(const p6d_mesh_table* t, const float* xyz, const int32_t* offsets) {
    std::unique_ptr<PrunedTable> pt(new PrunedTable());     // freed if anything below throws
    pt->h_slots.resize(t->n_slots);
    size_t total = 0;
    for (int s = 0; s < t->n_slots; ++s) {
        const int n = t->h_slots[s].count;
        PrunedSlot& ps = pt->h_slots[s];
        ps.nb = (n + PR_BLOCK - 1) / PR_BLOCK;
        ps.floats = pr_floats(ps.nb);
        ps.offset = static_cast<int64_t>(total);
        total += static_cast<size_t>(ps.floats);
        pt->max_nb = std::max(pt->max_nb, ps.nb);
        pt->max_count = std::max(pt->max_count, n);
    }
    std::vector<float> buf(total > 0 ? total : 4, 0.0f);
    for (int s = 0; s < t->n_slots; ++s) {
        const int n = t->h_slots[s].count;
        if (n == 0) continue;
        const PrunedSlot& ps = pt->h_slots[s];
        const float* src = xyz + 3 * static_cast<size_t>(offsets[s]);
        std::vector<int> idx(n);
        for (int i = 0; i < n; ++i) idx[i] = i;
        kd_split(src, idx, 0, n);
        const int np = PR_BLOCK * ps.nb, nbp = (ps.nb + 3) / 4 * 4;
        float* x = buf.data() + ps.offset;
        float* cen = x + 3 * np;
        float* sub = cen + 3 * nbp;
        const int ns = 4 * ps.nb;
        uint16_t* perm = reinterpret_cast<uint16_t*>(sub + 3 * ns);
        for (int b = 0; b < ps.nb; ++b) {
            double c[3] = {0.0, 0.0, 0.0};
            const int cnt = std::min(PR_BLOCK, n - PR_BLOCK * b);
            for (int l = 0; l < PR_BLOCK; ++l) {
                const int p = PR_BLOCK * b + l;
                const int i = idx[l < cnt ? p : PR_BLOCK * b];       // padding repeats the block's first point
                for (int k = 0; k < 3; ++k) x[k * np + p] = src[3 * i + k];
                perm[p] = l < cnt ? static_cast<uint16_t>(i) : 0xffffu;
                if (l < cnt)
                    for (int k = 0; k < 3; ++k) c[k] += src[3 * i + k];
            }
            for (int k = 0; k < 3; ++k) cen[k * nbp + b] = static_cast<float>(c[k] / cnt);
            for (int q = 0; q < PR_BLOCK / PR_SUB; ++q) {
                double sc[3] = {0.0, 0.0, 0.0};
                const int first = PR_BLOCK * b + PR_SUB * q;
                const int scnt = std::max(0, std::min(PR_SUB, n - first));
                for (int l = 0; l < scnt; ++l)
                    for (int k = 0; k < 3; ++k) sc[k] += x[k * np + first + l];
                // an empty sub-block (padding only) takes the block's first point: its sphere has radius 0
                for (int k = 0; k < 3; ++k)
                    sub[k * ns + 4 * b + q] = scnt > 0 ? static_cast<float>(sc[k] / scnt) : x[k * np + PR_BLOCK * b];
            }
        }
    }
    if (cudaMalloc(&pt->d_sorted, buf.size() * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&pt->d_slots, t->n_slots * sizeof(PrunedSlot)) != cudaSuccess ||
        cudaMemcpy(pt->d_sorted, buf.data(), buf.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(pt->d_slots, pt->h_slots.data(), t->n_slots * sizeof(PrunedSlot), cudaMemcpyHostToDevice) !=
            cudaSuccess) {
        cudaGetLastError();
        if (pt->d_sorted) cudaFree(pt->d_sorted);
        if (pt->d_slots) cudaFree(pt->d_slots);
        return nullptr;
    }
    return pt.release();
}

// Called by p6d_mesh_table_create once the table is complete.  Null (no block structure) for a mesh of more than
// 65,534 points, or out of memory: not fatal for the table, the pruned kernel is just not available.
PrunedTable* build_pruned(const p6d_mesh_table* t, const float* xyz, const int32_t* offsets) {
    if (t->max_count > 65534) return nullptr;    // permutation is stored as uint16
    try {
        return build_blocks(t, xyz, offsets);
    } catch (...) {                              // out of host memory
        return nullptr;
    }
}

void free_pruned(PrunedTable* pt) {
    if (!pt) return;
    cudaFree(pt->d_sorted);
    cudaFree(pt->d_slots);
    delete pt;
}

struct PrunedArgs {
    const float* sorted;
    const PrunedSlot* pslots;
};

// shared memory (floats) for a table whose largest mesh has nb blocks:  staged block | gt quads | pred SoA |
// dadd | dadds | pred spheres | gt spheres
__host__ __device__ inline size_t pr_smem_floats(int nb, int nmax) {
    const int np = PR_BLOCK * nb;
    return static_cast<size_t>(pr_floats(nb)) + 3 * np + 3 * np + 2 * static_cast<size_t>((nmax + 3) / 4 * 4) + 4 * nb + 16 * nb;
}

// one gt block (8 quads) against the lane's pred point
__device__ __forceinline__ float eval_block(const float4* __restrict__ q, float px, float py, float pz, float m) {
    float m2 = __int_as_float(0x7f800000);
#pragma unroll
    for (int k = 0; k < PR_BLOCK / 4; ++k) {
        const float4 X = q[3 * k], Y = q[3 * k + 1], Z = q[3 * k + 2];
        pair_tile(px, py, pz, make_float2(X.x, X.y), make_float2(Y.x, Y.y), make_float2(Z.x, Z.y), m);
        pair_tile(px, py, pz, make_float2(X.z, X.w), make_float2(Y.z, Y.w), make_float2(Z.z, Z.w), m2);
    }
    return min_nan(m, m2);
}

// one gt sub-block (2 quads) against the lane's pred point
__device__ __forceinline__ float eval_sub(const float4* __restrict__ q, float px, float py, float pz, float m) {
    float m2 = __int_as_float(0x7f800000);
#pragma unroll
    for (int k = 0; k < PR_SUB / 4; ++k) {
        const float4 X = q[3 * k], Y = q[3 * k + 1], Z = q[3 * k + 2];
        pair_tile(px, py, pz, make_float2(X.x, X.y), make_float2(Y.x, Y.y), make_float2(Z.x, Z.y), m);
        pair_tile(px, py, pz, make_float2(X.z, X.w), make_float2(Y.z, Y.w), make_float2(Z.z, Z.w), m2);
    }
    return min_nan(m, m2);
}

// two gt sub-blocks at once: twice the independent chains for the same instructions (the candidate loop is serial
// in m otherwise, and at 2 CTAs per SM there are only 4 warps per scheduler to hide it)
__device__ __forceinline__ float eval_two(const float4* __restrict__ q0, const float4* __restrict__ q1, float px, float py,
                                          float pz, float m) {
    const float a = eval_sub(q0, px, py, pz, m);
    const float b = eval_sub(q1, px, py, pz, __int_as_float(0x7f800000));
    return min_nan(a, b);
}

// T threads per CTA = one pose per T threads; MINB = CTAs per SM the register budget is sized for.  Instantiations
// (see launch_eval_pruned): <256,2> (<= 128 registers) where shared memory admits two CTAs (2,048 points), <256,3>,
// <256,4> (64 registers) below that, and <128,8> for meshes of <= 512 points: 16 blocks give a 256-thread CTA two
// blocks per warp, and with three CTA barriers per pose ncu showed `barrier` as its top stall (2.7 warps per issue
// cycle); half the CTA, twice the poses in flight.
template <int T, int MINB>
__global__ void __launch_bounds__(T, MINB) adds_pruned_kernel(EvalArgs a, PrunedArgs pa, int nb_max, int nmax) {
    constexpr int PR_WARPS = T / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int np_max = PR_BLOCK * nb_max;
    float* s_sorted = reinterpret_cast<float*>(smem_raw);
    float* s_gt = s_sorted + pr_floats(nb_max);
    float* s_pred = s_gt + 3 * np_max;
    float* s_dadd = s_pred + 3 * np_max;
    float* s_dadds = s_dadd + (nmax + 3) / 4 * 4;
    float4* s_cp = reinterpret_cast<float4*>(s_dadds + (nmax + 3) / 4 * 4);
    float4* s_cg = s_cp + nb_max;                // gt spheres, one per sub-block: [4 * nb_max]
    __shared__ uint64_t s_bar;
    __shared__ float s_pose[14];
    __shared__ float s_mean[2];
    __shared__ long long s_oid;
    __shared__ int s_next;
    __shared__ int s_blk[2];    // pred blocks of phase C' are claimed warp by warp (double-buffered across poses)

    const unsigned full = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        mbar_init(&s_bar, 1);
        fence_mbar_init();
        s_blk[0] = PR_WARPS;
        s_blk[1] = PR_WARPS;
    }
    int par = 0;
    long long staged_oid = -1;
    uint32_t phase = 0;
    // dynamic pose scheduler, one pose ahead (see adds_cta_kernel)
    if (tid == 0) s_next = atomicAdd(a.work_counter, 1);
    __syncthreads();

    for (;;) {
        const int64_t it = s_next;
        if (it >= a.B) break;
        const int64_t b = a.order ? a.order[it] : it;
        load_pose(a, b, tid, s_pose, &s_oid);
        __syncthreads();  // (A) also: the previous pose's readers of shared memory are done
        if (tid == 64) s_next = atomicAdd(a.work_counter, 1);   // read after barriers (B) and (C)
        const long long oid = s_oid;
        if (!slot_known(oid, a.n_slots, a.slots)) {  // CTA-uniform
            if (tid == 0) write_skipped(a, b, true);
            __syncthreads();
            continue;
        }
        const SlotInfo s = a.slots[oid];
        const PrunedSlot ps = pa.pslots[oid];
        const int n = s.count, nb = ps.nb, np = PR_BLOCK * nb, nbp = (nb + 3) / 4 * 4;
        if (oid != staged_oid) {
            stage_mesh(s_sorted, pa.sorted + ps.offset, ps.floats, &s_bar, phase, tid);
            phase ^= 1;
            staged_oid = oid;
        }
        const float* mx = s_sorted;
        const float* my = mx + np;
        const float* mz = my + np;
        const float* cen = mz + np;
        const float* sub = cen + 3 * nbp;
        const int ns = 4 * nb;
        const uint16_t* perm = reinterpret_cast<const uint16_t*>(sub + 3 * ns);
        const int mode = s.xform_mode;

        // phase B': the warp's blocks -> both clouds, ADD distances, bounding spheres
        {
            float Rp[9], Rg[9], tp[3], tg[3];
            quat_to_mat(s_pose, Rp);
            quat_to_mat(s_pose + 4, Rg);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                tp[k] = s_pose[8 + k];
                tg[k] = s_pose[11 + k];
            }
            for (int blk = warp; blk < nb; blk += PR_WARPS) {
                const int p = PR_BLOCK * blk + lane;
                const unsigned orig = perm[p];
                const bool valid = orig != 0xffffu;
                const float x = mx[p], y = my[p], z = mz[p];
                float px, py, pz, qx, qy, qz;
                xform_point(mode, x, y, z, Rp, tp, px, py, pz);
                xform_point(mode, x, y, z, Rg, tg, qx, qy, qz);
                s_pred[p] = px;
                s_pred[np + p] = py;
                s_pred[2 * np + p] = pz;
                float* gq = s_gt + (p >> 2) * 12 + (p & 3);
                gq[0] = valid ? qx : GT_SENTINEL;
                gq[4] = valid ? qy : GT_SENTINEL;
                gq[8] = valid ? qz : GT_SENTINEL;
                if (valid) s_dadd[orig] = __fsqrt_rn(sq3(__fsub_rn(px, qx), __fsub_rn(py, qy), __fsub_rn(pz, qz)));
                // spheres: centre = the transformed centroid (any point would do), radius from the actual points
                const float cx = cen[blk], cy = cen[nbp + blk], cz = cen[2 * nbp + blk];
                const int sb = 4 * blk + (lane >> 3);
                const float sx = sub[sb], sy = sub[ns + sb], sz = sub[2 * ns + sb];
                float cpx, cpy, cpz, cgx, cgy, cgz;
                xform_point(XF_FMA_CHAIN, cx, cy, cz, Rp, tp, cpx, cpy, cpz);     // pred: the whole block
                xform_point(XF_FMA_CHAIN, sx, sy, sz, Rg, tg, cgx, cgy, cgz);     // gt: the lane's sub-block
                const float dp = sqrtf(sq3(px - cpx, py - cpy, pz - cpz));
                const float dg = sqrtf(sq3(qx - cgx, qy - cgy, qz - cgz));
                // maxima over the valid lanes through the bit patterns (non-negative floats order like unsigned
                // integers; a NaN sorts above every number and so survives into the radius)
                const unsigned rp = __reduce_max_sync(full, valid ? __float_as_uint(dp) : 0u);
                unsigned rg = valid ? __float_as_uint(dg) : 0u;
                rg = max(rg, __shfl_xor_sync(full, rg, 1));
                rg = max(rg, __shfl_xor_sync(full, rg, 2));
                rg = max(rg, __shfl_xor_sync(full, rg, 4));
                if (lane == 0) s_cp[blk] = make_float4(cpx, cpy, cpz, __uint_as_float(rp) * 1.00001f);
                if ((lane & 7) == 0) s_cg[sb] = make_float4(cgx, cgy, cgz, __uint_as_float(rg) * 1.00001f);
            }
        }
        __syncthreads();  // (B)

        // phase C': one warp per pred block, one pred point per lane
        {
            const float4* gq4 = reinterpret_cast<const float4*>(s_gt);      // block B at gq4[24 B ..], sub-block at gq4[6 SB ..]
            // the number of sub-blocks left over differs from block to block: the first block of a warp is its own
            // index, the next ones are claimed from a counter, so no warp waits at barrier (C) for a slow one
            int A = warp;
            while (A < nb) {
                const int p = PR_BLOCK * A + lane;
                const unsigned orig = perm[p];
                const bool valid = orig != 0xffffu;
                const float px = s_pred[p], py = s_pred[np + p], pz = s_pred[2 * np + p];
                float m = eval_block(gq4 + 24 * A, px, py, pz, __int_as_float(0x7f800000));
                const float4 cA = s_cp[A];
                for (int c0 = 0; c0 < ns; c0 += 32) {
                    // the bound uses the current minima: recomputed per chunk of 32 candidate sub-blocks
                    const float mmax = __uint_as_float(__reduce_max_sync(full, valid ? __float_as_uint(m) : 0u));
                    const float th = sqrtf(mmax) * 1.0001f + cA.w;
                    const int Bq = c0 + lane;
                    bool cand = false;
                    if (Bq < ns && (Bq >> 2) != A) {
                        const float4 cB = s_cg[Bq];
                        const float dx = cA.x - cB.x, dy = cA.y - cB.y, dz = cA.z - cB.z;
                        const float d2 = dx * dx + dy * dy + dz * dz;
                        const float rhs = th + cB.w;
                        // skip only when the test holds in numbers; NaN / inf on either side -> evaluate
                        const bool skip = d2 * 0.9999f >= rhs * rhs && d2 < 3.0e38f;
                        cand = !skip;
                    }
                    unsigned todo = __ballot_sync(full, cand);
                    while (todo) {
                        const int b0 = __ffs(todo) - 1;
                        todo &= todo - 1;
                        if (todo) {
                            const int b1 = __ffs(todo) - 1;
                            todo &= todo - 1;
                            m = eval_two(gq4 + 6 * (c0 + b0), gq4 + 6 * (c0 + b1), px, py, pz, m);
                        } else {
                            m = eval_sub(gq4 + 6 * (c0 + b0), px, py, pz, m);
                        }
                    }
                }
                // sqrt is monotone and correctly rounded: sqrt(min s) == min sqrt(s)
                if (valid) s_dadds[orig] = __fsqrt_rn(m);
                int nxt = 0;
                if (lane == 0) nxt = atomicAdd(&s_blk[par], 1);
                A = __shfl_sync(full, nxt, 0);
            }
        }
        __syncthreads();  // (C)
        if (tid == 0) s_blk[par] = PR_WARPS;      // re-armed for the pose after the next; nobody reads it before barrier (A)
        par ^= 1;

        // phase D: ordered means (ATen summation order) on warps 0 and 1, decision, outputs
        if (tid < 64) {
            ordered_means(s_dadd, s_dadds, n, tid, lane, true, s_mean, [](const float* p) { return *p; });
            if (tid == 0) write_pose(a, b, oid, s, s_mean[0], s_mean[1], true);
        }
        // barrier (A) of the next pose protects the shared arrays
    }
}

// dynamic shared memory of the table's largest mesh
static size_t pruned_smem_bytes(const p6d_mesh_table* t) {
    const int nb = t->pruned->max_nb > 0 ? t->pruned->max_nb : 1;
    return sizeof(float) * pr_smem_floats(nb, t->max_count);
}

bool pruned_fits(const p6d_mesh_table* t, int limit) {   // t has a block structure
    return pruned_smem_bytes(t) + 1024 <= static_cast<size_t>(limit);
}

// The pruned kernel for one evaluation launch, for any mesh size that fits (launch_eval decides when it pays).
int launch_eval_pruned(const p6d_mesh_table* table, const EvalArgs& args, cudaStream_t st) {
    const PrunedTable* ptab = table->pruned;
    if (!ptab) {
        set_error("p6d_add_eval_pruned: this table has no block structure (a mesh with more than 65,534 points, or out of "
                  "memory at creation)");
        return P6D_ETOOBIG;
    }
    int limit = 0;
    int rc = max_optin_smem(table->device, &limit);
    if (rc) return rc;
    if (!pruned_fits(table, limit)) {
        set_error("largest mesh has %d points; the pruned ADD-S kernel keeps both clouds and the sorted mesh in "
                  "shared memory and accepts at most %d points on this device (p6d_add_eval takes larger meshes)",
                  table->max_count, (limit - 1024) / 4 / 12 / 32 * 32);
        return P6D_ETOOBIG;
    }
    const int nb = ptab->max_nb > 0 ? ptab->max_nb : 1;
    const size_t smem = pruned_smem_bytes(table);
    EvalArgs a = args;
    if ((rc = claim_counter(table, st, &a.work_counter))) return rc;
    // the instantiation whose register budget matches what shared memory lets be resident (see the kernel's comment)
    struct Shape { const void* fn; int threads, minb; };
    const Shape shapes[] = {{(const void*)adds_pruned_kernel<128, 8>, 128, 8}, {(const void*)adds_pruned_kernel<256, 4>, 256, 4},
                            {(const void*)adds_pruned_kernel<256, 3>, 256, 3}, {(const void*)adds_pruned_kernel<256, 2>, 256, 2}};
    const Shape* pick = &shapes[3];
    int per_sm = 0;
    for (const Shape& sh : shapes) {
        if (sh.threads == 128 && nb > 16) continue;           // small CTAs for meshes of <= 512 points only
        if ((rc = ctas_per_sm(sh.fn, sh.threads, table->device, smem, &per_sm))) return rc;
        if (per_sm >= sh.minb || &sh == &shapes[3]) {
            pick = &sh;
            break;
        }
    }
    int64_t grid = static_cast<int64_t>(table->sm_count) * per_sm;
    if (grid > a.B) grid = a.B;
    PrunedArgs pa{ptab->d_sorted, ptab->d_slots};
    int nb_arg = nb, nmax_arg = table->max_count;
    void* kargs[] = {&a, &pa, &nb_arg, &nmax_arg};
    P6D_CUDA(cudaLaunchKernel(pick->fn, dim3(static_cast<unsigned>(grid)), dim3(pick->threads), kargs, smem, st));
    P6D_CUDA(cudaGetLastError());
    return P6D_OK;
}

}  // namespace p6d
