// b200reg — NDT registration (B3): voxel-Gaussian map build, score/gradient/Hessian, Newton + More-Thuente
// line search with the control flow resident on the device, batched hypothesis scoring for relocalization.
//
// Replaces pclomp::NormalDistributionsTransform (pointcloud_match/ndt_omp/include/pclomp/ndt_omp.h:117-261,
// ndt_omp_impl.hpp:47-880) and pclomp::VoxelGridCovariance (voxel_grid_covariance_omp_impl.hpp:49-442).
//
// set_target  min/max reduction -> leaf id per point -> radix sort (point order preserved inside a leaf) ->
//             run-length segments -> one warp per leaf accumulates sum(p), sum(p p^T) in fp64 *in input order*
//             (9 lanes own the 9 sums, points are fetched 32 at a time) -> one thread per leaf: mean, covariance,
//             3x3 eigen-decomposition, eigenvalue inflation, inverse -> dense cell -> leaf table.
// align       k_ndt_eval is launched back to back; every launch evaluates score/gradient/Hessian (or the fp64
//             Hessian) at the pose the control block asks for, and the last block to finish reduces the block
//             partials in a fixed order and advances the Newton / More-Thuente state machine (computeTransformation
//             + computeStepLengthMT) by one evaluation.  The host only polls a done flag every few launches.
//             gridDim.y indexes independent alignments (hypotheses), each with its own control block.
#include "ndt.cuh"

#include <cub/cub.cuh>

#include <cmath>
#include <thread>
#include <vector>

namespace b200 {
namespace ndt {

constexpr int EVAL_THREADS = 256;
constexpr int LAUNCH_BATCH = 8;   // evaluations enqueued between two polls of the done flag

enum Phase : int { PH_SINGLE_DERIV = 0, PH_SINGLE_HESS, PH_INIT, PH_MT_FIRST, PH_MT_LOOP, PH_MT_HESS };
enum Mode : int { MODE_DERIV_H = 0, MODE_DERIV_NOH, MODE_HESS_D };

struct Ctl {  // one per alignment, global memory
    // evaluation request, read by every block of a launch
    float M[16];   // row-major transform the source is evaluated under
    AngleTables tab;
    int mode;
    int done;
    unsigned ticket;
    int phase;
    // computeTransformation state
    double p[6], g[6], H[36], score;
    int nr_iterations, converged, evals, hess_evals;
    double trans_probability;
    float final_T[16];  // row-major
    // computeStepLengthMT state
    double x_t[6], dir[6];
    double a_l, f_l, g_l, a_u, f_u, g_u, a_t, phi_0, d_phi_0, phi_t, d_phi_t, psi_t, d_psi_t;
    double step_min, step_max;
    int step_iterations, interval_converged, open_interval, req;
    long long solve_cycles, step_cycles;
};

struct AlignConsts {
    double step_size, trans_eps;
    int max_iter;
    int n_src;
};

// ------------------------------------------------------------------ target build
__device__ __forceinline__ int f2ord(float f) {  // order-preserving float -> int
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

// pcl::getMinMax3D over the finite points of pts[0, n) (voxel_grid_covariance_omp_impl.hpp:72); this block covers the
// indices x0, x0 + xstride, ...
__device__ __forceinline__ void minmax_range(const float4* __restrict__ pts, int64_t n, int64_t x0, int64_t xstride,
                                             int* __restrict__ mm /*[6]: min xyz, max xyz (ordered ints)*/) {
    float mn[3] = {3.402823466e+38f, 3.402823466e+38f, 3.402823466e+38f}, mx[3] = {-3.402823466e+38f, -3.402823466e+38f, -3.402823466e+38f};
    for (int64_t i = x0; i < n; i += xstride) {
        const float4 p = __ldg(pts + i);
        if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) continue;
        mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
        mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k)
        for (int o = 16; o > 0; o >>= 1) {
            mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
            mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            atomicMin(mm + k, f2ord(mn[k]));
            atomicMax(mm + 3 + k, f2ord(mx[k]));
        }
    }
}
__global__ void k_ndt_minmax(const float4* __restrict__ pts, int64_t n, int* __restrict__ mm) {
    minmax_range(pts, n, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x, mm);
}
__global__ void k_ndt_minmax_init(int* mm) {
    if (threadIdx.x < 3) mm[threadIdx.x] = 0x7fffffff;
    else if (threadIdx.x < 6) mm[threadIdx.x] = (int)0x80000000;
}

struct GridDims {
    int min_b[3], max_b[3], div_b[3], mul[3];
    float inv_leaf;
};

// leaf id of a point (:218-223); non-finite points get the sentinel key and sort last
__device__ __forceinline__ uint32_t leaf_key(const float4 p, const GridDims& gd, uint32_t sentinel) {
    uint32_t key = sentinel;
    if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
        const int i0 = (int)(floorf(p.x * gd.inv_leaf) - (float)gd.min_b[0]);
        const int i1 = (int)(floorf(p.y * gd.inv_leaf) - (float)gd.min_b[1]);
        const int i2 = (int)(floorf(p.z * gd.inv_leaf) - (float)gd.min_b[2]);
        key = (uint32_t)(i0 * gd.mul[0] + i1 * gd.mul[1] + i2 * gd.mul[2]);
    }
    return key;
}
__global__ void k_ndt_keys(const float4* __restrict__ pts, int n, GridDims gd, uint32_t sentinel, uint32_t* __restrict__ keys,
                           int32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = leaf_key(__ldg(pts + i), gd, sentinel);
    vals[i] = i;
}

// One warp per leaf: fp64 sums of p and p p^T in input order (:233-237).  Lane c < 3 owns sum(p_c); lanes 3..8 own
// the six distinct products (p_a p_b is commutative, so the full 3x3 of the reference holds the same six values).
// The reference's Leaf() starts cov_ at the identity (voxel_grid_covariance_omp.h:103-112) and accumulates on top.
__global__ void __launch_bounds__(256) k_ndt_accumulate(const float4* __restrict__ pts, const int32_t* __restrict__ sorted_idx,
                                                        const uint32_t* __restrict__ uniq, const int32_t* __restrict__ run_off,
                                                        const int32_t* __restrict__ run_cnt, const int32_t* __restrict__ nruns,
                                                        uint32_t sentinel, double* __restrict__ sums /*[nruns][9]*/,
                                                        float* __restrict__ centroid /*[nruns][3]*/) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int nr = *nruns;
    // (a, b) component selectors of this lane: 0..2 = x,y,z, 3 = the constant 1
    const int sa = lane < 3 ? lane : lane == 3 ? 0 : lane == 4 ? 0 : lane == 5 ? 0 : lane == 6 ? 1 : lane == 7 ? 1 : 2;
    const int sb = lane < 3 ? 3 : lane == 3 ? 0 : lane == 4 ? 1 : lane == 5 ? 2 : lane == 6 ? 1 : lane == 7 ? 2 : 2;
    for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < nr; r += warps) {
        if (uniq[r] == sentinel) continue;  // the non-finite bucket
        const int off = run_off[r], cnt = run_cnt[r];
        double acc = (lane == 3 || lane == 6 || lane == 8) ? 1.0 : 0.0;
        float facc = 0.0f;  // lanes 9..11: leaf.centroid, the fp32 running sum of x / y / z in input order (vgc_impl:241-242)
        for (int base = 0; base < cnt; base += 32) {
            float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
            if (base + lane < cnt) p = __ldg(pts + __ldg(sorted_idx + off + base + lane));
            const int m = min(32, cnt - base);
            for (int j = 0; j < m; ++j) {
                const float x = __shfl_sync(0xffffffffu, p.x, j), y = __shfl_sync(0xffffffffu, p.y, j), z = __shfl_sync(0xffffffffu, p.z, j);
                const double a = (double)(sa == 0 ? x : sa == 1 ? y : z);
                const double b = sb == 3 ? 1.0 : (double)(sb == 0 ? x : sb == 1 ? y : z);
                acc += a * b;
                facc += lane == 9 ? x : lane == 10 ? y : z;
            }
        }
        if (lane < 9) sums[(size_t)r * 9 + lane] = acc;
        else if (lane < 12) centroid[(size_t)r * 3 + (lane - 9)] = facc / (float)cnt;  // leaf.centroid /= (float) nr_points (:289)
    }
}

// One thread per leaf: second pass of applyFilter (:282-367)
__global__ void k_ndt_finalize(const uint32_t* __restrict__ uniq, const int32_t* __restrict__ run_cnt, const int32_t* __restrict__ nruns,
                               uint32_t sentinel, const double* __restrict__ sums, int min_pts, double eig_ratio, LeafF* __restrict__ leafF,
                               LeafD* __restrict__ leafD, double* __restrict__ covs, int32_t* __restrict__ npts, uint8_t* __restrict__ valid,
                               int32_t* __restrict__ cell2leaf, int32_t* __restrict__ n_valid) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= *nruns) return;
    valid[r] = 0;
    const uint32_t id = uniq[r];
    if (id == sentinel) { npts[r] = 0; return; }
    const int n = run_cnt[r];
    npts[r] = n;
    const double* s = sums + (size_t)r * 9;
    const double pt_sum[3] = {s[0], s[1], s[2]};
    double mean[3];
    for (int a = 0; a < 3; ++a) mean[a] = pt_sum[a] / n;
    LeafD L;
    for (int a = 0; a < 3; ++a) L.mean[a] = mean[a];
    for (int a = 0; a < 9; ++a) L.icov[a] = 0.0;
    if (n < min_pts) { leafD[r] = L; return; }
    const double S[9] = {s[3], s[4], s[5], s[4], s[6], s[7], s[5], s[7], s[8]};
    const double np = n;
    double cov[9];
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) cov[a * 3 + b] = (S[a * 3 + b] - 2 * (pt_sum[a] * mean[b])) / np + mean[a] * mean[b];
    const double f = (np - 1.0) / np;
    for (int a = 0; a < 9; ++a) cov[a] *= f;
    double A[9], w[3], V[9];
    for (int a = 0; a < 3; ++a)  // SelfAdjointEigenSolver reads the lower triangle
        for (int b = 0; b < 3; ++b) A[a * 3 + b] = (a >= b) ? cov[a * 3 + b] : cov[b * 3 + a];
    eigen_selfadjoint3(A, w, V);  // eigensolver.compute(leaf.cov_), Eigen's own algorithm (ndt.cuh)
    if (w[0] < 0 || w[1] < 0 || w[2] <= 0) { npts[r] = -1; leafD[r] = L; return; }
    const double min_ev = eig_ratio * w[2];
    if (w[0] < min_ev) {
        w[0] = min_ev;
        if (w[1] < min_ev) w[1] = min_ev;
        double Vi[9], VL[9];
        inverse3(V, Vi);
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) VL[a * 3 + b] = V[a * 3 + b] * w[b];
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) cov[a * 3 + b] = VL[a * 3] * Vi[b] + VL[a * 3 + 1] * Vi[3 + b] + VL[a * 3 + 2] * Vi[6 + b];
    }
    inverse3(cov, L.icov);
    double mxc = L.icov[0], mnc = L.icov[0];
    for (int a = 1; a < 9; ++a) { mxc = fmax(mxc, L.icov[a]); mnc = fmin(mnc, L.icov[a]); }
    for (int a = 0; a < 9; ++a) covs[(size_t)r * 9 + a] = cov[a];
    leafD[r] = L;
    if (mxc == CUDART_INF || mnc == -CUDART_INF) { npts[r] = -1; return; }
    LeafF F;
    for (int a = 0; a < 3; ++a) F.mean[a] = mean[a];
    for (int a = 0; a < 9; ++a) F.icov[a] = (float)L.icov[a];
    F.pad = 0.f;
    leafF[r] = F;
    valid[r] = 1;
    cell2leaf[id] = r;
    atomicAdd(n_valid, 1);
}

// One thread per leaf: the score store (ndt.cuh) from leafD, indexed by the same leaf slot so cell2leaf and nbr7 address
// it unchanged.  The off-diagonal pairs are stored summed: xt' C xt = xt' ((C + C') / 2) xt.  Leaves without a valid
// Gaussian are never referenced by cell2leaf / nbr7 and get zeros.
__global__ void k_ndt_score_store(const LeafD* __restrict__ leafD, const uint8_t* __restrict__ valid, int nruns, Dbl4* __restrict__ sA,
                                  Dbl4* __restrict__ sB, double* __restrict__ sC) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nruns) return;
    Dbl4 a = {0.0, 0.0, 0.0, 0.0}, b = {0.0, 0.0, 0.0, 0.0};
    double c = 0.0;
    if (valid[r]) {
        const LeafD L = leafD[r];
        const double* C = L.icov;
        a = {L.mean[0], L.mean[1], L.mean[2], C[0]};
        b = {C[1] + C[3], C[2] + C[6], C[4], C[5] + C[7]};
        c = C[8];
    }
    sA[r] = a;
    sB[r] = b;
    sC[r] = c;
}

// DIRECT7 neighbourhood table: one 32-byte record per grid cell = the leaf slots of the cell and its six face neighbours
// in the reference's order (vgc_impl:423-430), -1 where the neighbour is outside the grid or holds no usable leaf, and the
// number of leaves in [7].  A point whose own cell lies inside the grid then resolves its whole neighbourhood with ONE
// 256-bit load instead of seven scattered 4-byte probes (the probes were most of the L1 wavefronts of the score kernel).
__global__ void k_ndt_build_nbr7(const int32_t* __restrict__ cell2leaf, int64_t ncells, int d0, int d1, int d2, int32_t* __restrict__ nbr7) {
    const int64_t id = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (id >= ncells) return;
    const int ix = (int)(id % d0), iy = (int)((id / d0) % d1), iz = (int)(id / ((int64_t)d0 * d1));
    int out[8], cnt = 0;
#pragma unroll
    for (int s = 0; s < 7; ++s) {
        int dx, dy, dz;
        nbr_offset(7, s, dx, dy, dz);
        const int x = ix + dx, y = iy + dy, z = iz + dz;
        int lf = -1;
        if (x >= 0 && x < d0 && y >= 0 && y < d1 && z >= 0 && z < d2) lf = cell2leaf[x + (int64_t)y * d0 + (int64_t)z * d0 * d1];
        out[s] = lf;
        cnt += lf >= 0 ? 1 : 0;
    }
    out[7] = cnt;
    int4* dst = reinterpret_cast<int4*>(nbr7 + id * 8);
    dst[0] = make_int4(out[0], out[1], out[2], out[3]);
    dst[1] = make_int4(out[4], out[5], out[6], out[7]);
}

// ------------------------------------------------------------------ source ordering
// The derivative and score kernels read, per source point, up to 7 cells of the dense table and 64, 72 or 96 leaf bytes
// for every hit.  In scan order (a Livox rosette) the 32 lanes of a warp touch 32 unrelated voxels and every load
// instruction costs 32 L1 wavefronts (ncu: l1tex at 94 % of peak in k_ndt_score_batch).  Sorting the source once by the
// Morton code of its voxel (in the sensor frame - a rigid transform keeps neighbours together) makes neighbouring
// lanes hit the same or adjacent leaves.  Only the order of the fp64 sums changes.
__device__ __forceinline__ uint32_t spread10(uint32_t v) {
    v &= 0x3FFu;
    v = (v | (v << 16)) & 0x030000FFu;
    v = (v | (v << 8)) & 0x0300F00Fu;
    v = (v | (v << 4)) & 0x030C30C3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
__device__ __forceinline__ uint32_t morton_key(const float4 p, float inv_cell) {
    uint32_t key = 0xFFFFFFFFu;
    if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
        const int cx = min(max((int)floorf(p.x * inv_cell) + 512, 0), 1023), cy = min(max((int)floorf(p.y * inv_cell) + 512, 0), 1023),
                  cz = min(max((int)floorf(p.z * inv_cell) + 512, 0), 1023);
        key = spread10((uint32_t)cx) | (spread10((uint32_t)cy) << 1) | (spread10((uint32_t)cz) << 2);
    }
    return key;
}
__global__ void k_ndt_source_keys(const float4* __restrict__ pts, int n, float inv_cell, uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = morton_key(__ldg(pts + i), inv_cell);
    vals[i] = i;
}
__global__ void k_ndt_gather(const float4* __restrict__ in, const int32_t* __restrict__ idx, int n, float4* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __ldg(in + __ldg(idx + i));
}

// Per-yaw orderings for the score kernel.  Under a hypothesis of yaw psi a sensor-frame voxel becomes a rotated cube that
// straddles up to 8 map cells, so a warp of sensor-Morton-ordered points spreads over more map cells (and more leaf lines
// per load) than it needs to.  Yaw bin b orders the scan by the Morton code of Rz(psi_b) p, psi_b = 2 pi b / bins: the
// map-axis order of the rotation part of every pose whose yaw is nearest psi_b (translation only shifts the cells).  The
// bins must be fine: a point 100 m out moves by one cell when psi is off by 0.01 rad.  For random yaws, 32 bins (mean
// error 0.05 rad) cut the distinct leaf lines per warp load by 2.5 %, 512 bins (0.003 rad) by 18 %, against 26 % for a
// per-hypothesis sort (tools/score_order_lines.py --random-yaw).
// score_yaw_bin() picks the bin from the pose alone and the ordering of a bin is a fixed function of (source, bin), so a
// hypothesis's score never depends on how the batch is cut.  The orderings are built on first use (Ndt::yaw_orderings)
// and kept until the next set_source: a relocalization batch needs only the bins of its yaws, and align-only callers
// never pay for them.
constexpr int YAW_BINS_MAX = 512;
// bins per source: the largest power of two <= YAW_BINS_MAX whose orderings all fit in 256 MiB (512 up to 32k points).
// That bounds the ordering store of an engine; building bins also holds sort buffers of 24 bytes per (bin, point) being
// built (+25 % growth slack, released once every bin exists) and cub's temporary storage.
constexpr int64_t YAW_ORDER_MAX_BYTES = (int64_t)256 << 20;

__device__ __forceinline__ int score_yaw_bin(float r00, float r10, int bins) {  // bins: a power of two
    const float psi = atan2f(r10, r00);
    if (!isfinite(psi)) return 0;  // non-finite pose
    const int b = (int)rintf(psi * ((float)bins * 0.159154943091895336f));
    return b & (bins - 1);
}
// need[b] = 1 for the yaw bin of every pose (h x 16 col-major: R00 = [0], R10 = [1])
__global__ void k_ndt_yaw_need(const float* __restrict__ poses, int64_t h, int bins, int32_t* __restrict__ need) {
    for (int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; a < h; a += (int64_t)gridDim.x * blockDim.x)
        need[score_yaw_bin(poses[a * 16], poses[a * 16 + 1], bins)] = 1;
}
// grid = (point blocks, bins to build): key = (j, Morton key of Rz(psi_b) p) for the j-th bin b = list[j], value = the
// point's index in the caller's order
__global__ void k_ndt_source_keys_yaw(const float4* __restrict__ pts, int n, float inv_cell, const int32_t* __restrict__ list, int bins,
                                      uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int j = blockIdx.y;
    float s, c;
    sincospif(2.0f * (float)list[j] / (float)bins, &s, &c);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 p = __ldg(pts + i);
        const float4 q = make_float4(c * p.x - s * p.y, s * p.x + c * p.y, p.z, 0.f);
        const size_t o = (size_t)j * n + i;
        keys[o] = ((uint64_t)j << 32) | morton_key(q, inv_cell);
        vals[o] = i;
    }
}

// ------------------------------------------------------------------ independent (source, target) pairs
// The clouds of a chunk of pairs lie end to end; off[j] .. off[j+1]-1 are pair j's points, grid row y = pair y.  The dense
// cell tables of the targets are laid out end to end as well: pair j's leaf id l becomes the key cell_base + l, so ONE
// stable sort, run-length encoding and scan serve every target, and k_ndt_accumulate / k_ndt_finalize run unchanged.
struct PairGrid {
    GridDims gd;
    uint32_t cell_base;
    int live;  // 0: the pair is not built (its target failed); its points take the sentinel key
};
__global__ void k_ndt_minmax_init_pairs(int* mm, int np) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 6 * np) mm[i] = (i % 6) < 3 ? 0x7fffffff : (int)0x80000000;
}
__global__ void k_ndt_minmax_pairs(const float4* __restrict__ pts, const int64_t* __restrict__ off, int* __restrict__ mm) {
    const int64_t b = off[blockIdx.y];
    minmax_range(pts + b, off[blockIdx.y + 1] - b, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x, mm + 6 * blockIdx.y);
}
__global__ void k_ndt_keys_pairs(const float4* __restrict__ pts, const int64_t* __restrict__ off, const PairGrid* __restrict__ pg, uint32_t sentinel,
                                 uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int64_t b = off[blockIdx.y], n = off[blockIdx.y + 1] - b;
    const PairGrid g = pg[blockIdx.y];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t key = sentinel;
        if (g.live) {
            const uint32_t l = leaf_key(__ldg(pts + b + i), g.gd, 0xFFFFFFFFu);
            if (l != 0xFFFFFFFFu) key = g.cell_base + l;
        }
        keys[b + i] = key;
        vals[b + i] = (int32_t)(b + i);
    }
}
// sources: key = (pair, Morton key of the voxel), so that one stable sort orders every pair's points as set_source does
__global__ void k_ndt_source_keys_pairs(const float4* __restrict__ pts, const int64_t* __restrict__ off, float inv_cell, uint64_t* __restrict__ keys,
                                        int32_t* __restrict__ vals) {
    const int64_t b = off[blockIdx.y], n = off[blockIdx.y + 1] - b;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        keys[b + i] = ((uint64_t)blockIdx.y << 32) | morton_key(__ldg(pts + b + i), inv_cell);
        vals[b + i] = (int32_t)(b + i);
    }
}

// ------------------------------------------------------------------ Newton / More-Thuente state machine (thread 0 of the last block)
// H x = rhs the way JacobiSVD(H).solve(rhs) answers it for symmetric H (ndt_omp_impl.hpp:112-114): a pseudo-inverse that
// drops singular values below max(sv) * 6 eps.  When H is comfortably full rank that is simply H^-1 rhs, which a pivoted
// 6x6 elimination delivers in ~2 us of one thread; only a (nearly) rank-deficient H takes the literal two-sided Jacobi
// SVD below.
__device__ __noinline__ bool lu_solve6(const double* Hs, const double* rhs, double* x) {
    double a[6][7];
    for (int i = 0; i < 6; ++i) {
        for (int j = 0; j < 6; ++j) a[i][j] = Hs[i * 6 + j];
        a[i][6] = rhs[i];
    }
    double pmax = 0.0, pmin = 1.7976931348623157e308, rinv[6];
    for (int k = 0; k < 6; ++k) {
        int piv = k;
        double best = fabs(a[k][k]);
        for (int i = k + 1; i < 6; ++i)
            if (fabs(a[i][k]) > best) { best = fabs(a[i][k]); piv = i; }
        if (!(best > 0.0)) return false;
        if (piv != k)
            for (int j = k; j < 7; ++j) { const double t = a[k][j]; a[k][j] = a[piv][j]; a[piv][j] = t; }
        pmax = fmax(pmax, best);
        pmin = fmin(pmin, best);
        const double inv = 1.0 / a[k][k];
        rinv[k] = inv;
        for (int i = k + 1; i < 6; ++i) {
            const double f = a[i][k] * inv;
            for (int j = k + 1; j < 7; ++j) a[i][j] -= f * a[k][j];
        }
    }
    if (!(pmin > 1e-9 * pmax)) return false;  // too close to rank deficient for the shortcut (also catches NaN)
    for (int i = 5; i >= 0; --i) {
        double sacc = a[i][6];
        for (int j = i + 1; j < 6; ++j) sacc -= a[i][j] * x[j];
        x[i] = sacc * rinv[i];  // the pivots' reciprocals are already there: six fewer fp64 divisions on the serial path
    }
    return true;
}

// JacobiSVD<Matrix<double,6,6>>(H, FullU | FullV).solve(rhs), literally: two-sided Jacobi sweeps E/SVD/JacobiSVD.h:666-745,
// 2x2 real SVD E/misc/RealSvd2x2.h:18-51 (makeJacobi E/Jacobi/Jacobi.h:83-113, rotation product :53-59), signs / scale / sort
// JacobiSVD.h:747-792, rank with threshold 6 eps and solve E/SVD/SVDBase.h:149-157,198-205,308-318 (E/ = the Eigen sources
// vendored in the reference).  Only a (nearly) rank-deficient or non-finite H gets here.
__device__ __noinline__ void jacobi_svd_solve6(const double* H, const double* rhs, double* x) {
    const int n = 6;
    const double eps = 2.220446049250313e-16, dmin = 2.2250738585072014e-308, precision = 2.0 * eps;
    double scale = 0.0;
    bool bad = false;
    for (int i = 0; i < 36; ++i) {
        const double a = fabs(H[i]);
        if (a != a) bad = true;
        if (a > scale) scale = a;
    }
    if (bad || isinf(scale)) {  // InvalidInput: no decomposition; the caller sees a NaN step and stops (ndt_omp_impl.hpp:119-123)
        for (int i = 0; i < 6; ++i) x[i] = CUDART_NAN;
        return;
    }
    if (scale == 0.0) scale = 1.0;
    double W[6][6], U[6][6], V[6][6];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            W[i][j] = H[i * 6 + j] / scale;
            U[i][j] = V[i][j] = i == j ? 1.0 : 0.0;
        }
    double maxDiag = 0.0;
    for (int i = 0; i < n; ++i) maxDiag = fabs(W[i][i]) > maxDiag ? fabs(W[i][i]) : maxDiag;
    bool finished = false;
    int guard = 0;
    while (!finished && ++guard < 1000) {
        finished = true;
        for (int p = 1; p < n; ++p) {
            for (int q = 0; q < p; ++q) {
                const double thr = fmax(dmin, precision * maxDiag);
                if (fabs(W[p][q]) > thr || fabs(W[q][p]) > thr) {
                    finished = false;
                    double m00 = W[p][p], m01 = W[p][q], m10 = W[q][p], m11 = W[q][q];
                    double c1, s1;
                    const double t = m00 + m11, d = m10 - m01;
                    if (fabs(d) < dmin) {
                        s1 = 0.0; c1 = 1.0;
                    } else {
                        const double u = t / d;
                        const double tmp = sqrt(1.0 + u * u);
                        s1 = 1.0 / tmp;
                        c1 = u / tmp;
                    }
                    if (!(c1 == 1.0 && s1 == 0.0)) {
                        const double a0 = m00, a1 = m01, b0 = m10, b1 = m11;
                        m00 = c1 * a0 + s1 * b0; m01 = c1 * a1 + s1 * b1;
                        m10 = -s1 * a0 + c1 * b0; m11 = -s1 * a1 + c1 * b1;
                    }
                    double cr, sr;
                    {
                        const double deno = 2.0 * fabs(m01);
                        if (deno < dmin) {
                            cr = 1.0; sr = 0.0;
                        } else {
                            const double tau = (m00 - m11) / deno;
                            const double w = sqrt(tau * tau + 1.0);
                            const double tt = tau > 0.0 ? 1.0 / (tau + w) : 1.0 / (tau - w);
                            const double sign_t = tt > 0.0 ? 1.0 : -1.0;
                            const double nn = 1.0 / sqrt(tt * tt + 1.0);
                            sr = -sign_t * (m01 / fabs(m01)) * fabs(tt) * nn;
                            cr = nn;
                        }
                    }
                    const double c2 = cr, s2 = -sr;
                    const double cl = c1 * c2 - s1 * s2, sl = c1 * s2 + s1 * c2;
                    if (!(cl == 1.0 && sl == 0.0)) {
                        for (int k = 0; k < n; ++k) {
                            const double xi = W[p][k], yi = W[q][k];
                            W[p][k] = cl * xi + sl * yi;
                            W[q][k] = -sl * xi + cl * yi;
                        }
                        for (int k = 0; k < n; ++k) {
                            const double xi = U[k][p], yi = U[k][q];
                            U[k][p] = cl * xi + sl * yi;
                            U[k][q] = -sl * xi + cl * yi;
                        }
                    }
                    if (!(cr == 1.0 && -sr == 0.0)) {
                        for (int k = 0; k < n; ++k) {
                            const double xi = W[k][p], yi = W[k][q];
                            W[k][p] = cr * xi - sr * yi;
                            W[k][q] = sr * xi + cr * yi;
                        }
                        for (int k = 0; k < n; ++k) {
                            const double xi = V[k][p], yi = V[k][q];
                            V[k][p] = cr * xi - sr * yi;
                            V[k][q] = sr * xi + cr * yi;
                        }
                    }
                    maxDiag = fmax(maxDiag, fmax(fabs(W[p][p]), fabs(W[q][q])));
                }
            }
        }
    }
    double sv[6];
    for (int i = 0; i < n; ++i) {
        const double a = W[i][i];
        sv[i] = fabs(a);
        if (a < 0.0)
            for (int k = 0; k < n; ++k) U[k][i] = -U[k][i];
    }
    for (int i = 0; i < n; ++i) sv[i] *= scale;
    int nonzero = n;
    for (int i = 0; i < n; ++i) {
        int pos = 0;
        double mx = sv[i];
        for (int j = 1; j < n - i; ++j)
            if (sv[i + j] > mx) { mx = sv[i + j]; pos = j; }
        if (mx == 0.0) { nonzero = i; break; }
        if (pos) {
            pos += i;
            const double ts = sv[i]; sv[i] = sv[pos]; sv[pos] = ts;
            for (int k = 0; k < n; ++k) {
                double tv = U[k][pos]; U[k][pos] = U[k][i]; U[k][i] = tv;
                tv = V[k][pos]; V[k][pos] = V[k][i]; V[k][i] = tv;
            }
        }
    }
    const double pthr = fmax(sv[0] * (6.0 * eps), dmin);
    int r = nonzero - 1;
    while (r >= 0 && sv[r] < pthr) --r;
    const int rank = r + 1;
    double tmp[6];
    for (int k = 0; k < rank; ++k) {
        double d = 0.0;
        for (int i = 0; i < n; ++i) d += U[i][k] * rhs[i];
        tmp[k] = (1.0 / sv[k]) * d;
    }
    for (int i = 0; i < n; ++i) {
        double d = 0.0;
        for (int k = 0; k < rank; ++k) d += V[i][k] * tmp[k];
        x[i] = d;
    }
}

__device__ inline void svd_solve6(const double* H, const double* rhs, double* x) {
    double Hs[36];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) Hs[i * 6 + j] = 0.5 * (H[i * 6 + j] + H[j * 6 + i]);
    if (!lu_solve6(Hs, rhs, x)) jacobi_svd_solve6(H, rhs, x);
}

// parity probe of the Newton direction (b200_ndt_newton_direction): io = [H(36) | rhs(6) | x(6) | path(1)]
__global__ void k_ndt_solve_probe(double* io, int force_svd) {
    if (threadIdx.x || blockIdx.x) return;
    double H[36], rhs[6], x[6];
    for (int i = 0; i < 36; ++i) H[i] = io[i];
    for (int i = 0; i < 6; ++i) rhs[i] = io[36 + i];
    double Hs[36];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) Hs[i * 6 + j] = 0.5 * (H[i * 6 + j] + H[j * 6 + i]);
    double path = 0.0;
    if (force_svd || !lu_solve6(Hs, rhs, x)) { jacobi_svd_solve6(H, rhs, x); path = 1.0; }
    for (int i = 0; i < 6; ++i) io[42 + i] = x[i];
    io[48] = path;
}

// updateIntervalMT (ndt_omp_impl.hpp:594-620)
__device__ inline bool mt_update_interval(Ctl& c, double f_t, double g_t) {
    const double a_t = c.a_t;
    if (f_t > c.f_l) { c.a_u = a_t; c.f_u = f_t; c.g_u = g_t; return false; }
    if (g_t * (c.a_l - a_t) > 0) { c.a_l = a_t; c.f_l = f_t; c.g_l = g_t; return false; }
    if (g_t * (c.a_l - a_t) < 0) {
        c.a_u = c.a_l; c.f_u = c.f_l; c.g_u = c.g_l;
        c.a_l = a_t; c.f_l = f_t; c.g_l = g_t;
        return false;
    }
    return true;
}

// trialValueSelectionMT (ndt_omp_impl.hpp:623-698): the four cases of More & Thuente's safeguarded cubic/quadratic step
__device__ inline double mt_trial_value(const Ctl& c, double f_t, double g_t) {
    const double a_l = c.a_l, f_l = c.f_l, g_l = c.g_l, a_u = c.a_u, f_u = c.f_u, g_u = c.g_u, a_t = c.a_t;
    auto cubic_min = [](double a0, double f0, double g0, double a1, double f1, double g1) {
        const double z = 3 * (f1 - f0) / (a1 - a0) - g1 - g0;
        const double w = sqrt(z * z - g1 * g0);
        return a0 + (a1 - a0) * (w - g0 - z) / (g1 - g0 + 2 * w);
    };
    if (f_t > f_l) {
        const double a_c = cubic_min(a_l, f_l, g_l, a_t, f_t, g_t);
        const double a_q = a_l - 0.5 * (a_l - a_t) * g_l / (g_l - (f_l - f_t) / (a_l - a_t));
        return fabs(a_c - a_l) < fabs(a_q - a_l) ? a_c : 0.5 * (a_q + a_c);
    }
    if (g_t * g_l < 0) {
        const double a_c = cubic_min(a_l, f_l, g_l, a_t, f_t, g_t);
        const double a_s = a_l - (a_l - a_t) / (g_l - g_t) * g_l;
        return fabs(a_c - a_t) >= fabs(a_s - a_t) ? a_c : a_s;
    }
    if (fabs(g_t) <= fabs(g_l)) {
        const double a_c = cubic_min(a_l, f_l, g_l, a_t, f_t, g_t);
        const double a_s = a_l - (a_l - a_t) / (g_l - g_t) * g_l;
        const double a_n = fabs(a_c - a_t) < fabs(a_s - a_t) ? a_c : a_s;
        return a_t > a_l ? fmin(a_t + 0.66 * (a_u - a_t), a_n) : fmax(a_t + 0.66 * (a_u - a_t), a_n);
    }
    return cubic_min(a_u, f_u, g_u, a_t, f_t, g_t);
}

// The next evaluation is requested at x_t; its transform and angle tables are built after the state machine returns
// (fulfil_request), with the six sine / cosine pairs computed on six lanes.
__device__ inline void request_eval(Ctl& c, const double* x, int mode) {
    (void)x;  // always c.x_t
    c.mode = mode;
    c.req = 1;
}
__device__ inline void fulfil_request(Ctl& c, const Trig& t) {
    pose_matrix_core(c.x_t, t.cf[0], t.sf[0], t.cf[1], t.sf[1], t.cf[2], t.sf[2], c.M);
    for (int i = 0; i < 16; ++i) c.final_T[i] = c.M[i];  // final_transformation_ follows every trial (:749-753,783-788)
    angle_tables_core(t.cd[0], t.sd[0], t.cd[1], t.sd[1], t.cd[2], t.sd[2], c.tab);
    c.req = 0;
}

__device__ inline void finish(Ctl& c, const AlignConsts& k, bool converged) {
    c.trans_probability = c.score / (double)k.n_src;
    c.converged = converged ? 1 : 0;
    c.done = 1;
}

// computeTransformation's loop body up to the first trial of the line search (:107-126, 701-760)
__device__ inline void newton_step(Ctl& c, const AlignConsts& k) {
    double ng[6], dp[6];
    for (int i = 0; i < 6; ++i) ng[i] = -c.g[i];
    const long long t0 = clock64();
    svd_solve6(c.H, ng, dp);
    c.solve_cycles += clock64() - t0;
    double dn = 0;
    for (int i = 0; i < 6; ++i) dn += dp[i] * dp[i];
    dn = sqrt(dn);
    if (dn == 0 || dn != dn) { finish(c, k, dn == dn); return; }
    for (int i = 0; i < 6; ++i) c.dir[i] = dp[i] / dn;
    // computeStepLengthMT prologue
    c.phi_0 = -c.score;
    double d_phi_0 = 0;
    for (int i = 0; i < 6; ++i) d_phi_0 += c.g[i] * c.dir[i];
    d_phi_0 = -d_phi_0;
    if (d_phi_0 >= 0) {
        if (d_phi_0 == 0) {  // no step: delta_p = 0 (:716-718)
            c.a_t = 0;
            c.step_iterations = 0;
            c.phase = -1;
            return;
        }
        d_phi_0 *= -1;
        for (int i = 0; i < 6; ++i) c.dir[i] *= -1;
    }
    c.d_phi_0 = d_phi_0;
    c.step_iterations = 0;
    const double mu = 1.e-4;
    c.step_max = k.step_size;
    c.step_min = k.trans_eps / 2;
    c.a_l = 0; c.a_u = 0;
    c.f_l = c.phi_0 - c.phi_0 - mu * d_phi_0 * c.a_l;
    c.g_l = d_phi_0 - mu * d_phi_0;
    c.f_u = c.phi_0 - c.phi_0 - mu * d_phi_0 * c.a_u;
    c.g_u = d_phi_0 - mu * d_phi_0;
    c.interval_converged = (c.step_max - c.step_min) < 0;
    c.open_interval = 1;
    double a_t = dn;
    a_t = fmin(a_t, c.step_max);
    a_t = fmax(a_t, c.step_min);
    c.a_t = a_t;
    for (int i = 0; i < 6; ++i) c.x_t[i] = c.p[i] + c.dir[i] * a_t;
    request_eval(c, c.x_t, MODE_DERIV_H);
    c.phase = PH_MT_FIRST;
}

// tail of computeTransformation's loop body (:129-141)
__device__ inline void finish_iteration(Ctl& c, const AlignConsts& k) {
    const double dn = c.a_t;
    for (int i = 0; i < 6; ++i) c.p[i] = c.p[i] + c.dir[i] * dn;
    bool conv = false;
    if (c.nr_iterations > k.max_iter || (c.nr_iterations && (fabs(dn) < k.trans_eps))) conv = true;
    c.nr_iterations++;
    if (conv) finish(c, k, true);
    else newton_step(c, k);
}

// `res` = the 43 (or 36) reduced sums of the evaluation that just finished
__device__ void advance(Ctl& c, const AlignConsts& k, const double* res) {
    const double mu = 1.e-4, nu = 0.9;
    const int mode = c.mode;
    if (mode == MODE_HESS_D) {
        c.hess_evals++;
        for (int i = 0; i < 36; ++i) c.H[i] = res[i];
    } else {
        c.evals++;
        c.score = res[0];
        for (int i = 0; i < 6; ++i) c.g[i] = res[1 + i];
        for (int i = 0; i < 36; ++i) c.H[i] = (mode == MODE_DERIV_H) ? res[7 + i] : 0.0;
    }
    switch (c.phase) {
        case PH_SINGLE_DERIV:
        case PH_SINGLE_HESS:
            c.done = 1;
            return;
        case PH_INIT:
            newton_step(c, k);
            break;
        case PH_MT_FIRST:
        case PH_MT_LOOP: {
            c.phi_t = -c.score;
            double d = 0;
            for (int i = 0; i < 6; ++i) d += c.g[i] * c.dir[i];
            c.d_phi_t = -d;
            c.psi_t = c.phi_t - c.phi_0 - mu * c.d_phi_0 * c.a_t;
            c.d_psi_t = c.d_phi_t - mu * c.d_phi_0;
            if (c.phase == PH_MT_LOOP) {  // rest of the while body after the evaluation (:793-823)
                if (c.open_interval && (c.psi_t <= 0 && c.d_psi_t >= 0)) {
                    c.open_interval = 0;
                    c.f_l = c.f_l + c.phi_0 - mu * c.d_phi_0 * c.a_l;
                    c.g_l = c.g_l + mu * c.d_phi_0;
                    c.f_u = c.f_u + c.phi_0 - mu * c.d_phi_0 * c.a_u;
                    c.g_u = c.g_u + mu * c.d_phi_0;
                }
                if (c.open_interval) c.interval_converged = mt_update_interval(c, c.psi_t, c.d_psi_t);
                else c.interval_converged = mt_update_interval(c, c.phi_t, c.d_phi_t);
                c.step_iterations++;
            }
            // while condition (:763)
            if (!c.interval_converged && c.step_iterations < 10 && !(c.psi_t <= 0 && c.d_phi_t <= -nu * c.d_phi_0)) {
                double a_t = c.open_interval ? mt_trial_value(c, c.psi_t, c.d_psi_t) : mt_trial_value(c, c.phi_t, c.d_phi_t);
                a_t = fmin(a_t, c.step_max);
                a_t = fmax(a_t, c.step_min);
                c.a_t = a_t;
                for (int i = 0; i < 6; ++i) c.x_t[i] = c.p[i] + c.dir[i] * a_t;
                request_eval(c, c.x_t, MODE_DERIV_NOH);
                c.phase = PH_MT_LOOP;
            } else if (c.step_iterations) {  // computeHessian with the final trial's cloud (:830)
                c.mode = MODE_HESS_D;
                c.phase = PH_MT_HESS;
            } else {
                finish_iteration(c, k);
            }
            break;
        }
        case PH_MT_HESS:
            finish_iteration(c, k);
            break;
    }
    while (c.phase == -1 && !c.done) {  // zero directional derivative: the line search returns step length 0 (:716-718)
        c.phase = -2;
        finish_iteration(c, k);
    }
}

// One level of the recursive-halving warp reduction of an N-vector held in v[0..N): lanes with bit MASK set keep the upper
// half [H, N) (moved to the front), the others the lower half [0, H); each adds what its partner hands over.  `base` is the
// original index of v[0], `len` how many entries of this lane's vector are real (the upper half is shorter when N is odd).
template <int N, int MASK>
__device__ __forceinline__ void halve_level(double (&v)[NACC], int lane, int& base, int& len) {
    constexpr int H = (N + 1) / 2;
    const bool up = (lane & MASK) != 0;
#pragma unroll
    for (int i = 0; i < H; ++i) {
        const double lo = v[i];
        const double hi = (i + H < N) ? v[i + H] : 0.0;
        const double keep = up ? hi : lo;
        const double send = up ? lo : hi;
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, MASK);
    }
    base += up ? H : 0;
    len = up ? max(len - H, 0) : min(len, H);
}

// ------------------------------------------------------------------ evaluation kernel
constexpr int kPairCap = 2048;  // (point, leaf) pairs a block can queue
struct EvalSmem {
    int2 pairs[kPairCap];
    int wcnt[2][EVAL_THREADS / 32];
    float M[12];
    AngleTables tab;
    int mode;
    double red[EVAL_THREADS / 32][NACC];
    double res[NACC];
    int is_last, abort;
    Trig trig;
};

// LOOP = false: one evaluation per launch (the host enqueues launches back to back; batched alignments, single derivative
// evaluations).  LOOP = true: ONE cooperative launch runs a whole alignment - after every evaluation the last block to
// arrive advances the state machine and releases a generation counter the other blocks wait on (all blocks are resident:
// the launch is cooperative and the grid is one wave), so an align pays neither launch gaps, nor no-op launches after
// convergence, nor done-flag polls from the host.  Control-block reads bypass L1 (ld.cg): it changes between evaluations.
// Alignment blockIdx.y = blocks 0 .. nbx-1 of grid row y.  PAIRS = false: one target and source, every row spans the grid
// (nbx = gridDim.x), partials [h][NACC][nbx].  PAIRS = true: independent (source, target) pairs (b200_ndt_pairs_align):
// row y = pair y with its own view pe[y].v (source range, n_src, cell2leaf base, grid bounds, KDTREE centroids) and its
// own block count pe[y].nbx, fixed by its own source size - blocks past it leave at once; partials [pairs][part_stride];
// one evaluation per launch.  The work split (items per block, the ticket that elects the last block, the fixed-order
// reduction) depends on nbx and the view alone.
struct PairEval {
    View v;
    int nbx;
};
template <bool LOOP, bool PAIRS = false>
__global__ void __launch_bounds__(EVAL_THREADS, 1) k_ndt_eval(View v_arg, Ctl* ctls, AlignConsts k_arg, double* partials /*[h][NACC][nbx]*/,
                                                              unsigned int* gen /*LOOP: generation counter, zero at launch*/, int max_evals,
                                                              const PairEval* __restrict__ pe = nullptr, int part_stride = 0) {
    Ctl* ctl = ctls + blockIdx.y;
    __shared__ EvalSmem sm;
    const int tid = threadIdx.x;
    __shared__ View pair_view;
    int pair_nbx = 0;
    AlignConsts pair_k = k_arg;
    if (PAIRS) {
        pair_nbx = __ldg(&pe[blockIdx.y].nbx);
        if ((int)blockIdx.x >= pair_nbx) return;
        static_assert(sizeof(View) % 4 == 0 && sizeof(View) / 4 <= EVAL_THREADS, "View is copied word by word");
        if (tid < (int)(sizeof(View) / 4)) ((int*)&pair_view)[tid] = __ldg((const int*)&pe[blockIdx.y].v + tid);
        __syncthreads();
        pair_k.n_src = pair_view.n_src;  // trans_probability = score / n_src of this pair
    }
    const View& v = PAIRS ? pair_view : v_arg;
    const AlignConsts& k = PAIRS ? pair_k : k_arg;
    const int nbx = PAIRS ? pair_nbx : gridDim.x;
    double* const part = partials + (size_t)blockIdx.y * part_stride;  // PAIRS only
  for (int ev = 0; ev < max_evals; ++ev) {
    if (__ldcg(&ctl->done)) return;
    if (tid < 12) sm.M[tid] = __ldcg(&ctl->M[tid]);
    for (int i = tid; i < (int)(sizeof(AngleTables) / 4); i += EVAL_THREADS) ((int*)&sm.tab)[i] = __ldcg((const int*)&ctl->tab + i);
    if (tid == 0) sm.mode = __ldcg(&ctl->mode);
    __syncthreads();
    const int mode = sm.mode;
    const int nitems = v.n_src * v.nst;
    double acc[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) acc[i] = 0.0;
    auto evaluate = [&](int i, int lf) {
        const float4 p = __ldg(v.src + i);
        float tx, ty, tz;
        xform(sm.M, p.x, p.y, p.z, tx, ty, tz);
        if (mode == MODE_HESS_D) {
            LeafD L;
            const double2* src = reinterpret_cast<const double2*>(v.leafD + lf);
            double2* dst = reinterpret_cast<double2*>(&L);
#pragma unroll
            for (int q = 0; q < 6; ++q) dst[q] = __ldg(src + q);
            hessian_pair_d(v, sm.tab, L, p.x, p.y, p.z, tx, ty, tz, *reinterpret_cast<double(*)[36]>(&acc[0]));
        } else {
            LeafF L;
            const float4* src = reinterpret_cast<const float4*>(v.leafF + lf);
            float4* dst = reinterpret_cast<float4*>(&L);
#pragma unroll
            for (int q = 0; q < 4; ++q) dst[q] = __ldg(src + q);
            deriv_pair_f(v, sm.tab, L, p.x, p.y, p.z, tx, ty, tz, mode == MODE_DERIV_H, acc);
        }
    };
    // Two thirds of the (point, neighbourhood cell) items hold no leaf.  Evaluating items in place leaves each warp
    // running as long as its unluckiest lane (3-4 evaluations of ~500 instructions where the mean is 1.3), so the block
    // first compacts its valid pairs into a shared-memory list - positions from ballots and a fixed scan over the warps:
    // deterministic, so the fp64 sums stay reproducible - and then takes the list 256 entries at a time.
    const int first = blockIdx.x * EVAL_THREADS, stride = nbx * EVAL_THREADS;
    const int rounds = first < nitems ? (nitems - first + stride - 1) / stride : 0;
    if (rounds * EVAL_THREADS <= kPairCap) {
        const int lane = tid & 31, warp = tid >> 5;
        int base = 0;
        for (int r = 0; r < rounds; ++r) {
            const int item = first + tid + r * stride;
            int i = 0, lf = -1;
            if (item < nitems) {
                i = item / v.nst;
                const int s = item - i * v.nst;
                const float4 p = __ldg(v.src + i);
                float tx, ty, tz;
                xform(sm.M, p.x, p.y, p.z, tx, ty, tz);
                lf = nbr_leaf(v, tx, ty, tz, s);
            }
            const unsigned bal = __ballot_sync(0xffffffffu, lf >= 0);
            if (lane == 0) sm.wcnt[r & 1][warp] = __popc(bal);
            __syncthreads();  // the other buffer is free again: every warp passed the barrier of the previous round
            int off = base, total = 0;
#pragma unroll
            for (int w = 0; w < EVAL_THREADS / 32; ++w) {
                const int c = sm.wcnt[r & 1][w];
                if (w < warp) off += c;
                total += c;
            }
            if (lf >= 0) sm.pairs[off + __popc(bal & ((1u << lane) - 1u))] = make_int2(i, lf);
            base += total;
        }
        __syncthreads();
        for (int e = tid; e < base; e += EVAL_THREADS) {
            const int2 pr = sm.pairs[e];
            evaluate(pr.x, pr.y);
        }
    } else {  // more items per block than the list holds (scans beyond ~40k points): in place
        for (int item = first + tid; item < nitems; item += stride) {
            const int i = item / v.nst, s = item - i * v.nst;
            const float4 p = __ldg(v.src + i);
            float tx, ty, tz;
            xform(sm.M, p.x, p.y, p.z, tx, ty, tz);
            const int lf = nbr_leaf(v, tx, ty, tz, s);
            if (lf >= 0) evaluate(i, lf);
        }
    }
    // block reduction in a fixed order.  Inside the warp: recursive halving - at every level a lane keeps one half of its
    // vector and hands the other half to its partner, so the 43 sums cost 22 + 11 + 6 + 3 + 2 = 44 exchanges instead of
    // 43 x 5, and end up spread over the lanes (two per lane); then the warps in index order.
    {
        const int lane = tid & 31;
        int base = 0, len = NACC;
        halve_level<NACC, 16>(acc, lane, base, len);
        halve_level<(NACC + 1) / 2, 8>(acc, lane, base, len);
        halve_level<((NACC + 1) / 2 + 1) / 2, 4>(acc, lane, base, len);
        halve_level<(((NACC + 1) / 2 + 1) / 2 + 1) / 2, 2>(acc, lane, base, len);
        halve_level<((((NACC + 1) / 2 + 1) / 2 + 1) / 2 + 1) / 2, 1>(acc, lane, base, len);
        static_assert((((((NACC + 1) / 2 + 1) / 2 + 1) / 2 + 1) / 2 + 1) / 2 == 2, "two sums per lane after five levels");
        if (len > 0) sm.red[tid >> 5][base] = acc[0];
        if (len > 1) sm.red[tid >> 5][base + 1] = acc[1];
    }
    __syncthreads();
    if (tid < NACC) {
        double a = sm.red[0][tid];
#pragma unroll
        for (int w = 1; w < EVAL_THREADS / 32; ++w) a += sm.red[w][tid];
        if (PAIRS) __stcg(part + (size_t)tid * nbx + blockIdx.x, a);
        else __stcg(partials + ((size_t)blockIdx.y * NACC + tid) * nbx + blockIdx.x, a);
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned t = atomicAdd(&ctl->ticket, 1u);
        sm.is_last = (t == (unsigned)nbx - 1u);
    }
    __syncthreads();
    if (!sm.is_last) {
        if (!LOOP) return;
        // wait for the last block to publish the next request (or the end of the alignment)
        if (tid == 0) {
            volatile unsigned int* g = gen;
            unsigned spins = 0;
            sm.abort = 0;
            while (*g == (unsigned)ev) {
                __nanosleep(64);
                if (++spins > (1u << 24)) { sm.abort = 1; break; }  // watchdog (~seconds): never hang the device
            }
            __threadfence();
        }
        __syncthreads();
        if (sm.abort) return;
        continue;
    }
    __threadfence();
    // The last block finishes the evaluation.  Everything below is a serial chain on ONE thread, so what matters is its
    // latency: (1) the partials are reduced by whole warps (lanes stride over the blocks, fixed shuffle tree: deterministic)
    // instead of 148 dependent L2 loads per column; (2) the control block is staged in shared memory, so the state machine's
    // many small reads and writes are 30-cycle shared-memory accesses instead of L2 round trips, and goes back in one
    // coalesced copy.
    static_assert(sizeof(Ctl) % 4 == 0, "Ctl is copied word by word");
    __shared__ Ctl sctl;
    for (int i = tid; i < (int)(sizeof(Ctl) / 4); i += EVAL_THREADS) ((int*)&sctl)[i] = __ldcg((const int*)ctl + i);
    {
        const int lane = tid & 31, warp = tid >> 5;
        for (int col = warp; col < NACC; col += EVAL_THREADS / 32) {
            const double* src = PAIRS ? part + (size_t)col * nbx : partials + ((size_t)blockIdx.y * NACC + col) * nbx;
            double a = 0.0;
            for (int b = lane; b < nbx; b += 32) a += __ldcg(src + b);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) sm.res[col] = a;
        }
    }
    __syncthreads();
    if (tid == 0) {
        sctl.ticket = 0;
        const long long t0 = clock64();
        advance(sctl, k, sm.res);
        sctl.step_cycles += clock64() - t0;
    }
    __syncthreads();
    if (sctl.req) {  // block-uniform
        if (tid < 6) trig_of_angle(sctl.x_t, tid, sm.trig);
        __syncthreads();
        if (tid == 0) fulfil_request(sctl, sm.trig);
        __syncthreads();
    }
    for (int i = tid; i < (int)(sizeof(Ctl) / 4); i += EVAL_THREADS) __stcg((int*)ctl + i, ((const int*)&sctl)[i]);
    if (!LOOP) return;
    __threadfence();
    __syncthreads();
    if (tid == 0) atomicAdd(gen, 1u);  // release: generation ev -> ev + 1
    __syncthreads();
  }
}

// one thread per alignment: computeTransformation prologue (:77-105)
__global__ void k_ndt_init(Ctl* ctls, int h, const float* __restrict__ guesses /*h x 16 col-major*/, const double* __restrict__ p_in /*h x 6 or null*/,
                           int phase) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= h) return;
    Ctl& c = ctls[a];
    c.done = 0; c.ticket = 0; c.phase = phase;
    c.nr_iterations = 0; c.converged = 0; c.evals = 0; c.hess_evals = 0;
    c.trans_probability = 0; c.score = 0; c.solve_cycles = 0; c.step_cycles = 0; c.req = 0;
    c.step_iterations = 0; c.a_t = 0;
    for (int i = 0; i < 6; ++i) { c.g[i] = 0; c.dir[i] = 0; c.x_t[i] = 0; }
    for (int i = 0; i < 36; ++i) c.H[i] = 0;
    if (phase == PH_INIT) {
        const float* G = guesses + (size_t)a * 16;
        float T[16];
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) T[i * 4 + j] = G[j * 4 + i];
        // align() starts from final_transformation_ = I and pre-applies the guess when it is not the identity (:83-88)
        for (int i = 0; i < 16; ++i) { c.M[i] = T[i]; c.final_T[i] = T[i]; }
        const float R[9] = {T[0], T[1], T[2], T[4], T[5], T[6], T[8], T[9], T[10]};
        float eul[3];
        euler_012(R, eul);
        c.p[0] = T[3]; c.p[1] = T[7]; c.p[2] = T[11];
        c.p[3] = eul[0]; c.p[4] = eul[1]; c.p[5] = eul[2];
        angle_tables(c.p, c.tab);
        c.mode = MODE_DERIV_H;
    } else {
        for (int i = 0; i < 6; ++i) c.p[i] = p_in[(size_t)a * 6 + i];
        pose_matrix(c.p, c.M);
        for (int i = 0; i < 16; ++i) c.final_T[i] = c.M[i];
        angle_tables(c.p, c.tab);
        c.mode = (phase == PH_SINGLE_HESS) ? MODE_HESS_D : MODE_DERIV_H;
    }
}

__global__ void k_ndt_count_done(const Ctl* ctls, int h, int* out) {
    int cnt = 0;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < h; a += gridDim.x * blockDim.x) cnt += ctls[a].done ? 0 : 1;
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(out, cnt);
}

// ------------------------------------------------------------------ calculateScore for a batch of poses (:836-880)
// grid = (point chunks, hypotheses): a block scores SCORE_CHUNK source points under one pose, fp64 throughout like the
// reference, and leaves one partial sum; k_ndt_score_finish adds the partials of a hypothesis in chunk order.  The points
// are read in the ordering of the pose's yaw bin: src_yaw + yaw_slot[bin] * n_src (yaw_bins = 0: the sensor order of v.src).
constexpr int SCORE_THREADS = 128;
constexpr int SCORE_CHUNK = 1024;

template <int NST>
__global__ void __launch_bounds__(SCORE_THREADS) k_ndt_score_batch(View v, const float* __restrict__ poses /*h x 16 col-major*/,
                                                                   const float4* __restrict__ src_yaw, const int32_t* __restrict__ yaw_slot, int yaw_bins,
                                                                   double* __restrict__ partial /*[h][nchunks]*/) {
    __shared__ float M[12];
    __shared__ double red[SCORE_THREADS / 32];
    __shared__ const float4* src_s;
    const int h = blockIdx.y, tid = threadIdx.x;
    if (tid < 12) M[tid] = poses[(size_t)h * 16 + (tid & 3) * 4 + (tid >> 2)];
    if (tid == 0) {
        src_s = v.src;
        if (yaw_bins) {  // Ndt::yaw_orderings() has built the bin of every pose of the batch; a missing one scores NaN
            const int slot = yaw_slot[score_yaw_bin(poses[(size_t)h * 16], poses[(size_t)h * 16 + 1], yaw_bins)];
            src_s = slot >= 0 ? src_yaw + (size_t)slot * v.n_src : nullptr;
        }
    }
    __syncthreads();
    const float4* __restrict__ src = src_s;
    if (!src) {
        if (tid == 0) partial[(size_t)h * gridDim.x + blockIdx.x] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    double acc = 0.0;
    const int i_end = min(v.n_src, (int)(blockIdx.x + 1) * SCORE_CHUNK);
    for (int i = blockIdx.x * SCORE_CHUNK + tid; i < i_end; i += SCORE_THREADS) {
        const float4 p = __ldg(src + i);
        float tx, ty, tz;
        xform(M, p.x, p.y, p.z, tx, ty, tz);
        int lf[NST];
        int cnt = 0;
        bool looked_up = false;
        if (NST == 7 && v.nbr7) {  // the whole neighbourhood with one 256-bit load when the point's own cell is inside the grid
            const int ix = (int)floorf(tx / v.leaf) - v.min_b[0], iy = (int)floorf(ty / v.leaf) - v.min_b[1], iz = (int)floorf(tz / v.leaf) - v.min_b[2];
            if (ix >= 0 && iy >= 0 && iz >= 0 && ix <= v.max_b[0] - v.min_b[0] && iy <= v.max_b[1] - v.min_b[1] && iz <= v.max_b[2] - v.min_b[2]) {
                const int* rec = v.nbr7 + ((size_t)ix * v.mul[0] + (size_t)iy * v.mul[1] + (size_t)iz * v.mul[2]) * 8;
                int r[8];
                asm volatile("ld.global.nc.v8.s32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                             : "l"(rec));
#pragma unroll
                for (int s = 0; s < NST; ++s) lf[s] = r[s < 7 ? s : 0];
                cnt = r[7];
                looked_up = true;
            }
        }
        if (!looked_up) {
#pragma unroll
            for (int s = 0; s < NST; ++s) {
                lf[s] = nbr_leaf(v, tx, ty, tz, s);
                cnt += lf[s] >= 0 ? 1 : 0;
            }
        }
        // score_inc / neighborhood.size() (:876): the size is inverted once per point (<= 1 ulp per term, far inside the
        // 1e-12 score tolerance) - the fp64 division was 13 % of this kernel's instructions
        const double rcnt = cnt > 0 ? 1.0 / (double)cnt : 0.0;
        // the quadratic form from the symmetric score store (ndt.cuh): 72 instead of 96 leaf bytes and 9 instead of 20
        // fp64 operations per pair; it differs from the reference's xt' C xt by rounding only (~1e-14 relative per term)
#pragma unroll
        for (int s = 0; s < NST; ++s) {
            if (lf[s] < 0) continue;
            const Dbl4 a = load_dbl4_256(v.sA + lf[s]);   // mean, c00
            const Dbl4 b = load_dbl4_256(v.sB + lf[s]);   // s01, s02, c11, s12
            const double c22 = __ldg(v.sC + lf[s]);
            const double x0 = (double)tx - a.x, x1 = (double)ty - a.y, x2 = (double)tz - a.z;
            const double q = fma(x0, fma(b.y, x2, fma(b.x, x1, a.w * x0)), fma(x1, fma(b.w, x2, b.z * x1), x2 * (c22 * x2)));
            const double e = exp(-v.d2 * q / 2);
            const double inc = -v.d1 * e - v.d3;
            acc += inc * rcnt;
        }
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((tid & 31) == 0) red[tid >> 5] = acc;
    __syncthreads();
    if (tid == 0) {
        double a = red[0];
#pragma unroll
        for (int w = 1; w < SCORE_THREADS / 32; ++w) a += red[w];
        partial[(size_t)h * gridDim.x + blockIdx.x] = a;
    }
}
__global__ void k_ndt_score_finish(const double* __restrict__ partial, int nchunks, int64_t h, int n_src, double* __restrict__ scores) {
    const int64_t a = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (a >= h) return;
    double s = 0.0;
    for (int c = 0; c < nchunks; ++c) s += partial[a * nchunks + c];
    scores[a] = s / (double)n_src;
}

// number of (point, voxel) pairs and probes of one evaluation at the poses' transforms (roofline bookkeeping)
__global__ void k_ndt_nbhd_total(View v, const float* __restrict__ M16_rowmajor, unsigned long long* out) {
    unsigned long long cnt = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < v.n_src; i += gridDim.x * blockDim.x) {
        const float4 p = __ldg(v.src + i);
        float tx, ty, tz;
        xform(M16_rowmajor, p.x, p.y, p.z, tx, ty, tz);
        for (int s = 0; s < v.nst; ++s) cnt += nbr_leaf(v, tx, ty, tz, s) >= 0 ? 1 : 0;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(out, cnt);
}

// same count for a batch of poses (col-major 4x4 each): grid = (point chunks, hypotheses)
__global__ void k_ndt_pairs_batch(View v, const float* __restrict__ poses, unsigned long long* out) {
    __shared__ float M[12];
    const int h = blockIdx.y;
    if (threadIdx.x < 12) M[threadIdx.x] = poses[(size_t)h * 16 + (threadIdx.x & 3) * 4 + (threadIdx.x >> 2)];
    __syncthreads();
    unsigned long long cnt = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < v.n_src; i += gridDim.x * blockDim.x) {
        const float4 p = __ldg(v.src + i);
        float tx, ty, tz;
        xform(M, p.x, p.y, p.z, tx, ty, tz);
        for (int s = 0; s < v.nst; ++s) cnt += nbr_leaf(v, tx, ty, tz, s) >= 0 ? 1 : 0;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(out, cnt);
}

// Order-preserving map double -> uint64 (NaN -> 0, below every real score)
__device__ __forceinline__ unsigned long long dbl_key(double s) {
    if (s != s) return 0ull;
    unsigned long long u = (unsigned long long)__double_as_longlong(s);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
// This rank's winner: pair[0] = highest score key of the slice, pair[1] = lowest global index holding it (one block)
__global__ void __launch_bounds__(256) k_local_best(const double* __restrict__ scores, int64_t h, int64_t h_begin, int64_t h_stride,
                                                    unsigned long long* __restrict__ pair) {
    __shared__ unsigned long long sk[256], si[256];
    unsigned long long bk = 0, bi = ~0ull;
    for (int64_t i = threadIdx.x; i < h; i += blockDim.x) {
        const unsigned long long key = dbl_key(scores[i]);
        if (key > bk) { bk = key; bi = (unsigned long long)(h_begin + i * h_stride); }  // ascending i per thread: ties keep the lower index
    }
    sk[threadIdx.x] = bk;
    si[threadIdx.x] = bi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            const unsigned long long k2 = sk[threadIdx.x + o], i2 = si[threadIdx.x + o];
            if (k2 > sk[threadIdx.x] || (k2 == sk[threadIdx.x] && i2 < si[threadIdx.x])) { sk[threadIdx.x] = k2; si[threadIdx.x] = i2; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { pair[0] = sk[0]; pair[1] = sk[0] ? si[0] : ~0ull; }
}

// ------------------------------------------------------------------ getFitnessScore: exact nearest neighbour in the target
// pcl::Registration::getFitnessScore(max_range) (PCL, third party; used by the loop-closure gate mapOptmization.cpp:693,719):
// mean over the transformed source points of the squared distance to their nearest target point (kd-tree nearestKSearch(1)
// = exact), points farther than max_range skipped.  The target is already sorted by voxel for the NDT build; a second
// dense table maps every non-empty cell to its run of points, and a warp searches cube shells of growing radius around
// the query until no unexplored cell can hold a closer point.
__global__ void k_ndt_cell_runs(const uint32_t* __restrict__ uniq, const int32_t* __restrict__ nruns, uint32_t sentinel, int32_t* __restrict__ cell2run) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= *nruns) return;
    if (uniq[r] != sentinel) cell2run[uniq[r]] = r;
}

struct FitView {
    const float4* pts;       // target points sorted by cell
    const int32_t* cell2run;
    const int32_t* run_off;
    const int32_t* run_cnt;
    int min_b[3], div_b[3];
    float leaf, inv_leaf;
};

// squared distance from (x, y, z) to its nearest target point; one warp, the result in every lane
__device__ __forceinline__ float fitness_nn(const FitView& f, float x, float y, float z, int lane) {
    float best = 3.402823466e+38f;
    if (isfinite(x) && isfinite(y) && isfinite(z)) {
        // start cell, clamped into the grid
        int c[3] = {(int)floorf(x * f.inv_leaf) - f.min_b[0], (int)floorf(y * f.inv_leaf) - f.min_b[1], (int)floorf(z * f.inv_leaf) - f.min_b[2]};
        const float qv[3] = {x, y, z};
#pragma unroll
        for (int a = 0; a < 3; ++a) c[a] = min(max(c[a], 0), f.div_b[a] - 1);
        const int rmax = max(max(f.div_b[0], f.div_b[1]), f.div_b[2]);
        for (int r = 0; r <= rmax; ++r) {
            // explored box [lo, hi] in cells; shell = box(r) minus box(r-1)
            int lo[3], hi[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) { lo[a] = max(c[a] - r, 0); hi[a] = min(c[a] + r, f.div_b[a] - 1); }
            const int nx = hi[0] - lo[0] + 1, ny = hi[1] - lo[1] + 1, nz = hi[2] - lo[2] + 1;
            const int ncell = nx * ny * nz;
            for (int i = 0; i < ncell; ++i) {  // warp-uniform walk over the box, shell cells only
                const int ix = lo[0] + i % nx, iy = lo[1] + (i / nx) % ny, iz = lo[2] + i / (nx * ny);
                if (r > 0 && abs(ix - c[0]) < r && abs(iy - c[1]) < r && abs(iz - c[2]) < r) continue;  // inner cells were done
                const int run = __ldg(f.cell2run + ((size_t)iz * f.div_b[1] + iy) * f.div_b[0] + ix);
                if (run < 0) continue;
                const int off = __ldg(f.run_off + run), cnt = __ldg(f.run_cnt + run);
                for (int j = lane; j < cnt; j += 32) {
                    const float4 t = __ldg(f.pts + off + j);
                    const float dx = x - t.x, dy = y - t.y, dz = z - t.z;
                    const float d2 = (dx * dx + dy * dy) + dz * dz;  // FLANN L2_Simple: sequential float accumulation
                    best = fminf(best, d2);
                }
            }
            float wb = best;
            for (int o = 16; o > 0; o >>= 1) wb = fminf(wb, __shfl_xor_sync(0xffffffffu, wb, o));
            best = wb;
            // lower bound on the distance to anything outside the explored box: nearest face that is not a grid face
            float lb = 3.402823466e+38f;
            bool all_grid = true;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (lo[a] > 0) { all_grid = false; lb = fminf(lb, qv[a] - (float)(lo[a] + f.min_b[a]) * f.leaf); }
                if (hi[a] < f.div_b[a] - 1) { all_grid = false; lb = fminf(lb, (float)(hi[a] + 1 + f.min_b[a]) * f.leaf - qv[a]); }
            }
            if (all_grid) break;
            // a small safety margin absorbs the rounding of the face coordinates
            if (lb > 0.f && best <= (lb - 1e-4f * f.leaf) * (lb - 1e-4f * f.leaf)) break;
        }
    }
    return best;
}

__global__ void __launch_bounds__(256) k_ndt_fitness(FitView f, const float4* __restrict__ src, int n, const float* __restrict__ M12g, double* __restrict__ d2_out) {
    __shared__ float M[12];
    if (threadIdx.x < 12) M[threadIdx.x] = M12g[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= n) return;
    const float4 p = __ldg(src + q);
    float x, y, z;
    xform(M, p.x, p.y, p.z, x, y, z);
    const float best = fitness_nn(f, x, y, z, lane);
    if (lane == 0) d2_out[q] = (double)best;
}

// Independent pairs: grid row y = pair y; its source range, its target index and its final transformation, read from its
// control block on the device (row-major; the first 12 floats are the 3x4 the source is moved by).
struct PairFit {
    FitView f;
    const float4* src;
    int n;
};
__global__ void __launch_bounds__(256) k_ndt_fitness_pairs(const PairFit* __restrict__ pf, const Ctl* __restrict__ ctls, const int64_t* __restrict__ d2_off,
                                                           double* __restrict__ d2_out) {
    __shared__ float M[12];
    if (threadIdx.x < 12) M[threadIdx.x] = ctls[blockIdx.y].final_T[threadIdx.x];
    __syncthreads();
    const PairFit& P = pf[blockIdx.y];
    const int lane = threadIdx.x & 31;
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q >= P.n) return;
    const float4 p = __ldg(P.src + q);
    float x, y, z;
    xform(M, p.x, p.y, p.z, x, y, z);
    const float best = fitness_nn(P.f, x, y, z, lane);
    if (lane == 0) d2_out[d2_off[blockIdx.y] + q] = (double)best;
}

// one block, fixed order: deterministic, and the same for a pair as for the single-target path
__device__ __forceinline__ void fitness_reduce_block(const double* __restrict__ d2, int n, double max_range, double* __restrict__ out /*sum, count*/) {
    __shared__ double ssum[256];
    __shared__ double scnt[256];
    double s = 0.0, c = 0.0;
    const int per = (n + blockDim.x - 1) / blockDim.x;
    const int b = threadIdx.x * per, e = min(n, b + per);
    for (int i = b; i < e; ++i) {
        const double v = d2[i];
        if (v <= max_range && v < 3.0e38) { s += v; c += 1.0; }
    }
    ssum[threadIdx.x] = s;
    scnt[threadIdx.x] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        double S = 0.0, C = 0.0;
        for (int i = 0; i < (int)blockDim.x; ++i) { S += ssum[i]; C += scnt[i]; }
        out[0] = S;
        out[1] = C;
    }
}
__global__ void k_ndt_fitness_reduce(const double* __restrict__ d2, int n, double max_range, double* __restrict__ out) {
    fitness_reduce_block(d2, n, max_range, out);
}
// block y = pair y: d2[d2_off[y] .. d2_off[y + 1]) -> out[2y], out[2y + 1]
__global__ void k_ndt_fitness_reduce_pairs(const double* __restrict__ d2, const int64_t* __restrict__ d2_off, double max_range, double* __restrict__ out) {
    const int64_t b = d2_off[blockIdx.x], e = d2_off[blockIdx.x + 1];
    fitness_reduce_block(d2 + b, (int)(e - b), max_range, out + 2 * blockIdx.x);
}

// ------------------------------------------------------------------ host object
struct Ndt {
    b200_ndt_params prm;
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    bool coop_launch = false;  // device supports cooperative launches (one-launch align)
    int eval_blocks_per_sm = 0;
    // target
    GridDims gd{};
    int64_t ncells = 0;
    int nruns = 0, n_valid = 0;
    DevBuf<float4> d_tgt, d_src, d_src_raw, d_tgt_sorted;
    DevBuf<uint32_t> s_keys_in, s_keys_out;
    DevBuf<int32_t> s_vals_in, s_vals_out, d_cell2run;
    // score kernel only: the orderings of the yaw bins built so far for this source, slot by slot ([slots][n_src])
    int yaw_bins = 0, yaw_built = 0;  // bins of this source (0: sensor order), orderings built
    int yaw_calls = 0;                // score calls on this source so far
    std::vector<int32_t> yaw_slot;    // bin -> slot in d_src_yaw, or -1 (mirrored in d_yaw_slot)
    DevBuf<float4> d_src_yaw;
    DevBuf<int32_t> d_yaw_slot, d_yaw_need, d_yaw_list;
    PinnedBuf<int32_t> h_yaw;         // [0, MAX): need, [MAX, 2 MAX): slot table, [2 MAX, 3 MAX): bins to build
    DevBuf<uint64_t> y_keys_in, y_keys_out;
    DevBuf<int32_t> y_vals_in, y_vals_out;
    DevBuf<uint8_t> s_tmp;
    DevBuf<double> d_fit;
    bool have_fitness_index = false;
    int64_t n_tgt = 0;
    DevBuf<int32_t> d_cell2leaf, d_nbr7;
    DevBuf<LeafF> d_leafF;
    DevBuf<LeafD> d_leafD;
    DevBuf<Dbl4> d_sA, d_sB;   // score store (k_ndt_score_store)
    DevBuf<double> d_sC;
    DevBuf<double> d_cov, d_sums;
    DevBuf<float> d_centroid;
    DevBuf<int32_t> d_npts, d_vals_in, d_vals_out, d_run_cnt, d_run_off, d_small;
    DevBuf<uint32_t> d_keys_in, d_keys_out, d_uniq;
    DevBuf<uint8_t> d_valid, cub_tmp;
    PinnedBuf<float4> h_stage;
    PinnedBuf<int32_t> h_small;
    int n_src = 0;
    bool have_target = false, have_nbr7 = false;
    // align
    DevBuf<Ctl> d_ctl;
    DevBuf<double> d_partials, d_p_in, d_scores;
    DevBuf<float> d_poses;
    PinnedBuf<Ctl> h_ctl;
    PinnedBuf<double> h_scores;
    PinnedBuf<float> h_poses;
    DevBuf<unsigned long long> d_best, d_bar;
    PinnedBuf<unsigned long long> h_best;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t evs0 = nullptr, evs1 = nullptr;  // around the score kernel alone (roofline of k_ndt_score_batch)
    // upload of page-locked caller clouds: copy stream + a ring of chunk events
    static constexpr int kChunkEvents = 9;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_chunk[kChunkEvents] = {};
    DevBuf<uint8_t> d_raw;
    double d1 = 0, d2 = 0, d3 = 0;
    float last_ms = 0.f;
    int last_launches = 0;

    int32_t init(const b200_ndt_params* p, int dev);
    void destroy();
    void gauss();
    int nst() const { return prm.search == 0 ? 27 : prm.search; }  // stencil cells per point (KDTREE filters the 27-cell block by centroid distance)
    View view() const;
    int32_t upload(const float* xyz, int64_t n, int64_t stride, DevBuf<float4>& dst);
    int32_t set_target(const float* xyz, int64_t n, int64_t stride);
    int32_t build_target(int64_t n);
    int32_t set_source(const float* xyz, int64_t n, int64_t stride);
    int32_t run(int h, const float* d_guesses, const double* d_p, int phase);
    template <class Launch>
    int32_t until_done(int h, int max_launches, int& launches, Launch launch);
    int32_t yaw_orderings(const float* d_poses16, int64_t h);
    int32_t score_batch_device(const float* d_poses16, int64_t h, double* d_out);
    int32_t fitness(const float* T16_colmajor, double max_range, double* score, int64_t* nr);
};

int32_t Ndt::init(const b200_ndt_params* p, int dev) {
    prm = *p;
    if (!(prm.resolution > 0.f)) B200_FAIL(B200_ERR_ARG, "resolution must be > 0");
    if (prm.search != 1 && prm.search != 27 && prm.search != 0) prm.search = 7;  // 0 = KDTREE, 1 / 7 / 27 = DIRECT1 / DIRECT7 / DIRECT26
    if (prm.min_pts <= 0) prm.min_pts = 6;
    if (!(prm.eig_ratio > 0)) prm.eig_ratio = 0.01;
    device = dev;
    CUDA_SET_DEVICE(dev);
    CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    sm_count = prop.multiProcessorCount;
    coop_launch = prop.cooperativeLaunch != 0;
    CUDA_TRY(cudaEventCreate(&ev0));
    CUDA_TRY(cudaEventCreate(&ev1));
    CUDA_TRY(cudaEventCreate(&evs0));
    CUDA_TRY(cudaEventCreate(&evs1));
    CUDA_TRY(d_small.reserve(16));
    CUDA_TRY(h_small.reserve(16));
    CUDA_TRY(d_best.reserve(4));
    CUDA_TRY(h_best.reserve(4));
    gauss();
    return B200_OK;
}

void Ndt::destroy() {
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
    d_tgt.release(); d_src.release(); d_src_raw.release(); d_tgt_sorted.release(); s_keys_in.release(); s_keys_out.release();
    s_vals_in.release(); s_vals_out.release(); d_src_yaw.release(); d_yaw_slot.release(); d_yaw_need.release(); d_yaw_list.release(); h_yaw.release(); y_keys_in.release(); y_keys_out.release(); y_vals_in.release(); y_vals_out.release(); d_cell2run.release(); s_tmp.release(); d_fit.release(); d_cell2leaf.release(); d_nbr7.release(); d_leafF.release(); d_leafD.release(); d_sA.release(); d_sB.release(); d_sC.release(); d_cov.release(); d_sums.release(); d_centroid.release();
    d_npts.release(); d_vals_in.release(); d_vals_out.release(); d_run_cnt.release(); d_run_off.release(); d_small.release();
    d_keys_in.release(); d_keys_out.release(); d_uniq.release(); d_valid.release(); cub_tmp.release();
    h_stage.release(); h_small.release(); d_ctl.release(); d_partials.release(); d_p_in.release(); d_scores.release(); d_poses.release();
    h_ctl.release(); h_scores.release(); h_poses.release(); d_best.release(); d_bar.release(); h_best.release();
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (evs0) cudaEventDestroy(evs0);
    if (evs1) cudaEventDestroy(evs1);
    if (copy_stream) {
        cudaStreamSynchronize(copy_stream);
        for (auto& e : ev_chunk) if (e) cudaEventDestroy(e);
        cudaStreamDestroy(copy_stream);
        copy_stream = nullptr;
    }
    d_raw.release();
    if (stream) cudaStreamDestroy(stream);
    stream = nullptr;
}

void Ndt::gauss() {  // ndt_omp_impl.hpp:77-81
    const double c1 = 10 * (1 - prm.outlier_ratio);
    const double c2 = prm.outlier_ratio / std::pow((double)prm.resolution, 3);
    d3 = -std::log(c2);
    d1 = -std::log(c1 + c2) - d3;
    d2 = -2 * std::log((-std::log(c1 * std::exp(-0.5) + c2) - d3) / d1);
}

View Ndt::view() const {
    View v;
    v.src = d_src.p; v.n_src = n_src;
    v.cell2leaf = d_cell2leaf.p; v.leafF = d_leafF.p; v.leafD = d_leafD.p;
    v.sA = d_sA.p; v.sB = d_sB.p; v.sC = d_sC.p;
    v.nbr7 = have_nbr7 ? d_nbr7.p : nullptr;
    for (int k = 0; k < 3; ++k) { v.min_b[k] = gd.min_b[k]; v.max_b[k] = gd.max_b[k]; v.mul[k] = gd.mul[k]; }
    v.leaf = prm.resolution;
    v.nst = nst();
    v.kdtree = prm.search == 0 ? 1 : 0;
    v.kd_r2 = (float)((double)prm.resolution * (double)prm.resolution);
    v.centroid = d_centroid.p;
    v.d1 = d1; v.d2 = d2; v.d3 = d3;
    return v;
}

// strided host cloud -> pinned float4 staging -> device, in chunks: while chunk c crosses PCIe, chunk c+1 is being packed
// by a few host threads
// strided xyz records -> float4 (x, y, z, 0), for clouds that crossed PCIe as the caller laid them out
__global__ void k_ndt_unpack(const uint8_t* __restrict__ raw, int64_t stride, int64_t n, float4* __restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = reinterpret_cast<const float*>(raw + i * stride);
    dst[i] = make_float4(p[0], p[1], p[2], 0.0f);
}

// Host cloud -> device float4.
//  * page-locked caller memory (b200_host_alloc, cudaHostRegister) with records of at most 16 bytes: the raw bytes cross PCIe
//    straight from the caller's buffer in 1M-point chunks on a copy stream and are unpacked on the device, chunk c while
//    chunk c + 1 is still in flight - no host pass over the cloud at all (a 10M-point xyz cloud is 120 MB = ~2.3 ms of PCIe);
//  * anything else: packed into the pinned stage by a few host threads, chunk c + 1 while chunk c crosses PCIe.
int32_t Ndt::upload(const float* xyz, int64_t n, int64_t stride, DevBuf<float4>& dst) {
    CUDA_TRY(dst.reserve((size_t)n));
    const int64_t chunk = 1 << 20;
    cudaPointerAttributes at{};
    const bool pinned = stride % 4 == 0 && stride <= 16 && cudaPointerGetAttributes(&at, xyz) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();  // cudaPointerGetAttributes on plain malloc memory may leave an error behind on old drivers
    if (pinned) {
        const size_t raw_bytes = (size_t)(n - 1) * stride + 12;
        CUDA_TRY(d_raw.reserve(raw_bytes));
        if (!copy_stream) {
            CUDA_TRY(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
            for (auto& e : ev_chunk) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        CUDA_TRY(cudaEventRecord(ev_chunk[0], stream));           // the copy stream starts after whatever used d_raw / dst before
        CUDA_TRY(cudaStreamWaitEvent(copy_stream, ev_chunk[0], 0));
        int c = 0;
        for (int64_t c0 = 0; c0 < n; c0 += chunk, ++c) {
            const int64_t c1 = std::min<int64_t>(n, c0 + chunk);
            const size_t b0 = (size_t)c0 * stride, b1 = c1 == n ? raw_bytes : (size_t)c1 * stride;
            CUDA_TRY(cudaMemcpyAsync(d_raw.p + b0, (const uint8_t*)xyz + b0, b1 - b0, cudaMemcpyHostToDevice, copy_stream));
            cudaEvent_t ev = ev_chunk[1 + c % (kChunkEvents - 1)];
            CUDA_TRY(cudaEventRecord(ev, copy_stream));
            CUDA_TRY(cudaStreamWaitEvent(stream, ev, 0));
            k_ndt_unpack<<<(unsigned)((c1 - c0 + 255) / 256), 256, 0, stream>>>(d_raw.p + b0, stride, c1 - c0, dst.p + c0);
            LAUNCH_COUNT(1);
        }
        return B200_OK;
    }
    CUDA_TRY(h_stage.reserve((size_t)n));
    const int nt = n > chunk ? 8 : 1;
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t c1 = std::min<int64_t>(n, c0 + chunk);
        if (nt == 1) pack_xyz_float4((const float*)((const char*)xyz + c0 * stride), c1 - c0, stride, h_stage.p + c0);
        else {
            std::vector<std::thread> th;
            const int64_t per = (c1 - c0 + nt - 1) / nt;
            for (int t = 0; t < nt; ++t) {
                const int64_t b = c0 + t * per, e = std::min<int64_t>(c1, b + per);
                if (b >= e) break;
                th.emplace_back([=]() { pack_xyz_float4((const float*)((const char*)xyz + b * stride), e - b, stride, h_stage.p + b); });
            }
            for (auto& t : th) t.join();
        }
        CUDA_TRY(cudaMemcpyAsync(dst.p + c0, h_stage.p + c0, (size_t)(c1 - c0) * sizeof(float4), cudaMemcpyHostToDevice, stream));
    }
    return B200_OK;
}

int32_t Ndt::set_target(const float* xyz, int64_t n, int64_t stride) {
    if (n < 1 || !xyz || stride < 12) B200_FAIL(B200_ERR_ARG, "bad target cloud");
    if (n > (int64_t)0x7fffff00) B200_FAIL(B200_ERR_ARG, "target cloud too large");
    CUDA_SET_DEVICE(device);
    int32_t rc = upload(xyz, n, stride, d_tgt);
    if (rc) return rc;
    return build_target(n);
}

// applyFilter's grid (:67-103) from the min / max of the finite points (ordered ints, as k_ndt_minmax leaves them)
static int32_t grid_from_minmax(const int* mm6, float resolution, GridDims& gd, int64_t& ncells) {
    float mn[3], mx[3];
    for (int k = 0; k < 3; ++k) {
        int a = mm6[k], b = mm6[3 + k];
        a = a >= 0 ? a : a ^ 0x7fffffff;
        b = b >= 0 ? b : b ^ 0x7fffffff;
        memcpy(&mn[k], &a, 4);
        memcpy(&mx[k], &b, 4);
    }
    if (!(mn[0] <= mx[0])) B200_FAIL(B200_ERR_ARG, "target cloud has no finite point");
    const float inv_leaf = 1.0f / resolution;
    const int64_t dx = (int64_t)((mx[0] - mn[0]) * inv_leaf) + 1, dy = (int64_t)((mx[1] - mn[1]) * inv_leaf) + 1,
                  dz = (int64_t)((mx[2] - mn[2]) * inv_leaf) + 1;
    if ((double)dx * (double)dy * (double)dz > (double)INT32_MAX) B200_FAIL(B200_ERR_RANGE, "leaf size too small for the target: integer leaf indices would overflow");
    gd.inv_leaf = inv_leaf;
    for (int k = 0; k < 3; ++k) {
        gd.min_b[k] = (int)std::floor(mn[k] * inv_leaf);
        gd.max_b[k] = (int)std::floor(mx[k] * inv_leaf);
        gd.div_b[k] = gd.max_b[k] - gd.min_b[k] + 1;
    }
    gd.mul[0] = 1; gd.mul[1] = gd.div_b[0]; gd.mul[2] = gd.div_b[0] * gd.div_b[1];
    ncells = (int64_t)gd.div_b[0] * gd.div_b[1] * gd.div_b[2];
    if (ncells > ((int64_t)1 << 30)) B200_FAIL(B200_ERR_RANGE, "NDT grid too large for the dense cell table (> 2^30 cells)");
    return B200_OK;
}

int32_t Ndt::build_target(int64_t n) {
    have_target = false;
    have_fitness_index = false;
    n_tgt = n;
    CUDA_TRY(cudaEventRecord(ev0, stream));
    int* mm = d_small.p;
    k_ndt_minmax_init<<<1, 32, 0, stream>>>(mm);
    k_ndt_minmax<<<sm_count * 8, 256, 0, stream>>>(d_tgt.p, n, mm);
    CUDA_TRY(cudaMemcpyAsync(h_small.p, mm, 6 * sizeof(int), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    const int32_t grc = grid_from_minmax(h_small.p, prm.resolution, gd, ncells);
    if (grc) return grc;
    CUDA_TRY(d_cell2leaf.reserve((size_t)ncells));
    CUDA_TRY(cudaMemsetAsync(d_cell2leaf.p, 0xFF, (size_t)ncells * sizeof(int32_t), stream));
    CUDA_TRY(d_keys_in.reserve(n)); CUDA_TRY(d_keys_out.reserve(n)); CUDA_TRY(d_uniq.reserve(n));
    CUDA_TRY(d_vals_in.reserve(n)); CUDA_TRY(d_vals_out.reserve(n)); CUDA_TRY(d_run_cnt.reserve(n)); CUDA_TRY(d_run_off.reserve(n));
    const int nb = (int)((n + 255) / 256);
    const uint32_t sentinel = (uint32_t)ncells;  // key of non-finite points: one past the last leaf id, sorts last
    k_ndt_keys<<<nb, 256, 0, stream>>>(d_tgt.p, (int)n, gd, sentinel, d_keys_in.p, d_vals_in.p);
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) <= ncells) ++end_bit;
    size_t t1 = 0, t2 = 0, t3 = 0;
    int32_t* d_nruns = d_small.p + 8;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, d_keys_in.p, d_keys_out.p, d_vals_in.p, d_vals_out.p, (int)n, 0, end_bit, stream);
    cub::DeviceRunLengthEncode::Encode(nullptr, t2, d_keys_out.p, d_uniq.p, d_run_cnt.p, d_nruns, (int)n, stream);
    cub::DeviceScan::ExclusiveSum(nullptr, t3, d_run_cnt.p, d_run_off.p, (int)n, stream);
    size_t tmp = std::max(t1, std::max(t2, t3));
    CUDA_TRY(cub_tmp.reserve(tmp));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp.p, tmp, d_keys_in.p, d_keys_out.p, d_vals_in.p, d_vals_out.p, (int)n, 0, end_bit, stream));
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(cub_tmp.p, tmp, d_keys_out.p, d_uniq.p, d_run_cnt.p, d_nruns, (int)n, stream));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(cub_tmp.p, tmp, d_run_cnt.p, d_run_off.p, (int)n, stream));
    CUDA_TRY(cudaMemcpyAsync(h_small.p, d_nruns, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    nruns = h_small.p[0];
    CUDA_TRY(d_sums.reserve((size_t)nruns * 9));
    CUDA_TRY(d_centroid.reserve((size_t)nruns * 3 + 4));
    CUDA_TRY(d_leafF.reserve(nruns)); CUDA_TRY(d_leafD.reserve(nruns)); CUDA_TRY(d_cov.reserve((size_t)nruns * 9));
    CUDA_TRY(d_sA.reserve(nruns)); CUDA_TRY(d_sB.reserve(nruns)); CUDA_TRY(d_sC.reserve(nruns));
    CUDA_TRY(d_npts.reserve(nruns)); CUDA_TRY(d_valid.reserve(nruns));
    int32_t* d_nvalid = d_small.p + 9;
    CUDA_TRY(cudaMemsetAsync(d_nvalid, 0, sizeof(int32_t), stream));
    CUDA_TRY(cudaMemsetAsync(d_cov.p, 0, (size_t)nruns * 9 * sizeof(double), stream));
    const int acc_blocks = std::min((nruns + 7) / 8, sm_count * 8);
    k_ndt_accumulate<<<std::max(acc_blocks, 1), 256, 0, stream>>>(d_tgt.p, d_vals_out.p, d_uniq.p, d_run_off.p, d_run_cnt.p, d_nruns, sentinel, d_sums.p, d_centroid.p);
    k_ndt_finalize<<<(nruns + 127) / 128, 128, 0, stream>>>(d_uniq.p, d_run_cnt.p, d_nruns, sentinel, d_sums.p, prm.min_pts, prm.eig_ratio, d_leafF.p,
                                                            d_leafD.p, d_cov.p, d_npts.p, d_valid.p, d_cell2leaf.p, d_nvalid);
    k_ndt_score_store<<<(nruns + 127) / 128, 128, 0, stream>>>(d_leafD.p, d_valid.p, nruns, d_sA.p, d_sB.p, d_sC.p);
    LAUNCH_COUNT(6);
    have_nbr7 = prm.search == 7 && ncells <= ((int64_t)1 << 26);  // 32 B per cell: at most 2 GB
    if (have_nbr7) {
        CUDA_TRY(d_nbr7.reserve((size_t)ncells * 8));
        k_ndt_build_nbr7<<<(unsigned)((ncells + 255) / 256), 256, 0, stream>>>(d_cell2leaf.p, ncells, gd.div_b[0], gd.div_b[1], gd.div_b[2], d_nbr7.p);
        LAUNCH_COUNT(1);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ev1, stream));
    CUDA_TRY(cudaMemcpyAsync(h_small.p, d_nvalid, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    n_valid = h_small.p[0];
    cudaEventElapsedTime(&last_ms, ev0, ev1);
    have_target = true;
    return B200_OK;
}

int32_t Ndt::set_source(const float* xyz, int64_t n, int64_t stride) {
    if (n < 1 || !xyz || stride < 12 || n > (1 << 28)) B200_FAIL(B200_ERR_ARG, "bad source cloud");
    CUDA_SET_DEVICE(device);
    // the score kernel's per-yaw orderings of the previous source are void; they are built again on demand
    yaw_bins = 0;
    yaw_built = 0;
    yaw_calls = 0;
    yaw_slot.clear();
    int32_t rc = upload(xyz, n, stride, d_src_raw);
    if (rc) return rc;
    CUDA_TRY(d_src.reserve((size_t)n));
    CUDA_TRY(s_keys_in.reserve(n)); CUDA_TRY(s_keys_out.reserve(n)); CUDA_TRY(s_vals_in.reserve(n)); CUDA_TRY(s_vals_out.reserve(n));
    const int nb = (int)((n + 255) / 256);
    k_ndt_source_keys<<<nb, 256, 0, stream>>>(d_src_raw.p, (int)n, 1.0f / prm.resolution, s_keys_in.p, s_vals_in.p);
    size_t tmp = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp, s_keys_in.p, s_keys_out.p, s_vals_in.p, s_vals_out.p, (int)n, 0, 32, stream));
    CUDA_TRY(s_tmp.reserve(tmp));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(s_tmp.p, tmp, s_keys_in.p, s_keys_out.p, s_vals_in.p, s_vals_out.p, (int)n, 0, 32, stream));
    k_ndt_gather<<<nb, 256, 0, stream>>>(d_src_raw.p, s_vals_out.p, (int)n, d_src.p);
    LAUNCH_COUNT(2);
    int bins = 0;
    for (int nb = YAW_BINS_MAX; nb >= 2; nb >>= 1)
        if (n * nb * (int64_t)sizeof(float4) <= YAW_ORDER_MAX_BYTES) { bins = nb; break; }
    if (bins) {
        CUDA_TRY(d_yaw_slot.reserve(YAW_BINS_MAX)); CUDA_TRY(d_yaw_need.reserve(YAW_BINS_MAX)); CUDA_TRY(d_yaw_list.reserve(YAW_BINS_MAX));
        CUDA_TRY(h_yaw.reserve(3 * YAW_BINS_MAX));
        CUDA_TRY(cudaMemsetAsync(d_yaw_slot.p, 0xFF, YAW_BINS_MAX * sizeof(int32_t), stream));
    }
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    yaw_bins = bins;
    yaw_slot.assign(bins, -1);
    n_src = (int)n;
    return B200_OK;
}

// Enqueues evaluations of the h alignments in d_ctl until every one is done (or max_launches): batches of launches between
// polls of the done count.
template <class Launch>
int32_t Ndt::until_done(int h, int max_launches, int& launches, Launch launch) {
    int* d_left = d_small.p + 10;
    while (launches - 1 < max_launches) {
        // first poll after 12 evaluations: a typical relocalization align (8 iterations, 9-10 evaluations) then ends with one
        // poll and two or three no-op launches instead of two polls and seven no-ops
        const int batch = launches == 1 ? LAUNCH_BATCH + 4 : LAUNCH_BATCH;
        for (int b = 0; b < batch; ++b) launch();
        launches += batch;
        CUDA_TRY(cudaMemsetAsync(d_left, 0, sizeof(int), stream));
        k_ndt_count_done<<<std::min((h + 255) / 256, 64), 256, 0, stream>>>(d_ctl.p, h, d_left);
        ++launches;
        CUDA_TRY(cudaMemcpyAsync(h_small.p, d_left, sizeof(int), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (h_small.p[0] == 0) break;
    }
    return B200_OK;
}

// Runs h independent state machines to completion.  d_guesses (h x 16, col-major) for PH_INIT, d_p (h x 6) otherwise.
int32_t Ndt::run(int h, const float* d_guesses, const double* d_p, int phase) {
    if (!have_target) B200_FAIL(B200_ERR_ARG, "no target set");
    if (n_src < 1) B200_FAIL(B200_ERR_ARG, "no source set");
    CUDA_TRY(d_ctl.reserve(h));
    CUDA_TRY(h_ctl.reserve(h));
    const int64_t items = (int64_t)n_src * nst();
    if (!eval_blocks_per_sm) {
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&eval_blocks_per_sm, k_ndt_eval<false>, EVAL_THREADS, 0));
        if (eval_blocks_per_sm < 1) eval_blocks_per_sm = 1;
    }
    // one resident wave: blocks of all alignments together fill the SMs once (grid-stride inside)
    int nbx = (int)std::min<int64_t>((items + EVAL_THREADS - 1) / EVAL_THREADS, (int64_t)std::max(1, eval_blocks_per_sm * sm_count / h));
    if (nbx < 1) nbx = 1;
    CUDA_TRY(d_partials.reserve((size_t)h * NACC * nbx));
    gauss();  // recomputed at every computeTransformation (ndt_omp_impl.hpp:77-81)
    const View v = view();
    AlignConsts k{prm.step_size, prm.trans_eps, prm.max_iter, n_src};
    CUDA_TRY(cudaEventRecord(ev0, stream));
    k_ndt_init<<<(h + 63) / 64, 64, 0, stream>>>(d_ctl.p, h, d_guesses, d_p, phase);
    int launches = 1;
    const bool single = phase != PH_INIT;
    // worst case per alignment: (max_iter + 2) iterations x (1 + 10 trials + 1 Hessian) evaluations
    const int max_launches = single ? 1 : (prm.max_iter + 3) * 12 + 1;
    static const bool persistent_ok = !(getenv("B200_NDT_LOOP") && atoi(getenv("B200_NDT_LOOP")) == 0);
    if (!single && h == 1 && persistent_ok && coop_launch) {  // one alignment: the whole Newton / line-search loop in one launch
        unsigned int* d_gen = (unsigned int*)(d_small.p + 11);
        CUDA_TRY(cudaMemsetAsync(d_gen, 0, sizeof(unsigned int), stream));
        Ctl* ctls = d_ctl.p;
        double* parts = d_partials.p;
        int max_evals = max_launches;
        const PairEval* no_pairs = nullptr;
        int no_stride = 0;
        void* args[] = {(void*)&v, (void*)&ctls, (void*)&k, (void*)&parts, (void*)&d_gen, (void*)&max_evals, (void*)&no_pairs, (void*)&no_stride};
        CUDA_TRY(cudaLaunchCooperativeKernel((const void*)k_ndt_eval<true>, dim3(nbx, 1), dim3(EVAL_THREADS), args, 0, stream));
        ++launches;
    } else if (single) {
        k_ndt_eval<false><<<dim3(nbx, h), EVAL_THREADS, 0, stream>>>(v, d_ctl.p, k, d_partials.p, nullptr, 1);
        ++launches;
    } else {
        const int32_t rc = until_done(h, max_launches, launches, [&]() {
            k_ndt_eval<false><<<dim3(nbx, h), EVAL_THREADS, 0, stream>>>(v, d_ctl.p, k, d_partials.p, nullptr, 1);
        });
        if (rc) return rc;
    }
    CUDA_TRY(cudaEventRecord(ev1, stream));
    CUDA_TRY(cudaMemcpyAsync(h_ctl.p, d_ctl.p, (size_t)h * sizeof(Ctl), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    cudaEventElapsedTime(&last_ms, ev0, ev1);
    LAUNCH_COUNT(launches);
    last_launches = launches;
    if (!single)
        for (int a = 0; a < h; ++a)
            if (!h_ctl.p[a].done) B200_FAIL(B200_ERR_CUDA, "NDT alignment did not run to completion (evaluation bound or barrier watchdog)");
    return B200_OK;
}

// Builds the orderings of the yaw bins of the h poses that this source does not have yet: one stable sort by
// (bin, Morton key) over all of them, one gather into the next free slots.  A call first reads back which bins its poses
// need (one round trip, ~20 us) and builds only the missing ones, so a source scored once pays for the bins of that batch
// alone (4 bins for a 4-yaw relocalization grid: an 80k-key sort).  From the second call on, a batch of at least as many
// poses as bins builds every missing bin at once without the read-back; later calls then return at once.  Which bins
// exist never changes a score.
int32_t Ndt::yaw_orderings(const float* d_poses16, int64_t h) {
    if (!yaw_bins || yaw_built == yaw_bins) return B200_OK;
    int32_t* need = h_yaw.p;
    int32_t* slot = h_yaw.p + YAW_BINS_MAX;
    int32_t* list = h_yaw.p + 2 * YAW_BINS_MAX;  // the callers synchronise before they return: no copy from it is pending
    int m = 0;
    const bool all = h >= yaw_bins && yaw_calls > 0;
    ++yaw_calls;
    if (all) {
        for (int b = 0; b < yaw_bins; ++b)
            if (yaw_slot[b] < 0) list[m++] = b;
    } else {
        CUDA_TRY(cudaMemsetAsync(d_yaw_need.p, 0, yaw_bins * sizeof(int32_t), stream));
        k_ndt_yaw_need<<<(unsigned)std::min<int64_t>((h + 255) / 256, 64), 256, 0, stream>>>(d_poses16, h, yaw_bins, d_yaw_need.p);
        LAUNCH_COUNT(1);
        CUDA_TRY(cudaMemcpyAsync(need, d_yaw_need.p, yaw_bins * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        for (int b = 0; b < yaw_bins; ++b)
            if (need[b] && yaw_slot[b] < 0) list[m++] = b;
    }
    if (!m) return B200_OK;
    const int64_t n = n_src, ny = n * m;
    CUDA_TRY(d_src_yaw.reserve_keep((size_t)(yaw_built + m) * n, (size_t)yaw_built * n, stream, yaw_built + m == yaw_bins));
    CUDA_TRY(y_keys_in.reserve(ny)); CUDA_TRY(y_keys_out.reserve(ny)); CUDA_TRY(y_vals_in.reserve(ny)); CUDA_TRY(y_vals_out.reserve(ny));
    CUDA_TRY(cudaMemcpyAsync(d_yaw_list.p, list, m * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
    k_ndt_source_keys_yaw<<<dim3((unsigned)std::min<int64_t>((n + 255) / 256, 64), (unsigned)m), 256, 0, stream>>>(
        d_src_raw.p, (int)n, 1.0f / prm.resolution, d_yaw_list.p, yaw_bins, y_keys_in.p, y_vals_in.p);
    int end_bit = 32;
    while ((1 << (end_bit - 32)) < m) ++end_bit;
    size_t tmp = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp, y_keys_in.p, y_keys_out.p, y_vals_in.p, y_vals_out.p, (int)ny, 0, end_bit, stream));
    CUDA_TRY(s_tmp.reserve(tmp));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(s_tmp.p, tmp, y_keys_in.p, y_keys_out.p, y_vals_in.p, y_vals_out.p, (int)ny, 0, end_bit, stream));
    k_ndt_gather<<<(unsigned)((ny + 255) / 256), 256, 0, stream>>>(d_src_raw.p, y_vals_out.p, (int)ny, d_src_yaw.p + (size_t)yaw_built * n);
    LAUNCH_COUNT(2);
    for (int j = 0; j < m; ++j) yaw_slot[list[j]] = yaw_built + j;
    yaw_built += m;
    for (int b = 0; b < yaw_bins; ++b) slot[b] = yaw_slot[b];
    CUDA_TRY(cudaMemcpyAsync(d_yaw_slot.p, slot, yaw_bins * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
    if (yaw_built == yaw_bins) {  // complete: the sort buffers are not needed again for this source
        CUDA_TRY(cudaStreamSynchronize(stream));
        y_keys_in.release(); y_keys_out.release(); y_vals_in.release(); y_vals_out.release();
    }
    return B200_OK;
}

int32_t Ndt::score_batch_device(const float* d_poses16, int64_t h, double* d_out) {
    if (!have_target) B200_FAIL(B200_ERR_ARG, "no target set");
    if (n_src < 1) B200_FAIL(B200_ERR_ARG, "no source set");
    if (h > 65535) B200_FAIL(B200_ERR_ARG, "at most 65535 hypotheses per call");
    const int32_t rc = yaw_orderings(d_poses16, h);
    if (rc) return rc;
    gauss();
    const int nch = (n_src + SCORE_CHUNK - 1) / SCORE_CHUNK;
    CUDA_TRY(d_partials.reserve((size_t)h * nch));
    const dim3 grid(nch, (unsigned)h);
    const View v = view();
    CUDA_TRY(cudaEventRecord(evs0, stream));
    if (prm.search == 1) k_ndt_score_batch<1><<<grid, SCORE_THREADS, 0, stream>>>(v, d_poses16, d_src_yaw.p, d_yaw_slot.p, yaw_bins, d_partials.p);
    else if (nst() == 27) k_ndt_score_batch<27><<<grid, SCORE_THREADS, 0, stream>>>(v, d_poses16, d_src_yaw.p, d_yaw_slot.p, yaw_bins, d_partials.p);
    else k_ndt_score_batch<7><<<grid, SCORE_THREADS, 0, stream>>>(v, d_poses16, d_src_yaw.p, d_yaw_slot.p, yaw_bins, d_partials.p);
    CUDA_TRY(cudaEventRecord(evs1, stream));
    k_ndt_score_finish<<<(unsigned)((h + 127) / 128), 128, 0, stream>>>(d_partials.p, nch, h, n_src, d_out);
    LAUNCH_COUNT(2);
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

int32_t Ndt::fitness(const float* T16, double max_range, double* score, int64_t* nr) {
    if (!have_target) B200_FAIL(B200_ERR_ARG, "no target set");
    if (n_src < 1) B200_FAIL(B200_ERR_ARG, "no source set");
    if (!have_fitness_index) {  // built on first use: target points in cell order + cell -> run table
        CUDA_TRY(d_tgt_sorted.reserve((size_t)n_tgt));
        CUDA_TRY(d_cell2run.reserve((size_t)ncells));
        CUDA_TRY(cudaMemsetAsync(d_cell2run.p, 0xFF, (size_t)ncells * sizeof(int32_t), stream));
        k_ndt_gather<<<(unsigned)((n_tgt + 255) / 256), 256, 0, stream>>>(d_tgt.p, d_vals_out.p, (int)n_tgt, d_tgt_sorted.p);
        k_ndt_cell_runs<<<(nruns + 255) / 256, 256, 0, stream>>>(d_uniq.p, d_small.p + 8, (uint32_t)ncells, d_cell2run.p);
        LAUNCH_COUNT(2);
        have_fitness_index = true;
    }
    CUDA_TRY(d_fit.reserve((size_t)n_src + 2));
    CUDA_TRY(d_poses.reserve(16)); CUDA_TRY(h_poses.reserve(16)); CUDA_TRY(h_scores.reserve(8));
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 4; ++j) h_poses.p[i * 4 + j] = T16[j * 4 + i];
    CUDA_TRY(cudaMemcpyAsync(d_poses.p, h_poses.p, 12 * sizeof(float), cudaMemcpyHostToDevice, stream));
    FitView f;
    f.pts = d_tgt_sorted.p; f.cell2run = d_cell2run.p; f.run_off = d_run_off.p; f.run_cnt = d_run_cnt.p;
    for (int k = 0; k < 3; ++k) { f.min_b[k] = gd.min_b[k]; f.div_b[k] = gd.div_b[k]; }
    f.leaf = prm.resolution; f.inv_leaf = gd.inv_leaf;
    CUDA_TRY(cudaEventRecord(ev0, stream));
    // the fitness is defined on the source in its original order; any order gives the same set of distances
    k_ndt_fitness<<<(unsigned)(((size_t)n_src * 32 + 255) / 256), 256, 0, stream>>>(f, d_src.p, n_src, d_poses.p, d_fit.p);
    k_ndt_fitness_reduce<<<1, 256, 0, stream>>>(d_fit.p, n_src, max_range, d_fit.p + n_src);
    LAUNCH_COUNT(2);
    CUDA_TRY(cudaEventRecord(ev1, stream));
    CUDA_TRY(cudaMemcpyAsync(h_scores.p, d_fit.p + n_src, 2 * sizeof(double), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    cudaEventElapsedTime(&last_ms, ev0, ev1);
    const double S = h_scores.p[0], Cn = h_scores.p[1];
    if (nr) *nr = (int64_t)Cn;
    if (score) *score = Cn > 0 ? S / Cn : 1.7976931348623157e308;  // PCL returns DBL_MAX when nothing is in range
    return B200_OK;
}

}  // namespace ndt
}  // namespace b200

// ------------------------------------------------------------------ NCCL communicator (loaded at run time)
#include "comm.cuh"

// ------------------------------------------------------------------ C ABI (B3)
using namespace b200;
using b200::ndt::Ndt;
struct b200_ndt { Ndt k; };

static void fill_result(const ndt::Ctl& c, float* final16, b200_ndt_result* r, float ms) {
    if (final16)
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) final16[j * 4 + i] = c.final_T[i * 4 + j];
    if (r) {
        r->converged = c.converged;
        r->iters = c.nr_iterations;
        r->evals = c.evals;
        r->hess_evals = c.hess_evals;
        r->trans_probability = c.trans_probability;
        memcpy(r->hessian, c.H, sizeof(double) * 36);
        r->score = c.score;
        memcpy(r->p_final, c.p, sizeof(double) * 6);
        r->gpu_ms = ms;
    }
}

// ------------------------------------------------------------------ batched registration of independent (source, target) pairs
// The loop-closure call site (mapOptmization.cpp:683-693) registers a keyframe against a submap and gates on
// hasConverged() && getFitnessScore() <= threshold.  Here a whole batch of such pairs is built, aligned and scored in one
// pass per chunk: one upload, one min / max read-back, one sort of all targets, one sort of all sources, the Newton /
// line-search loop of every pair in the same launches, and the fitness of every pair at its final transformation on the
// device.  A pair's work split depends on its own sizes and the parameters only, so its result is bit-identical whatever
// else is in the batch, in which chunk it lands and on which rank it runs.
namespace {
constexpr int64_t kPairTgtBytes = 400;  // device bytes per target point (cloud, sorted copy, sort buffers, leaf records in the worst case)
constexpr int64_t kPairSrcBytes = 64;   // per source point (cloud, sorted copy, 64-bit keys, indices, distances)
constexpr int kPairMaxItemsPerThread = 8;  // (point, cell) items per thread of an evaluation: the block's pair list always holds them

int pairs_chunk_max() {  // B200_NDT_PAIRS_CHUNK = most pairs per chunk (development switch; results do not depend on it)
    static const int v = getenv("B200_NDT_PAIRS_CHUNK") ? atoi(getenv("B200_NDT_PAIRS_CHUNK")) : 0;
    return v > 0 ? std::min(v, 65535) : 65535;
}

void pack_ranges(const float* xyz, int64_t stride, const int64_t* off, const int64_t* ids, int64_t np, const int64_t* dst_off, float4* dst) {
    const int nt = dst_off[np] > (1 << 20) ? 8 : 1;
    auto work = [=](int t) {
        for (int64_t j = t; j < np; j += nt)
            pack_xyz_float4((const float*)((const char*)xyz + off[ids[j]] * stride), dst_off[j + 1] - dst_off[j], stride, dst + dst_off[j]);
    };
    if (nt == 1) { work(0); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(work, t);
    for (auto& t : th) t.join();
}
}  // namespace

struct b200_ndt_pairs {
    Ndt k;  // parameters, stream, events, staging and the target / source / alignment buffers, reused by every chunk
    DevBuf<uint64_t> d_skeys_in, d_skeys_out;
    DevBuf<int64_t> d_off, d_d2off;
    PinnedBuf<int64_t> h_off;
    DevBuf<int32_t> d_mm;
    PinnedBuf<int32_t> h_mm;
    DevBuf<ndt::PairGrid> d_pg;
    PinnedBuf<ndt::PairGrid> h_pg;
    DevBuf<ndt::PairEval> d_pe;
    PinnedBuf<ndt::PairEval> h_pe;
    DevBuf<ndt::PairFit> d_pf;
    PinnedBuf<ndt::PairFit> h_pf;
    DevBuf<double> d_fitsum;
    PinnedBuf<double> h_fitsum;
    DevBuf<uint8_t> d_xchg;
    PinnedBuf<uint8_t> h_xchg;
    // the last chunk this rank built (b200_ndt_pairs_leaves)
    std::vector<int64_t> last_ids;
    std::vector<uint32_t> last_base;
    std::vector<int64_t> last_ncells;
    std::vector<int> last_live;
    int last_nruns = 0;

    struct Call {
        const float *src_xyz, *tgt_xyz;
        const int64_t *src_off, *tgt_off;
        int64_t stride;
        const float* guesses16;
        double max_range;
        b200_ndt_pair_result* results;
    };
    int32_t chunk(const Call& c, const int64_t* ids, int64_t np, int64_t cell_limit, int64_t& used);
    int32_t local(const Call& c, int64_t P, int64_t first, int64_t step);
    void destroy() {
        cudaSetDevice(k.device);
        if (k.stream) cudaStreamSynchronize(k.stream);
        d_skeys_in.release(); d_skeys_out.release(); d_off.release(); d_d2off.release(); h_off.release(); d_mm.release(); h_mm.release();
        d_pg.release(); h_pg.release(); d_pe.release(); h_pe.release(); d_pf.release(); h_pf.release(); d_fitsum.release(); h_fitsum.release();
        d_xchg.release(); h_xchg.release();
        k.destroy();
    }
};

// Builds, aligns and scores pairs ids[0 .. np-1] (all with a non-empty source and target); `used` = how many of them fit the
// 32-bit key space / memory bound and were done (at least one).
int32_t b200_ndt_pairs::chunk(const Call& c, const int64_t* ids, int64_t np, int64_t cell_limit, int64_t& used) {
    using namespace ndt;
    Ndt& K = k;
    cudaStream_t s = K.stream;
    std::vector<int64_t> toff(np + 1, 0), soff(np + 1, 0);
    int64_t max_tn = 1, max_sn = 1;
    for (int64_t j = 0; j < np; ++j) {
        const int64_t tn = c.tgt_off[ids[j] + 1] - c.tgt_off[ids[j]], sn = c.src_off[ids[j] + 1] - c.src_off[ids[j]];
        toff[j + 1] = toff[j] + tn;
        soff[j + 1] = soff[j] + sn;
        max_tn = std::max(max_tn, tn);
        max_sn = std::max(max_sn, sn);
    }
    const int64_t nt = toff[np], ns = soff[np];
    // one upload of every cloud of the chunk
    CUDA_TRY(K.h_stage.reserve((size_t)(nt + ns)));
    pack_ranges(c.tgt_xyz, c.stride, c.tgt_off, ids, np, toff.data(), K.h_stage.p);
    pack_ranges(c.src_xyz, c.stride, c.src_off, ids, np, soff.data(), K.h_stage.p + nt);
    CUDA_TRY(K.d_tgt.reserve((size_t)nt));
    CUDA_TRY(K.d_src_raw.reserve((size_t)ns));
    CUDA_TRY(cudaMemcpyAsync(K.d_tgt.p, K.h_stage.p, (size_t)nt * sizeof(float4), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(K.d_src_raw.p, K.h_stage.p + nt, (size_t)ns * sizeof(float4), cudaMemcpyHostToDevice, s));
    CUDA_TRY(h_off.reserve(2 * (size_t)(np + 1)));
    CUDA_TRY(d_off.reserve(2 * (size_t)(np + 1)));
    memcpy(h_off.p, toff.data(), (np + 1) * sizeof(int64_t));
    memcpy(h_off.p + np + 1, soff.data(), (np + 1) * sizeof(int64_t));
    CUDA_TRY(cudaMemcpyAsync(d_off.p, h_off.p, 2 * (np + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    const int64_t* d_toff = d_off.p;
    const int64_t* d_soff = d_off.p + np + 1;
    // per-target min / max, read back once for the whole chunk
    CUDA_TRY(d_mm.reserve(6 * (size_t)np));
    CUDA_TRY(h_mm.reserve(6 * (size_t)np));
    k_ndt_minmax_init_pairs<<<(unsigned)((6 * np + 255) / 256), 256, 0, s>>>(d_mm.p, (int)np);
    k_ndt_minmax_pairs<<<dim3((unsigned)std::min<int64_t>((max_tn + 1023) / 1024, 256), (unsigned)np), 256, 0, s>>>(K.d_tgt.p, d_toff, d_mm.p);
    CUDA_TRY(cudaMemcpyAsync(h_mm.p, d_mm.p, 6 * np * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    LAUNCH_COUNT(2);
    // every target's grid, as Ndt::build_target derives it; the dense tables end to end
    CUDA_TRY(h_pg.reserve((size_t)np));
    CUDA_TRY(d_pg.reserve((size_t)np));
    int64_t cells = 0, n_live = 0;
    used = np;
    for (int64_t j = 0; j < np; ++j) {
        PairGrid& g = h_pg.p[j];
        memset(&g, 0, sizeof g);
        int64_t nc = 0;
        const int32_t st = grid_from_minmax(h_mm.p + 6 * j, K.prm.resolution, g.gd, nc);
        if (st) {
            memset(&g, 0, sizeof g);
            c.results[ids[j]].status = st;
            continue;
        }
        if (cells + nc > cell_limit && j > 0) { used = j; break; }
        g.cell_base = (uint32_t)cells;
        g.live = 1;
        cells += nc;
        ++n_live;
    }
    np = used;
    last_ids.assign(ids, ids + np);
    last_base.resize(np);
    last_ncells.resize(np);
    last_live.resize(np);
    for (int64_t j = 0; j < np; ++j) {
        const PairGrid& g = h_pg.p[j];
        last_base[j] = g.cell_base;
        last_ncells[j] = g.live ? (int64_t)g.gd.div_b[0] * g.gd.div_b[1] * g.gd.div_b[2] : 0;
        last_live[j] = g.live;
    }
    last_nruns = 0;
    if (!n_live) return B200_OK;
    const int64_t nt_u = toff[np], ns_u = soff[np];
    CUDA_TRY(cudaMemcpyAsync(d_pg.p, h_pg.p, np * sizeof(PairGrid), cudaMemcpyHostToDevice, s));
    // segmented target build: one stable sort of (cell_base + leaf id) over every target, then the single-target kernels
    const uint32_t sentinel = (uint32_t)cells;
    CUDA_TRY(K.d_keys_in.reserve(nt_u)); CUDA_TRY(K.d_keys_out.reserve(nt_u)); CUDA_TRY(K.d_uniq.reserve(nt_u));
    CUDA_TRY(K.d_vals_in.reserve(nt_u)); CUDA_TRY(K.d_vals_out.reserve(nt_u)); CUDA_TRY(K.d_run_cnt.reserve(nt_u)); CUDA_TRY(K.d_run_off.reserve(nt_u));
    k_ndt_keys_pairs<<<dim3((unsigned)std::min<int64_t>((max_tn + 255) / 256, 1024), (unsigned)np), 256, 0, s>>>(K.d_tgt.p, d_toff, d_pg.p, sentinel,
                                                                                                           K.d_keys_in.p, K.d_vals_in.p);
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) <= cells) ++end_bit;
    int32_t* d_nruns = K.d_small.p + 8;
    size_t t1 = 0, t2 = 0, t3 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, K.d_keys_in.p, K.d_keys_out.p, K.d_vals_in.p, K.d_vals_out.p, (int)nt_u, 0, end_bit, s);
    cub::DeviceRunLengthEncode::Encode(nullptr, t2, K.d_keys_out.p, K.d_uniq.p, K.d_run_cnt.p, d_nruns, (int)nt_u, s);
    cub::DeviceScan::ExclusiveSum(nullptr, t3, K.d_run_cnt.p, K.d_run_off.p, (int)nt_u, s);
    size_t tmp = std::max(t1, std::max(t2, t3));
    CUDA_TRY(K.cub_tmp.reserve(tmp));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(K.cub_tmp.p, tmp, K.d_keys_in.p, K.d_keys_out.p, K.d_vals_in.p, K.d_vals_out.p, (int)nt_u, 0, end_bit, s));
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(K.cub_tmp.p, tmp, K.d_keys_out.p, K.d_uniq.p, K.d_run_cnt.p, d_nruns, (int)nt_u, s));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(K.cub_tmp.p, tmp, K.d_run_cnt.p, K.d_run_off.p, (int)nt_u, s));
    CUDA_TRY(cudaMemcpyAsync(K.h_small.p, d_nruns, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    const int nruns = K.h_small.p[0];
    CUDA_TRY(K.d_sums.reserve((size_t)nruns * 9));
    CUDA_TRY(K.d_centroid.reserve((size_t)nruns * 3 + 4));
    CUDA_TRY(K.d_leafF.reserve(nruns)); CUDA_TRY(K.d_leafD.reserve(nruns)); CUDA_TRY(K.d_cov.reserve((size_t)nruns * 9));
    CUDA_TRY(K.d_npts.reserve(nruns)); CUDA_TRY(K.d_valid.reserve(nruns));
    CUDA_TRY(K.d_cell2leaf.reserve((size_t)cells));
    CUDA_TRY(K.d_cell2run.reserve((size_t)cells));
    CUDA_TRY(cudaMemsetAsync(K.d_cell2leaf.p, 0xFF, (size_t)cells * sizeof(int32_t), s));
    CUDA_TRY(cudaMemsetAsync(K.d_cell2run.p, 0xFF, (size_t)cells * sizeof(int32_t), s));
    int32_t* d_nvalid = K.d_small.p + 9;
    CUDA_TRY(cudaMemsetAsync(d_nvalid, 0, sizeof(int32_t), s));
    CUDA_TRY(cudaMemsetAsync(K.d_cov.p, 0, (size_t)nruns * 9 * sizeof(double), s));
    const int acc_blocks = std::min((nruns + 7) / 8, K.sm_count * 8);
    k_ndt_accumulate<<<std::max(acc_blocks, 1), 256, 0, s>>>(K.d_tgt.p, K.d_vals_out.p, K.d_uniq.p, K.d_run_off.p, K.d_run_cnt.p, d_nruns, sentinel,
                                                             K.d_sums.p, K.d_centroid.p);
    k_ndt_finalize<<<(nruns + 127) / 128, 128, 0, s>>>(K.d_uniq.p, K.d_run_cnt.p, d_nruns, sentinel, K.d_sums.p, K.prm.min_pts, K.prm.eig_ratio,
                                                       K.d_leafF.p, K.d_leafD.p, K.d_cov.p, K.d_npts.p, K.d_valid.p, K.d_cell2leaf.p, d_nvalid);
    // fitness index: target points in cell order, cell -> run
    CUDA_TRY(K.d_tgt_sorted.reserve((size_t)nt_u));
    k_ndt_gather<<<(unsigned)((nt_u + 255) / 256), 256, 0, s>>>(K.d_tgt.p, K.d_vals_out.p, (int)nt_u, K.d_tgt_sorted.p);
    k_ndt_cell_runs<<<(nruns + 255) / 256, 256, 0, s>>>(K.d_uniq.p, d_nruns, sentinel, K.d_cell2run.p);
    last_nruns = nruns;
    // sources: one stable sort by (pair, Morton key), so every pair is ordered as set_source orders it alone
    CUDA_TRY(d_skeys_in.reserve(ns_u)); CUDA_TRY(d_skeys_out.reserve(ns_u));
    CUDA_TRY(K.s_vals_in.reserve(ns_u)); CUDA_TRY(K.s_vals_out.reserve(ns_u)); CUDA_TRY(K.d_src.reserve((size_t)ns_u));
    k_ndt_source_keys_pairs<<<dim3((unsigned)std::min<int64_t>((max_sn + 255) / 256, 1024), (unsigned)np), 256, 0, s>>>(
        K.d_src_raw.p, d_soff, 1.0f / K.prm.resolution, d_skeys_in.p, K.s_vals_in.p);
    int s_end = 33;
    while (s_end < 64 && ((int64_t)1 << (s_end - 32)) < np) ++s_end;
    tmp = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp, d_skeys_in.p, d_skeys_out.p, K.s_vals_in.p, K.s_vals_out.p, (int)ns_u, 0, s_end, s));
    CUDA_TRY(K.s_tmp.reserve(tmp));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(K.s_tmp.p, tmp, d_skeys_in.p, d_skeys_out.p, K.s_vals_in.p, K.s_vals_out.p, (int)ns_u, 0, s_end, s));
    k_ndt_gather<<<(unsigned)((ns_u + 255) / 256), 256, 0, s>>>(K.d_src_raw.p, K.s_vals_out.p, (int)ns_u, K.d_src.p);
    LAUNCH_COUNT(7);
    // alignment: one control block and one view per built pair
    K.gauss();  // recomputed at every computeTransformation (ndt_omp_impl.hpp:77-81)
    View base = K.view();
    base.nbr7 = nullptr;
    CUDA_TRY(h_pe.reserve((size_t)n_live)); CUDA_TRY(d_pe.reserve((size_t)n_live));
    CUDA_TRY(h_pf.reserve((size_t)n_live)); CUDA_TRY(d_pf.reserve((size_t)n_live));
    CUDA_TRY(K.h_poses.reserve((size_t)n_live * 16)); CUDA_TRY(K.d_poses.reserve((size_t)n_live * 16));
    std::vector<int64_t> live(n_live), d2off(n_live + 1, 0);
    int max_nbx = 1;
    int64_t max_live_sn = 1;
    for (int64_t j = 0, a = 0; j < np; ++j) {
        const PairGrid& g = h_pg.p[j];
        if (!g.live) continue;
        live[a] = j;
        const int64_t sn = soff[j + 1] - soff[j];
        PairEval& e = h_pe.p[a];
        e.v = base;
        e.v.src = K.d_src.p + soff[j];
        e.v.n_src = (int)sn;
        e.v.cell2leaf = K.d_cell2leaf.p + g.cell_base;
        for (int q = 0; q < 3; ++q) { e.v.min_b[q] = g.gd.min_b[q]; e.v.max_b[q] = g.gd.max_b[q]; e.v.mul[q] = g.gd.mul[q]; }
        const int64_t items = sn * K.nst();
        e.nbx = (int)std::max<int64_t>(1, (items + EVAL_THREADS * kPairMaxItemsPerThread - 1) / (EVAL_THREADS * kPairMaxItemsPerThread));
        max_nbx = std::max(max_nbx, e.nbx);
        PairFit& f = h_pf.p[a];
        f.f.pts = K.d_tgt_sorted.p; f.f.cell2run = K.d_cell2run.p + g.cell_base; f.f.run_off = K.d_run_off.p; f.f.run_cnt = K.d_run_cnt.p;
        for (int q = 0; q < 3; ++q) { f.f.min_b[q] = g.gd.min_b[q]; f.f.div_b[q] = g.gd.div_b[q]; }
        f.f.leaf = K.prm.resolution; f.f.inv_leaf = g.gd.inv_leaf;
        f.src = e.v.src;
        f.n = (int)sn;
        d2off[a + 1] = d2off[a] + sn;
        max_live_sn = std::max(max_live_sn, sn);
        float* G = K.h_poses.p + a * 16;
        if (c.guesses16) memcpy(G, c.guesses16 + ids[j] * 16, 16 * sizeof(float));
        else for (int q = 0; q < 16; ++q) G[q] = (q % 5 == 0) ? 1.f : 0.f;
        ++a;
    }
    CUDA_TRY(cudaMemcpyAsync(d_pe.p, h_pe.p, n_live * sizeof(PairEval), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_pf.p, h_pf.p, n_live * sizeof(PairFit), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(K.d_poses.p, K.h_poses.p, n_live * 16 * sizeof(float), cudaMemcpyHostToDevice, s));
    CUDA_TRY(K.d_ctl.reserve(n_live)); CUDA_TRY(K.h_ctl.reserve(n_live));
    const int part_stride = NACC * max_nbx;
    CUDA_TRY(K.d_partials.reserve((size_t)n_live * part_stride));
    AlignConsts kc{K.prm.step_size, K.prm.trans_eps, K.prm.max_iter, 0};
    k_ndt_init<<<(unsigned)((n_live + 63) / 64), 64, 0, s>>>(K.d_ctl.p, (int)n_live, K.d_poses.p, nullptr, PH_INIT);
    int launches = 1;
    const int max_launches = (K.prm.max_iter + 3) * 12 + 1;
    int32_t rc = K.until_done((int)n_live, max_launches, launches, [&]() {
        k_ndt_eval<false, true><<<dim3(max_nbx, (unsigned)n_live), EVAL_THREADS, 0, s>>>(View{}, K.d_ctl.p, kc, K.d_partials.p, nullptr, 1, d_pe.p,
                                                                                            part_stride);
    });
    LAUNCH_COUNT(launches);
    if (rc) return rc;
    // getFitnessScore(max_range) of every pair at its final transformation, read from its control block on the device
    CUDA_TRY(d_d2off.reserve((size_t)n_live + 1));
    CUDA_TRY(h_off.reserve((size_t)n_live + 1));
    memcpy(h_off.p, d2off.data(), (n_live + 1) * sizeof(int64_t));  // h_off's chunk offsets reached the device before the last poll
    CUDA_TRY(cudaMemcpyAsync(d_d2off.p, h_off.p, (n_live + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    CUDA_TRY(K.d_fit.reserve((size_t)d2off[n_live]));
    CUDA_TRY(d_fitsum.reserve(2 * (size_t)n_live)); CUDA_TRY(h_fitsum.reserve(2 * (size_t)n_live));
    k_ndt_fitness_pairs<<<dim3((unsigned)((max_live_sn * 32 + 255) / 256), (unsigned)n_live), 256, 0, s>>>(d_pf.p, K.d_ctl.p, d_d2off.p, K.d_fit.p);
    k_ndt_fitness_reduce_pairs<<<(unsigned)n_live, 256, 0, s>>>(K.d_fit.p, d_d2off.p, c.max_range, d_fitsum.p);
    LAUNCH_COUNT(3);
    CUDA_TRY(cudaMemcpyAsync(K.h_ctl.p, K.d_ctl.p, n_live * sizeof(Ctl), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h_fitsum.p, d_fitsum.p, 2 * n_live * sizeof(double), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    for (int64_t a = 0; a < n_live; ++a) {
        const Ctl& ct = K.h_ctl.p[a];
        b200_ndt_pair_result& r = c.results[ids[live[a]]];
        fill_result(ct, r.final16, &r.ndt, 0.f);
        r.status = !ct.done ? B200_ERR_CUDA : ct.converged ? B200_OK : B200_NOT_CONVERGED;
        const double S = h_fitsum.p[2 * a], Cn = h_fitsum.p[2 * a + 1];
        r.n_in_range = (int64_t)Cn;
        r.fitness = Cn > 0 ? S / Cn : 1.7976931348623157e308;  // PCL returns DBL_MAX when nothing is in range
    }
    return B200_OK;
}

// This rank's pairs first, first + step, ... < P: statuses of the pairs that fail on their own, then chunks of the rest.
int32_t b200_ndt_pairs::local(const Call& c, int64_t P, int64_t first, int64_t step) {
    std::vector<int64_t> cand;
    for (int64_t p = first; p < P; p += step) {
        b200_ndt_pair_result& r = c.results[p];
        memset(&r, 0, sizeof r);
        const int64_t tn = c.tgt_off[p + 1] - c.tgt_off[p], sn = c.src_off[p + 1] - c.src_off[p];
        // the codes b200_ndt_set_target / b200_ndt_set_source return for these clouds
        if (tn < 1 || tn > (int64_t)0x7fffff00) r.status = B200_ERR_ARG;
        else if (sn < 1 || sn > (1 << 28)) r.status = B200_ERR_ARG;
        else cand.push_back(p);
    }
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    const int64_t budget = (int64_t)(0.6 * (double)free_b);
    const int64_t cell_limit = std::min<int64_t>(((int64_t)1 << 32) - 2, std::max<int64_t>(budget / 4 / 8, (int64_t)1 << 30));
    const int64_t max_np = pairs_chunk_max();
    for (size_t i = 0; i < cand.size();) {
        size_t e = i;
        int64_t bytes = 0, nt = 0, ns = 0;
        while (e < cand.size() && (int64_t)(e - i) < max_np) {
            const int64_t p = cand[e];
            const int64_t tn = c.tgt_off[p + 1] - c.tgt_off[p], sn = c.src_off[p + 1] - c.src_off[p];
            const int64_t add = tn * kPairTgtBytes + sn * kPairSrcBytes;
            if (e > i && (bytes + add > budget * 3 / 4 || nt + tn > (int64_t)0x7fffff00 || ns + sn > (int64_t)0x7fffff00)) break;
            bytes += add; nt += tn; ns += sn;
            ++e;
        }
        int64_t used = 0;
        const int32_t rc = chunk(c, cand.data() + i, (int64_t)(e - i), cell_limit, used);
        if (rc) return rc;
        i += (size_t)std::max<int64_t>(used, 1);
    }
    return B200_OK;
}

extern "C" {

int32_t b200_ndt_create(const b200_ndt_params* params, int32_t device, b200_ndt** out) {
    if (!params || !out) B200_FAIL(B200_ERR_ARG, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) B200_FAIL(B200_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) B200_FAIL(B200_ERR_ARG, "bad device ordinal");
    b200_ndt* h = new b200_ndt();
    int32_t rc = h->k.init(params, device);
    if (rc != B200_OK) { h->k.destroy(); delete h; return rc; }
    *out = h;
    return B200_OK;
}
int32_t b200_ndt_destroy(b200_ndt* n) {
    if (!n) return B200_OK;
    n->k.destroy();
    delete n;
    return B200_OK;
}
int32_t b200_ndt_set_target(b200_ndt* n, const float* xyz, int64_t cnt, int64_t stride) {
    if (!n) B200_FAIL(B200_ERR_ARG, "null handle");
    return n->k.set_target(xyz, cnt, stride);
}
/* setInputTarget for a map replicated over the ranks of `comm`: only `root` passes the cloud (xyz may be NULL elsewhere,
 * cnt must be the same everywhere); the packed points travel once over NVLink (ncclBroadcast, 16 B/point) and every
 * rank builds its own voxel Gaussians from them - identical on all ranks because the build is deterministic. */
int32_t b200_ndt_set_target_bcast(b200_comm* comm, b200_ndt* n, const float* xyz, int64_t cnt, int64_t stride, int32_t root) {
    if (!n || !comm || cnt < 1 || cnt > (int64_t)0x7fffff00) B200_FAIL(B200_ERR_ARG, "bad argument");
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    if (comm->rank == root) {
        if (!xyz || stride < 12) B200_FAIL(B200_ERR_ARG, "root needs the cloud");
        int32_t rc = k.upload(xyz, cnt, stride, k.d_tgt);
        if (rc) return rc;
    } else {
        CUDA_TRY(k.d_tgt.reserve((size_t)cnt));
    }
    NCCL_TRY(comm, comm->Broadcast(k.d_tgt.p, k.d_tgt.p, (size_t)cnt * sizeof(float4), ncclChar, root, comm->comm, k.stream));
    return k.build_target(cnt);
}

int32_t b200_ndt_set_source(b200_ndt* n, const float* xyz, int64_t cnt, int64_t stride) {
    if (!n) B200_FAIL(B200_ERR_ARG, "null handle");
    return n->k.set_source(xyz, cnt, stride);
}
int64_t b200_ndt_num_voxels(b200_ndt* n) { return n ? (int64_t)n->k.n_valid : 0; }
float b200_ndt_last_ms(b200_ndt* n) { return n ? n->k.last_ms : 0.f; }
int32_t b200_ndt_last_launches(b200_ndt* n) { return n ? n->k.last_launches : 0; }
/* parity probe (a-12): the Newton direction the device computes for Hessian H and right-hand side rhs, i.e. what
 * JacobiSVD(H).solve(rhs) answers (ndt_omp_impl.hpp:112-114).  *path = 0 pivoted-elimination shortcut (H comfortably full
 * rank), 1 literal two-sided Jacobi SVD; force_svd = 1 always takes the latter. */
int32_t b200_ndt_newton_direction(b200_ndt* n, const double* H36, const double* rhs6, int32_t force_svd, double* x6, int32_t* path) {
    if (!n || !H36 || !rhs6 || !x6) B200_FAIL(B200_ERR_ARG, "bad argument");
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    CUDA_TRY(k.d_p_in.reserve(64));
    double h[49] = {0};
    memcpy(h, H36, 36 * sizeof(double));
    memcpy(h + 36, rhs6, 6 * sizeof(double));
    CUDA_TRY(cudaMemcpyAsync(k.d_p_in.p, h, sizeof h, cudaMemcpyHostToDevice, k.stream));
    ndt::k_ndt_solve_probe<<<1, 32, 0, k.stream>>>(k.d_p_in.p, force_svd);
    LAUNCH_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(h, k.d_p_in.p, sizeof h, cudaMemcpyDeviceToHost, k.stream));
    CUDA_TRY(cudaStreamSynchronize(k.stream));
    CUDA_TRY(cudaGetLastError());
    memcpy(x6, h + 42, 6 * sizeof(double));
    if (path) *path = (int32_t)h[48];
    return B200_OK;
}

/* profiling aid: SM cycles the state machine (advance) and its Newton solves took over the last align */
int32_t b200_ndt_debug_cycles(b200_ndt* n, int64_t* step_cycles, int64_t* solve_cycles) {
    if (!n || !n->k.h_ctl.p) return -1;
    if (step_cycles) *step_cycles = (int64_t)n->k.h_ctl.p[0].step_cycles;
    if (solve_cycles) *solve_cycles = (int64_t)n->k.h_ctl.p[0].solve_cycles;
    return 0;
}

int64_t b200_ndt_leaves(b200_ndt* n, int64_t max, int64_t* ids, int32_t* npts, double* mean3, double* cov9, double* icov9) {
    if (!n || !n->k.have_target) return 0;
    Ndt& k = n->k;
    cudaSetDevice(k.device);
    const int nr = k.nruns;
    std::vector<uint8_t> valid(nr);
    std::vector<uint32_t> uniq(nr);
    std::vector<int32_t> np(nr);
    std::vector<ndt::LeafD> L(nr);
    std::vector<double> cov((size_t)nr * 9);
    cudaStreamSynchronize(k.stream);
    cudaMemcpy(valid.data(), k.d_valid.p, nr, cudaMemcpyDeviceToHost);
    cudaMemcpy(uniq.data(), k.d_uniq.p, nr * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaMemcpy(np.data(), k.d_npts.p, nr * sizeof(int32_t), cudaMemcpyDeviceToHost);
    cudaMemcpy(L.data(), k.d_leafD.p, nr * sizeof(ndt::LeafD), cudaMemcpyDeviceToHost);
    cudaMemcpy(cov.data(), k.d_cov.p, (size_t)nr * 9 * sizeof(double), cudaMemcpyDeviceToHost);
    int64_t cnt = 0;
    for (int r = 0; r < nr; ++r) {  // runs are sorted by leaf id
        if (!valid[r]) continue;
        if (cnt < max) {
            if (ids) ids[cnt] = (int64_t)uniq[r];
            if (npts) npts[cnt] = np[r];
            if (mean3) memcpy(mean3 + cnt * 3, L[r].mean, 24);
            if (cov9) memcpy(cov9 + cnt * 9, &cov[(size_t)r * 9], 72);
            if (icov9) memcpy(icov9 + cnt * 9, L[r].icov, 72);
        }
        ++cnt;
    }
    return cnt;
}

int32_t b200_ndt_grid(b200_ndt* n, int32_t* min_b3, int32_t* div_b3) {
    if (!n || !n->k.have_target) B200_FAIL(B200_ERR_ARG, "no target set");
    for (int k = 0; k < 3; ++k) {
        if (min_b3) min_b3[k] = n->k.gd.min_b[k];
        if (div_b3) div_b3[k] = n->k.gd.div_b[k];
    }
    return B200_OK;
}

int32_t b200_ndt_align(b200_ndt* n, const float* guess16, float* final16, b200_ndt_result* result) {
    if (!n || !guess16 || !final16) B200_FAIL(B200_ERR_ARG, "null argument");
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    CUDA_TRY(k.d_poses.reserve(16));
    CUDA_TRY(k.h_poses.reserve(16));
    memcpy(k.h_poses.p, guess16, 16 * sizeof(float));
    CUDA_TRY(cudaMemcpyAsync(k.d_poses.p, k.h_poses.p, 16 * sizeof(float), cudaMemcpyHostToDevice, k.stream));
    int32_t rc = k.run(1, k.d_poses.p, nullptr, ndt::PH_INIT);
    if (rc) return rc;
    const ndt::Ctl& c = k.h_ctl.p[0];
    fill_result(c, final16, result, k.last_ms);
    if (!c.done) { B200_FAIL(B200_NOT_CONVERGED, "evaluation budget exhausted"); }
    return c.converged ? B200_OK : B200_NOT_CONVERGED;
}

/* getMaxEigen() (ndt_omp.h:209-223): the largest eigenvalue of hessian_eigen_ (the Hessian the last align() ended with)
 * divided by 100000 - the quantity the localization node's "lost" heuristic watches (localization.cpp:424-470).  The
 * reference runs Eigen::EigenSolver (real Schur form) on the 6 x 6 matrix; the accumulated Hessian is symmetric up to rounding, so
 * its eigenvalues are real and a symmetric Jacobi sweep over (H + H^T) / 2 returns the same values to fp64 rounding.  A
 * 6 x 6 scalar diagnostic evaluated on the host from the result block - nothing of the hot path runs here. */
int32_t b200_ndt_max_eigen(const double* hessian36, double* max_eigen) {
    if (!hessian36 || !max_eigen) B200_FAIL(B200_ERR_ARG, "null argument");
    double A[36];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) A[i * 6 + j] = 0.5 * (hessian36[i * 6 + j] + hessian36[j * 6 + i]);
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < 6; ++i) {
            diag += A[i * 6 + i] * A[i * 6 + i];
            for (int j = i + 1; j < 6; ++j) off += A[i * 6 + j] * A[i * 6 + j];
        }
        if (off <= 1e-300 || off <= 1e-34 * diag) break;
        for (int p = 0; p < 5; ++p)
            for (int q = p + 1; q < 6; ++q) {
                const double apq = A[p * 6 + q];
                if (apq == 0.0) continue;
                const double theta = (A[q * 6 + q] - A[p * 6 + p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
                for (int k = 0; k < 6; ++k) {
                    const double akp = A[k * 6 + p], akq = A[k * 6 + q];
                    A[k * 6 + p] = c * akp - sn * akq;
                    A[k * 6 + q] = sn * akp + c * akq;
                }
                for (int k = 0; k < 6; ++k) {
                    const double apk = A[p * 6 + k], aqk = A[q * 6 + k];
                    A[p * 6 + k] = c * apk - sn * aqk;
                    A[q * 6 + k] = sn * apk + c * aqk;
                }
            }
    }
    double mx = A[0];
    for (int i = 1; i < 6; ++i) mx = std::max(mx, A[i * 6 + i]);
    *max_eigen = mx / 100000.0;
    return B200_OK;
}

/* align() for h independent initial guesses in one batch (global relocalization with refinement): results[h], finals h x 16 */
int32_t b200_ndt_align_batch(b200_ndt* n, const float* guesses16, int64_t h, float* finals16, b200_ndt_result* results) {
    if (!n || !guesses16 || h < 1 || h > 65535) B200_FAIL(B200_ERR_ARG, "bad argument");
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    CUDA_TRY(k.d_poses.reserve((size_t)h * 16));
    CUDA_TRY(k.h_poses.reserve((size_t)h * 16));
    memcpy(k.h_poses.p, guesses16, (size_t)h * 16 * sizeof(float));
    CUDA_TRY(cudaMemcpyAsync(k.d_poses.p, k.h_poses.p, (size_t)h * 16 * sizeof(float), cudaMemcpyHostToDevice, k.stream));
    int32_t rc = k.run((int)h, k.d_poses.p, nullptr, ndt::PH_INIT);
    if (rc) return rc;
    for (int64_t a = 0; a < h; ++a) fill_result(k.h_ctl.p[a], finals16 ? finals16 + a * 16 : nullptr, results ? results + a : nullptr, k.last_ms);
    return B200_OK;
}

static int32_t single_eval(Ndt& k, const double* p6, int phase) {
    CUDA_SET_DEVICE(k.device);
    CUDA_TRY(k.d_p_in.reserve(6));
    CUDA_TRY(k.h_scores.reserve(8));
    memcpy(k.h_scores.p, p6, 6 * sizeof(double));
    CUDA_TRY(cudaMemcpyAsync(k.d_p_in.p, k.h_scores.p, 6 * sizeof(double), cudaMemcpyHostToDevice, k.stream));
    return k.run(1, nullptr, k.d_p_in.p, phase);
}

int32_t b200_ndt_derivatives(b200_ndt* n, const double* p6, double* score, double* g6, double* H36) {
    if (!n || !p6) B200_FAIL(B200_ERR_ARG, "null argument");
    int32_t rc = single_eval(n->k, p6, ndt::PH_SINGLE_DERIV);
    if (rc) return rc;
    const ndt::Ctl& c = n->k.h_ctl.p[0];
    if (score) *score = c.score;
    if (g6) memcpy(g6, c.g, 48);
    if (H36) memcpy(H36, c.H, 288);
    return B200_OK;
}

int32_t b200_ndt_hessian(b200_ndt* n, const double* p6, double* H36) {
    if (!n || !p6 || !H36) B200_FAIL(B200_ERR_ARG, "null argument");
    int32_t rc = single_eval(n->k, p6, ndt::PH_SINGLE_HESS);
    if (rc) return rc;
    memcpy(H36, n->k.h_ctl.p[0].H, 288);
    return B200_OK;
}

int32_t b200_ndt_score_batch(b200_ndt* n, const float* poses16, int64_t h, double* scores) {
    if (!n || !poses16 || !scores || h < 1) B200_FAIL(B200_ERR_ARG, "bad argument");
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    CUDA_TRY(k.d_poses.reserve((size_t)h * 16)); CUDA_TRY(k.h_poses.reserve((size_t)h * 16));
    CUDA_TRY(k.d_scores.reserve(h)); CUDA_TRY(k.h_scores.reserve(h));
    memcpy(k.h_poses.p, poses16, (size_t)h * 16 * sizeof(float));
    CUDA_TRY(cudaMemcpyAsync(k.d_poses.p, k.h_poses.p, (size_t)h * 16 * sizeof(float), cudaMemcpyHostToDevice, k.stream));
    CUDA_TRY(cudaEventRecord(k.ev0, k.stream));
    int32_t rc = k.score_batch_device(k.d_poses.p, h, k.d_scores.p);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(k.ev1, k.stream));
    CUDA_TRY(cudaMemcpyAsync(k.h_scores.p, k.d_scores.p, (size_t)h * sizeof(double), cudaMemcpyDeviceToHost, k.stream));
    CUDA_TRY(cudaStreamSynchronize(k.stream));
    cudaEventElapsedTime(&k.last_ms, k.ev0, k.ev1);
    memcpy(scores, k.h_scores.p, (size_t)h * sizeof(double));
    return B200_OK;
}

/* pcl::Registration::getFitnessScore(max_range): mean squared distance from the source, moved by T16 (column-major 4x4;
 * NULL = the final transformation of the last align), to its exact nearest neighbours in the target */
int32_t b200_ndt_fitness_score(b200_ndt* n, const float* T16, double max_range, double* score, int64_t* n_in_range) {
    if (!n || !score) B200_FAIL(B200_ERR_ARG, "null argument");
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    float T[16];
    if (T16) memcpy(T, T16, sizeof T);
    else {
        if (!k.h_ctl.p) B200_FAIL(B200_ERR_ARG, "no alignment has been run");
        const ndt::Ctl& c = k.h_ctl.p[0];
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) T[j * 4 + i] = c.final_T[i * 4 + j];
    }
    return k.fitness(T, max_range, score, n_in_range);
}

/* roofline bookkeeping: number of (point, voxel) pairs one evaluation at pose p6 touches */
int64_t b200_ndt_nbhd_total(b200_ndt* n, const double* p6) {
    if (!n || !p6 || !n->k.have_target || n->k.n_src < 1) return -1;
    Ndt& k = n->k;
    cudaSetDevice(k.device);
    // build the float matrix on the host the same way (only used for counting)
    float M[16];
    {
        const float rx = (float)p6[3], ry = (float)p6[4], rz = (float)p6[5];
        const float cx = (float)std::cos((double)rx), sx = (float)std::sin((double)rx), cy = (float)std::cos((double)ry),
                    sy = (float)std::sin((double)ry), cz = (float)std::cos((double)rz), sz = (float)std::sin((double)rz);
        const float Rx[9] = {1, 0, 0, 0, cx, -sx, 0, sx, cx}, Ry[9] = {cy, 0, sy, 0, 1, 0, -sy, 0, cy}, Rz[9] = {cz, -sz, 0, sz, cz, 0, 0, 0, 1};
        float T1[9], T2[9];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) T1[i * 3 + j] = (Rx[i * 3] * Ry[j] + Rx[i * 3 + 1] * Ry[3 + j]) + Rx[i * 3 + 2] * Ry[6 + j];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) T2[i * 3 + j] = (T1[i * 3] * Rz[j] + T1[i * 3 + 1] * Rz[3 + j]) + T1[i * 3 + 2] * Rz[6 + j];
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) M[i * 4 + j] = T2[i * 3 + j];
            M[i * 4 + 3] = (float)p6[i];
        }
        M[12] = M[13] = M[14] = 0.f; M[15] = 1.f;
    }
    if (k.d_poses.reserve(16) != cudaSuccess || k.h_poses.reserve(16) != cudaSuccess) return -1;
    memcpy(k.h_poses.p, M, sizeof M);
    cudaMemcpyAsync(k.d_poses.p, k.h_poses.p, sizeof M, cudaMemcpyHostToDevice, k.stream);
    cudaMemsetAsync(k.d_best.p, 0, sizeof(unsigned long long), k.stream);
    ndt::k_ndt_nbhd_total<<<k.sm_count, 256, 0, k.stream>>>(k.view(), k.d_poses.p, k.d_best.p);
    cudaMemcpyAsync(k.h_best.p, k.d_best.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, k.stream);
    cudaStreamSynchronize(k.stream);
    return (int64_t)k.h_best.p[0];
}

/* Global relocalization: score hypotheses h_begin .. h_begin+h-1 on this rank (calculateScore; the cost that is
 * minimised is -score, i.e. the winner is the most likely pose), then the argmin across ranks: every rank contributes its
 * local winner as a 16-byte (order-preserving fp64 score key, global index) pair to one ncclAllGather and all ranks take
 * the same maximum of the gathered pairs - exact in fp64, ties to the lowest hypothesis index. */
static int32_t reloc_argmin_impl(b200_comm* comm, b200_ndt* n, const float* poses16, int64_t h, int64_t h_begin, int64_t h_stride, int64_t* best,
                                 double* best_score, float* gpu_ms) {
    if (!n || (h > 0 && !poses16) || h < 0 || h_begin < 0 || h_stride < 1) B200_FAIL(B200_ERR_ARG, "bad argument");
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    const int R = comm && comm->nranks > 1 ? comm->nranks : 1;
    const int64_t hh = std::max<int64_t>(h, 1);
    CUDA_TRY(k.d_poses.reserve((size_t)hh * 16)); CUDA_TRY(k.h_poses.reserve((size_t)hh * 16));
    CUDA_TRY(k.d_scores.reserve(hh));
    CUDA_TRY(k.d_best.reserve(2 + 2 * (size_t)R)); CUDA_TRY(k.h_best.reserve(2 + 2 * (size_t)R));
    if (h) {
        memcpy(k.h_poses.p, poses16, (size_t)h * 16 * sizeof(float));
        CUDA_TRY(cudaMemcpyAsync(k.d_poses.p, k.h_poses.p, (size_t)h * 16 * sizeof(float), cudaMemcpyHostToDevice, k.stream));
    }
    unsigned long long* d = k.d_best.p;  // [0..1] local (key, index), [2..2+2R) the pairs of all ranks
    CUDA_TRY(cudaEventRecord(k.ev0, k.stream));
    // a rank whose scoring fails still takes part in the collective (with "no hypothesis"), so the healthy ranks do not
    // block in NCCL; the error is returned after the exchange
    int32_t rc_local = B200_OK;
    std::string err_local;
    if (h) {
        rc_local = k.score_batch_device(k.d_poses.p, h, k.d_scores.p);
        if (rc_local) err_local = g_last_error;
    }
    ndt::k_local_best<<<1, 256, 0, k.stream>>>(k.d_scores.p, rc_local ? 0 : h, h_begin, h_stride, d);
    LAUNCH_COUNT(1);
    if (R > 1) NCCL_TRY(comm, comm->AllGather(d, d + 2, 2, ncclUint64, comm->comm, k.stream));
    else CUDA_TRY(cudaMemcpyAsync(d + 2, d, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, k.stream));
    CUDA_TRY(cudaEventRecord(k.ev1, k.stream));
    CUDA_TRY(cudaMemcpyAsync(k.h_best.p, d + 2, 2 * (size_t)R * sizeof(unsigned long long), cudaMemcpyDeviceToHost, k.stream));
    CUDA_TRY(cudaStreamSynchronize(k.stream));
    CUDA_TRY(cudaGetLastError());
    cudaEventElapsedTime(&k.last_ms, k.ev0, k.ev1);
    if (gpu_ms) *gpu_ms = k.last_ms;
    if (rc_local) { g_last_error = err_local; return rc_local; }
    unsigned long long key = 0, idx = ~0ull;
    for (int r = 0; r < R; ++r) {
        const unsigned long long kr = k.h_best.p[2 * r], ir = k.h_best.p[2 * r + 1];
        if (kr > key || (kr == key && kr != 0 && ir < idx)) { key = kr; idx = ir; }
    }
    if (key == 0 || idx == ~0ull) { if (best) *best = -1; if (best_score) *best_score = 0; return B200_NO_EFFECTIVE_POINTS; }
    const unsigned long long u = (key >> 63) ? (key & 0x7FFFFFFFFFFFFFFFull) : ~key;
    double sc;
    memcpy(&sc, &u, 8);
    if (best) *best = (int64_t)idx;
    if (best_score) *best_score = sc;
    return B200_OK;
}
/* device time of the k_ndt_score_batch launch of the last score / relocalization call (CUDA events around that kernel alone) */
float b200_ndt_last_score_kernel_ms(b200_ndt* n) {
    if (!n) return 0.f;
    float ms = 0.f;
    cudaSetDevice(n->k.device);
    if (cudaEventElapsedTime(&ms, n->k.evs0, n->k.evs1) != cudaSuccess) { cudaGetLastError(); return 0.f; }
    return ms;
}
/* roofline bookkeeping: number of (source point, occupied neighbourhood voxel) pairs summed over h poses */
int32_t b200_ndt_score_pairs(b200_ndt* n, const float* poses16, int64_t h, int64_t* pairs) {
    if (!n || !poses16 || h < 1 || h > 65535 || !pairs) B200_FAIL(B200_ERR_ARG, "bad argument");
    Ndt& k = n->k;
    if (!k.have_target || k.n_src < 1) B200_FAIL(B200_ERR_ARG, "no target / source set");
    CUDA_SET_DEVICE(k.device);
    CUDA_TRY(k.d_poses.reserve((size_t)h * 16)); CUDA_TRY(k.h_poses.reserve((size_t)h * 16));
    CUDA_TRY(k.d_best.reserve(4)); CUDA_TRY(k.h_best.reserve(4));
    memcpy(k.h_poses.p, poses16, (size_t)h * 16 * sizeof(float));
    CUDA_TRY(cudaMemcpyAsync(k.d_poses.p, k.h_poses.p, (size_t)h * 16 * sizeof(float), cudaMemcpyHostToDevice, k.stream));
    CUDA_TRY(cudaMemsetAsync(k.d_best.p, 0, sizeof(unsigned long long), k.stream));
    ndt::k_ndt_pairs_batch<<<dim3(8, (unsigned)h), 256, 0, k.stream>>>(k.view(), k.d_poses.p, k.d_best.p);
    CUDA_TRY(cudaMemcpyAsync(k.h_best.p, k.d_best.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, k.stream));
    CUDA_TRY(cudaStreamSynchronize(k.stream));
    CUDA_TRY(cudaGetLastError());
    *pairs = (int64_t)k.h_best.p[0];
    return B200_OK;
}
/* Device-side rendezvous of the ranks on this handle's stream (a one-word ncclAllReduce): work enqueued afterwards starts
 * on all ranks together.  bench.py calls it before each timed relocalization step so that the per-step device time is
 * not inflated by the host-side start skew of the ranks. */
int32_t b200_ndt_stream_barrier(b200_comm* comm, b200_ndt* n) {
    if (!n) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (!comm || comm->nranks < 2) return B200_OK;
    Ndt& k = n->k;
    CUDA_SET_DEVICE(k.device);
    CUDA_TRY(k.d_bar.reserve(2));
    NCCL_TRY(comm, comm->AllReduce(k.d_bar.p, k.d_bar.p + 1, 1, ncclUint64, ncclSum, comm->comm, k.stream));
    return B200_OK;
}

int32_t b200_reloc_argmin(b200_comm* comm, b200_ndt* n, const float* poses16, int64_t h, int64_t h_begin, int64_t* best, double* best_score,
                          float* gpu_ms) {
    return reloc_argmin_impl(comm, n, poses16, h, h_begin, 1, best, best_score, gpu_ms);
}
/* same with the slice interleaved over the ranks: local hypothesis i is global hypothesis h_begin + i * h_stride (rank r of N
 * passes h_begin = r, h_stride = N) - neighbouring, similarly expensive hypotheses land on different ranks */
int32_t b200_reloc_argmin_strided(b200_comm* comm, b200_ndt* n, const float* poses16, int64_t h, int64_t h_begin, int64_t h_stride, int64_t* best,
                                  double* best_score, float* gpu_ms) {
    return reloc_argmin_impl(comm, n, poses16, h, h_begin, h_stride, best, best_score, gpu_ms);
}


int32_t b200_ndt_pairs_create(const b200_ndt_params* params, int32_t device, b200_ndt_pairs** out) {
    if (!params || !out) B200_FAIL(B200_ERR_ARG, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) B200_FAIL(B200_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) B200_FAIL(B200_ERR_ARG, "bad device ordinal");
    b200_ndt_pairs* h = new b200_ndt_pairs();
    const int32_t rc = h->k.init(params, device);
    if (rc != B200_OK) { h->destroy(); delete h; return rc; }
    *out = h;
    return B200_OK;
}
int32_t b200_ndt_pairs_destroy(b200_ndt_pairs* h) {
    if (!h) return B200_OK;
    h->destroy();
    delete h;
    return B200_OK;
}

/* P independent registrations (loop-closure candidates): see include/b200reg.h.  With a communicator of N ranks, rank r
 * registers the pairs p = r (mod N); the results and every rank's call status travel in ONE ncclAllGather of fixed-size
 * slots (ceil(P / N) records each), so all ranks return the same code and the same P results, and a rank that failed
 * locally still takes part in the collective. */
int32_t b200_ndt_pairs_align(b200_comm* comm, b200_ndt_pairs* h, const float* src_xyz, const int64_t* src_off, const float* tgt_xyz,
                             const int64_t* tgt_off, int64_t stride_bytes, int64_t P, const float* guesses16, double max_range,
                             b200_ndt_pair_result* results) {
    if (!h || !src_xyz || !src_off || !tgt_xyz || !tgt_off || !results || P < 1 || stride_bytes < 12) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (src_off[0] < 0 || tgt_off[0] < 0) B200_FAIL(B200_ERR_ARG, "negative offset");
    for (int64_t p = 0; p < P; ++p)
        if (src_off[p + 1] < src_off[p] || tgt_off[p + 1] < tgt_off[p]) B200_FAIL(B200_ERR_ARG, "offsets must not decrease");
    Ndt& K = h->k;
    CUDA_SET_DEVICE(K.device);
    const int R = comm && comm->nranks > 1 ? comm->nranks : 1, me = R > 1 ? comm->rank : 0;
    const int64_t per = (P + R - 1) / R;
    const size_t rec = sizeof(b200_ndt_pair_result), slot = 8 + (size_t)per * rec;
    if (R > 1) {  // before any work: past this point every rank reaches the collective
        CUDA_TRY(h->h_xchg.reserve(slot * (R + 1)));
        CUDA_TRY(h->d_xchg.reserve(slot * (R + 1)));
    }
    const b200_ndt_pairs::Call c{src_xyz, tgt_xyz, src_off, tgt_off, stride_bytes, guesses16, max_range, results};
    CUDA_TRY(cudaEventRecord(K.ev0, K.stream));
    const int32_t rc_local = h->local(c, P, me, R);
    const std::string err_local = rc_local ? g_last_error : std::string();
    if (R == 1 && rc_local) return rc_local;
    if (R > 1) {
        uint8_t* hs = h->h_xchg.p;
        memset(hs, 0, 8);
        memcpy(hs, &rc_local, sizeof(int32_t));
        for (int64_t i = 0, p = me; p < P; ++i, p += R) memcpy(hs + 8 + i * rec, &results[p], rec);
        CUDA_TRY(cudaMemcpyAsync(h->d_xchg.p, hs, slot, cudaMemcpyHostToDevice, K.stream));
        NCCL_TRY(comm, comm->AllGather(h->d_xchg.p, h->d_xchg.p + slot, slot, ncclChar, comm->comm, K.stream));
        CUDA_TRY(cudaMemcpyAsync(hs + slot, h->d_xchg.p + slot, slot * R, cudaMemcpyDeviceToHost, K.stream));
        CUDA_TRY(cudaStreamSynchronize(K.stream));
        int32_t rc = B200_OK;
        int bad = -1;
        for (int q = 0; q < R; ++q) {
            const uint8_t* b = hs + slot * (q + 1);
            int32_t sq;
            memcpy(&sq, b, sizeof sq);
            if (sq && rc == B200_OK) { rc = sq; bad = q; }
            for (int64_t i = 0, p = q; p < P; ++i, p += R) {
                memcpy(&results[p], b + 8 + i * rec, rec);
                if (sq) results[p].status = sq;
            }
        }
        if (rc) {
            if (bad == me) g_last_error = err_local;
            else fail(rc, ("NDT pair registration failed on rank " + std::to_string(bad)).c_str(), __FILE__, __LINE__);
            return rc;
        }
    }
    CUDA_TRY(cudaEventRecord(K.ev1, K.stream));
    CUDA_TRY(cudaEventSynchronize(K.ev1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, K.ev0, K.ev1);
    K.last_ms = ms;
    for (int64_t p = 0; p < P; ++p) results[p].ndt.gpu_ms = ms;
    return B200_OK;
}

int64_t b200_ndt_pairs_leaves(b200_ndt_pairs* h, int64_t p, int64_t max, int64_t* ids, int32_t* npts, double* mean3, double* cov9, double* icov9) {
    if (!h) return -1;
    size_t j = 0;
    while (j < h->last_ids.size() && h->last_ids[j] != p) ++j;
    if (j == h->last_ids.size() || !h->last_live[j]) return -1;
    Ndt& k = h->k;
    cudaSetDevice(k.device);
    const int nr = h->last_nruns;
    std::vector<uint8_t> valid(nr);
    std::vector<uint32_t> uniq(nr);
    std::vector<int32_t> np(nr);
    std::vector<ndt::LeafD> L(nr);
    std::vector<double> cov((size_t)nr * 9);
    cudaStreamSynchronize(k.stream);
    cudaMemcpy(valid.data(), k.d_valid.p, nr, cudaMemcpyDeviceToHost);
    cudaMemcpy(uniq.data(), k.d_uniq.p, nr * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaMemcpy(np.data(), k.d_npts.p, nr * sizeof(int32_t), cudaMemcpyDeviceToHost);
    cudaMemcpy(L.data(), k.d_leafD.p, nr * sizeof(ndt::LeafD), cudaMemcpyDeviceToHost);
    cudaMemcpy(cov.data(), k.d_cov.p, (size_t)nr * 9 * sizeof(double), cudaMemcpyDeviceToHost);
    const uint64_t lo = h->last_base[j], hi = lo + (uint64_t)h->last_ncells[j];
    int64_t cnt = 0;
    for (int r = 0; r < nr; ++r) {  // runs are sorted by key = cell_base + leaf id
        if (!valid[r] || uniq[r] < lo || uniq[r] >= hi) continue;
        if (cnt < max) {
            if (ids) ids[cnt] = (int64_t)(uniq[r] - lo);
            if (npts) npts[cnt] = np[r];
            if (mean3) memcpy(mean3 + cnt * 3, L[r].mean, 24);
            if (cov9) memcpy(cov9 + cnt * 9, &cov[(size_t)r * 9], 72);
            if (icov9) memcpy(icov9 + cnt * 9, L[r].icov, 72);
        }
        ++cnt;
    }
    return cnt;
}

}  // extern "C"
