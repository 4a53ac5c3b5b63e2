// b200reg — LOAM-style scan-to-map optimisation (the estimator of jueying_slam), on the local-map index of map.cuh.
//
// Replaces, in jueying_slam/src/mapOptmization.cpp: cornerOptimization (:1255-1347), surfOptimization (:1349-1419),
// combineOptimizationCoeffs (:1420-1440), LMOptimization (:1442-1558) and the loop of scan2MapOptimization (:1560-1590);
// kdtree{Corner,Surf}FromMap->setInputCloud (:1568-1569) becomes b200_loam_set_map, or b200_loam_set_map_from_keyframes, which
// builds the two maps from the device keyframe store (extractSurroundingKeyFrames, loop.cu) and inserts them from the device.
//
// pcl::KdTreeFLANN::nearestKSearch(pointSel, 5) followed by the gate pointSearchSqDis[4] < 1.0 is an exact 5-NN query
// whose answer only matters when all five neighbours lie within 1 m: on a voxel index with 1 m cells that is precisely
// the 27-cell stencil search with max_range 1.0 that the IEKF path already uses (every point closer than 1 m is in the
// stencil; fewer than five hits <=> the gate fails).  So both feature clouds live in a b200::Map (resolution 1, NEARBY26,
// range 1) and the search kernel is the same knn5_group.
//
// Per iteration two launches: k_loam_search (8 lanes per feature point) and k_loam_accum (one thread per point: line /
// plane fit, coefficient, Jacobian row; fp64 block sums of A^T A, A^T b; the last block reduces the partials in block
// order and takes the LM step: 6x6 solve, degeneracy projection, transform update, convergence test).  The host polls a
// done flag every few iterations.  Arithmetic is fp32 in the reference's order (TU built with -fmad=false).
#include "loop.cuh"
#include "map.cuh"
#include "pointmath.cuh"

#include <algorithm>
#include <vector>

namespace b200 {
namespace loam {

constexpr int G = 8;
constexpr int NSUM = 28;  // 21 unique A^T A entries, 6 A^T b entries, selected-point count
constexpr int ACC_THREADS = 256;
constexpr int MAXB = 1024;

struct Ctl {
    float t6[6];   // transformTobeMapped: roll, pitch, yaw, x, y, z
    float T[12];   // pcl::getTransformation of t6, row-major 3x4
    float matP[36];
    int iter, done, converged, degenerate, n_sel, max_iter;
    unsigned int ticket;
    int pad;
    double AtA_first[36];
};

__device__ inline float fsin_cr(float a) { return (float)sin((double)a); }
__device__ inline float fcos_cr(float a) { return (float)cos((double)a); }

// pcl::getTransformation(x, y, z, roll, pitch, yaw) (PCL common/eigen.hpp), float
__device__ inline void pose_matrix(const float* t6, float* T) {
    const float roll = t6[0], pitch = t6[1], yaw = t6[2];
    const float A = fcos_cr(yaw), B = fsin_cr(yaw), C = fcos_cr(pitch), D = fsin_cr(pitch), E = fcos_cr(roll), F = fsin_cr(roll), DE = D * E, DF = D * F;
    T[0] = A * C; T[1] = A * DF - B * E; T[2] = B * F + A * DE; T[3] = t6[3];
    T[4] = B * C; T[5] = A * E + B * DF; T[6] = B * DE - A * F; T[7] = t6[4];
    T[8] = -D;    T[9] = C * F;          T[10] = C * E;         T[11] = t6[5];
}

// cv::eigen on a symmetric float matrix: eigenvalues descending, eigenvectors in the rows of V (cyclic Jacobi in fp32)
template <int N>
__device__ inline void eigen_desc_f(const float* Ain, float* w, float* V) {
    float A[N * N], U[N * N];
#pragma unroll
    for (int i = 0; i < N * N; ++i) A[i] = Ain[i];
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) U[i * N + j] = (i == j) ? 1.0f : 0.0f;
    for (int sweep = 0; sweep < 30; ++sweep) {
        float off = 0.f, diag = 0.f;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            diag += A[i * N + i] * A[i * N + i];
#pragma unroll
            for (int j = i + 1; j < N; ++j) off += A[i * N + j] * A[i * N + j];
        }
        if (off <= 1e-30f || off <= 1e-14f * diag) break;
#pragma unroll
        for (int p = 0; p < N - 1; ++p)
#pragma unroll
            for (int q = p + 1; q < N; ++q) {
                const float apq = A[p * N + q];
                if (apq != 0.0f) {
                    const float theta = (A[q * N + q] - A[p * N + p]) / (2.0f * apq);
                    const float t = (theta >= 0 ? 1.0f : -1.0f) / (fabsf(theta) + sqrtf(theta * theta + 1.0f));
                    const float c = 1.0f / sqrtf(t * t + 1.0f), s = t * c;
#pragma unroll
                    for (int k = 0; k < N; ++k) {
                        const float akp = A[k * N + p], akq = A[k * N + q];
                        A[k * N + p] = c * akp - s * akq;
                        A[k * N + q] = s * akp + c * akq;
                    }
#pragma unroll
                    for (int k = 0; k < N; ++k) {
                        const float apk = A[p * N + k], aqk = A[q * N + k];
                        A[p * N + k] = c * apk - s * aqk;
                        A[q * N + k] = s * apk + c * aqk;
                    }
#pragma unroll
                    for (int k = 0; k < N; ++k) {
                        const float ukp = U[k * N + p], ukq = U[k * N + q];
                        U[k * N + p] = c * ukp - s * ukq;
                        U[k * N + q] = s * ukp + c * ukq;
                    }
                }
            }
    }
    int order[N];
#pragma unroll
    for (int i = 0; i < N; ++i) order[i] = i;
    for (int i = 0; i < N - 1; ++i) {
        int m = i;
        for (int j = i + 1; j < N; ++j)
            if (A[order[j] * N + order[j]] > A[order[m] * N + order[m]]) m = j;
        const int t = order[i]; order[i] = order[m]; order[m] = t;
    }
    for (int i = 0; i < N; ++i) {
        w[i] = A[order[i] * N + order[i]];
        for (int k = 0; k < N; ++k) V[i * N + k] = U[k * N + order[i]];
    }
}

// cornerOptimization body for one point (:1281-1343): nb = its five nearest map points; returns whether it is selected
__device__ inline bool corner_feature(const float4* nb, float x0, float y0, float z0, float* coeff) {
    float cx = 0, cy = 0, cz = 0;
    for (int j = 0; j < 5; ++j) { cx += nb[j].x; cy += nb[j].y; cz += nb[j].z; }
    cx /= 5; cy /= 5; cz /= 5;
    float a11 = 0, a12 = 0, a13 = 0, a22 = 0, a23 = 0, a33 = 0;
    for (int j = 0; j < 5; ++j) {
        const float ax = nb[j].x - cx, ay = nb[j].y - cy, az = nb[j].z - cz;
        a11 += ax * ax; a12 += ax * ay; a13 += ax * az; a22 += ay * ay; a23 += ay * az; a33 += az * az;
    }
    a11 /= 5; a12 /= 5; a13 /= 5; a22 /= 5; a23 /= 5; a33 /= 5;
    const float A[9] = {a11, a12, a13, a12, a22, a23, a13, a23, a33};
    float D[3], V[9];
    eigen_desc_f<3>(A, D, V);
    if (!(D[0] > 3 * D[1])) return false;
    const float x1 = (float)((double)cx + 0.1 * (double)V[0]), y1 = (float)((double)cy + 0.1 * (double)V[1]), z1 = (float)((double)cz + 0.1 * (double)V[2]);
    const float x2 = (float)((double)cx - 0.1 * (double)V[0]), y2 = (float)((double)cy - 0.1 * (double)V[1]), z2 = (float)((double)cz - 0.1 * (double)V[2]);
    const float m11 = (x0 - x1) * (y0 - y2) - (x0 - x2) * (y0 - y1), m22 = (x0 - x1) * (z0 - z2) - (x0 - x2) * (z0 - z1),
                m33 = (y0 - y1) * (z0 - z2) - (y0 - y2) * (z0 - z1);
    const float a012 = sqrtf(m11 * m11 + m22 * m22 + m33 * m33);
    const float l12 = sqrtf((x1 - x2) * (x1 - x2) + (y1 - y2) * (y1 - y2) + (z1 - z2) * (z1 - z2));
    const float la = ((y1 - y2) * m11 + (z1 - z2) * m22) / a012 / l12;
    const float lb = -((x1 - x2) * m11 - (z1 - z2) * m33) / a012 / l12;
    const float lc = -((x1 - x2) * m22 + (y1 - y2) * m33) / a012 / l12;
    const float ld2 = a012 / l12;
    const float s = (float)(1.0 - 0.9 * (double)fabsf(ld2));
    coeff[0] = s * la; coeff[1] = s * lb; coeff[2] = s * lc; coeff[3] = s * ld2;
    return (double)s > 0.1;
}
// surfOptimization body for one point (:1375-1415)
__device__ inline bool surf_feature(const float4* nb, float x0, float y0, float z0, float* coeff) {
    float q[5][3], X[3];
#pragma unroll
    for (int r = 0; r < 5; ++r) { q[r][0] = nb[r].x; q[r][1] = nb[r].y; q[r][2] = nb[r].z; }
    qr_solve_neg1<float, 5>(q, X);
    float pa = X[0], pb = X[1], pc = X[2], pd = 1;
    const float ps = sqrtf(pa * pa + pb * pb + pc * pc);
    pa /= ps; pb /= ps; pc /= ps; pd /= ps;
    for (int j = 0; j < 5; ++j)
        if ((double)fabsf(pa * nb[j].x + pb * nb[j].y + pc * nb[j].z + pd) > 0.2) return false;
    const float pd2 = pa * x0 + pb * y0 + pc * z0 + pd;
    const float s = (float)(1.0 - 0.9 * (double)fabsf(pd2) / (double)sqrtf(sqrtf(x0 * x0 + y0 * y0 + z0 * z0)));
    coeff[0] = s * pa; coeff[1] = s * pb; coeff[2] = s * pc; coeff[3] = s * pd2;
    return (double)s > 0.1;
}

template <int MODE>
__global__ void __launch_bounds__(256, MODE == 0 ? 5 : 4) k_loam_search(MapView map, const float4* __restrict__ pts, int n, const Ctl* __restrict__ ctl,
                                                                      float4* __restrict__ nb_out, unsigned char* __restrict__ cnt_out) {
    if (ctl->done) return;
    __shared__ float T[12];
    const int tid = threadIdx.x;
    if (tid < 12) T[tid] = ctl->T[tid];
    __syncthreads();
    const int q = (blockIdx.x * blockDim.x + tid) / G, lg = tid % G;
    if (q >= n) return;
    const unsigned gmask = ((1u << G) - 1u) << ((tid & 31) / G * G);
    const float4 p = __ldg(pts + q);
    const float x = T[0] * p.x + T[1] * p.y + T[2] * p.z + T[3], y = T[4] * p.x + T[5] * p.y + T[6] * p.z + T[7],
                z = T[8] * p.x + T[9] * p.y + T[10] * p.z + T[11];  // pointAssociateToMap (:439-445)
    uint64_t wkey;
    float4 mine;
    __shared__ uint2 s_flat[MODE == 5 ? (256 / G) * kFlatStride : 1];
    const int c = knn5_group<G, MODE>(map, x, y, z, lg, gmask, lane_stencil<G>(lg, map.nstencil), wkey, mine,
                                      MODE == 5 ? s_flat + (tid / G) * kFlatStride : nullptr);
    if (lg < 5) nb_out[(size_t)q * 5 + lg] = mine;
    if (lg == 0) cnt_out[q] = (unsigned char)c;
}

struct AccSmem {
    float T[12];
    float trig[6];
    double red[ACC_THREADS / 32][NSUM];
    double res[NSUM];
    int is_last;
};

// thread 0 of the last block: LMOptimization from the reduced sums (:1504-1557)
__device__ void lm_step(Ctl& c, const double* sums) {
    const int n_sel = (int)sums[27];
    c.n_sel = n_sel;
    const int it = c.iter;
    c.iter = it + 1;
    if (c.iter >= c.max_iter) c.done = 1;
    if (n_sel < 50) return;  // LMOptimization returns false: the transform stays, the loop goes on
    float Af[36], Bf[6];
    {
        int k = 0;
        for (int r = 0; r < 6; ++r)
            for (int cc = r; cc < 6; ++cc) { Af[r * 6 + cc] = Af[cc * 6 + r] = (float)sums[k]; ++k; }
        for (int r = 0; r < 6; ++r) Bf[r] = (float)sums[21 + r];
    }
    if (it == 0) for (int i = 0; i < 36; ++i) c.AtA_first[i] = Af[i];
    double M[6][7];
    for (int r = 0; r < 6; ++r) { for (int cc = 0; cc < 6; ++cc) M[r][cc] = Af[r * 6 + cc]; M[r][6] = Bf[r]; }
    for (int k = 0; k < 6; ++k) {  // cv::solve(DECOMP_QR) on the normal equations, restated as pivoted elimination in fp64
        int piv = k;
        for (int r = k + 1; r < 6; ++r) if (fabs(M[r][k]) > fabs(M[piv][k])) piv = r;
        if (piv != k) for (int cc = 0; cc < 7; ++cc) { const double t = M[k][cc]; M[k][cc] = M[piv][cc]; M[piv][cc] = t; }
        for (int r = k + 1; r < 6; ++r) {
            const double f = M[r][k] / M[k][k];
            for (int cc = k; cc < 7; ++cc) M[r][cc] -= f * M[k][cc];
        }
    }
    double xs[6];
    for (int r = 5; r >= 0; --r) {
        double s = M[r][6];
        for (int cc = r + 1; cc < 6; ++cc) s -= M[r][cc] * xs[cc];
        xs[r] = s / M[r][r];
    }
    float X[6];
    for (int i = 0; i < 6; ++i) X[i] = (float)xs[i];
    if (it == 0) {  // degeneracy test on the first iteration (:1513-1535)
        float E[6], V[36], V2[36];
        eigen_desc_f<6>(Af, E, V);
        for (int i = 0; i < 36; ++i) V2[i] = V[i];
        bool deg = false;
        for (int i = 5; i >= 0; --i) {
            if (E[i] < 100.0f) {
                for (int j = 0; j < 6; ++j) V2[i * 6 + j] = 0;
                deg = true;
            } else break;
        }
        c.degenerate = deg ? 1 : 0;
        for (int r = 0; r < 6; ++r)
            for (int cc = 0; cc < 6; ++cc) {
                float s = 0;
                for (int k = 0; k < 6; ++k) s += V[k * 6 + r] * V2[k * 6 + cc];
                c.matP[r * 6 + cc] = s;
            }
    }
    if (c.degenerate) {
        float X2[6];
        for (int i = 0; i < 6; ++i) X2[i] = X[i];
        for (int r = 0; r < 6; ++r) {
            float s = 0;
            for (int k = 0; k < 6; ++k) s += c.matP[r * 6 + k] * X2[k];
            X[r] = s;
        }
    }
    for (int i = 0; i < 6; ++i) c.t6[i] += X[i];
    pose_matrix(c.t6, c.T);
    const float r2d = 180.0f / 3.14159265358979323846f;
    const float deltaR = sqrtf((X[0] * r2d) * (X[0] * r2d) + (X[1] * r2d) * (X[1] * r2d) + (X[2] * r2d) * (X[2] * r2d));
    const float deltaT = sqrtf((X[3] * 100) * (X[3] * 100) + (X[4] * 100) * (X[4] * 100) + (X[5] * 100) * (X[5] * 100));
    if ((double)deltaR < 0.01 && (double)deltaT < 0.05) { c.converged = 1; c.done = 1; }
}

// points [0, nc) are corner features, [nc, n) surface features
__global__ void __launch_bounds__(ACC_THREADS) k_loam_accum(const float4* __restrict__ pts, const float4* __restrict__ nb, const unsigned char* __restrict__ cnt,
                                                            int nc, int n, Ctl* ctl, double* partials, int single, uint8_t* __restrict__ flags_out,
                                                            float4* __restrict__ coeff_out) {
    if (ctl->done && !single) return;
    __shared__ AccSmem sm;
    const int tid = threadIdx.x, nb_x = gridDim.x;
    if (tid < 12) sm.T[tid] = ctl->T[tid];
    if (tid == 0) {
        const float* t6 = ctl->t6;  // LMOptimization's srx.. are sin/cos of transformTobeMapped[1], [2], [0] (:1445-1450)
        sm.trig[0] = fsin_cr(t6[1]); sm.trig[1] = fcos_cr(t6[1]); sm.trig[2] = fsin_cr(t6[2]);
        sm.trig[3] = fcos_cr(t6[2]); sm.trig[4] = fsin_cr(t6[0]); sm.trig[5] = fcos_cr(t6[0]);
    }
    __syncthreads();
    double acc[NSUM];
#pragma unroll
    for (int i = 0; i < NSUM; ++i) acc[i] = 0.0;
    for (int i = blockIdx.x * ACC_THREADS + tid; i < n; i += nb_x * ACC_THREADS) {
        bool sel = false;
        float co[4] = {0.f, 0.f, 0.f, 0.f};
        const float4 p = __ldg(pts + i);
        if (cnt[i] == 5) {  // fewer than five neighbours within 1 m <=> pointSearchSqDis[4] >= 1.0
            float4 nbp[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) nbp[j] = __ldg(nb + (size_t)i * 5 + j);
            const float* T = sm.T;
            const float x0 = T[0] * p.x + T[1] * p.y + T[2] * p.z + T[3], y0 = T[4] * p.x + T[5] * p.y + T[6] * p.z + T[7],
                        z0 = T[8] * p.x + T[9] * p.y + T[10] * p.z + T[11];
            sel = i < nc ? corner_feature(nbp, x0, y0, z0, co) : surf_feature(nbp, x0, y0, z0, co);
        }
        if (flags_out) {
            flags_out[i] = sel ? 1 : 0;
            coeff_out[i] = sel ? make_float4(co[0], co[1], co[2], co[3]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (!sel) continue;
        const float srx = sm.trig[0], crx = sm.trig[1], sry = sm.trig[2], cry = sm.trig[3], srz = sm.trig[4], crz = sm.trig[5];
        const float px = p.y, py = p.z, pz = p.x;               // lidar -> camera axes (:1471-1473)
        const float cx = co[1], cy = co[2], cz = co[0], ci = co[3];
        const float arx = (crx * sry * srz * px + crx * crz * sry * py - srx * sry * pz) * cx + (-srx * srz * px - crz * srx * py - crx * pz) * cy +
                          (crx * cry * srz * px + crx * cry * crz * py - cry * srx * pz) * cz;
        const float ary = ((cry * srx * srz - crz * sry) * px + (sry * srz + cry * crz * srx) * py + crx * cry * pz) * cx +
                          ((-cry * crz - srx * sry * srz) * px + (cry * srz - crz * srx * sry) * py - crx * sry * pz) * cz;
        const float arz = ((crz * srx * sry - cry * srz) * px + (-cry * crz - srx * sry * srz) * py) * cx + (crx * crz * px - crx * srz * py) * cy +
                          ((sry * srz + cry * crz * srx) * px + (crz * sry - cry * srx * srz) * py) * cz;
        const float row[6] = {arz, arx, ary, cz, cx, cy};
        const float b = -ci;
        int k = 0;
#pragma unroll
        for (int r = 0; r < 6; ++r)
#pragma unroll
            for (int c = r; c < 6; ++c) { acc[k] += (double)row[r] * (double)row[c]; ++k; }
#pragma unroll
        for (int r = 0; r < 6; ++r) acc[21 + r] += (double)row[r] * (double)b;
        acc[27] += 1.0;
    }
    if (single) return;
#pragma unroll
    for (int i = 0; i < NSUM; ++i) {
        double a = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if ((tid & 31) == 0) sm.red[tid >> 5][i] = a;
    }
    __syncthreads();
    if (tid < NSUM) {
        double a = sm.red[0][tid];
#pragma unroll
        for (int w = 1; w < ACC_THREADS / 32; ++w) a += sm.red[w][tid];
        __stcg(partials + (size_t)tid * nb_x + blockIdx.x, a);
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) sm.is_last = (atomicAdd(&ctl->ticket, 1u) == (unsigned)nb_x - 1u);
    __syncthreads();
    if (!sm.is_last) return;
    __threadfence();
    if (tid < NSUM) {
        const double* src = partials + (size_t)tid * nb_x;
        double a = 0.0;
        for (int b = 0; b < nb_x; ++b) a += __ldcg(src + b);
        sm.res[tid] = a;
    }
    __syncthreads();
    if (tid == 0) {
        ctl->ticket = 0;
        lm_step(*ctl, sm.res);
    }
}

__global__ void k_loam_init(Ctl* ctl, const float* __restrict__ t6, int max_iter) {
    if (threadIdx.x != 0) return;
    for (int i = 0; i < 6; ++i) ctl->t6[i] = t6[i];
    pose_matrix(ctl->t6, ctl->T);
    ctl->iter = 0; ctl->done = 0; ctl->converged = 0; ctl->degenerate = 0; ctl->n_sel = 0; ctl->max_iter = max_iter; ctl->ticket = 0;
    for (int i = 0; i < 36; ++i) { ctl->matP[i] = 0.f; ctl->AtA_first[i] = 0.0; }
}

}  // namespace loam
}  // namespace b200

using namespace b200;
struct b200_loam {
    Map corner, surf;
    bool have_maps = false, inited = false;
    int device = 0;
    cudaStream_t stream = nullptr;  // = corner.stream; the surf map's work is ordered through events
    loam::Ctl* d_ctl = nullptr;
    DevBuf<float4> d_pts, d_nb, d_coeff;
    DevBuf<unsigned char> d_cnt;
    DevBuf<uint8_t> d_flags;
    DevBuf<double> d_partials;
    DevBuf<float> d_t6;
    PinnedBuf<float4> h_stage;
    PinnedBuf<loam::Ctl> h_ctl;
    PinnedBuf<float> h_t6;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_map = nullptr;
    float last_ms = 0.f;
    int last_launches = 0;
};

static int32_t loam_stage(b200_loam* h, const float* corner, int64_t nc, int64_t sc, const float* surf, int64_t ns, int64_t ss, const float* t6, int max_iter) {
    const int64_t n = nc + ns;
    CUDA_TRY(h->h_stage.reserve(n));
    CUDA_TRY(h->d_pts.reserve(n)); CUDA_TRY(h->d_nb.reserve(n * 5)); CUDA_TRY(h->d_cnt.reserve(n));
    CUDA_TRY(h->d_t6.reserve(8)); CUDA_TRY(h->h_t6.reserve(8));
    if (nc) pack_xyz_float4(corner, nc, sc, h->h_stage.p);
    if (ns) pack_xyz_float4(surf, ns, ss, h->h_stage.p + nc);
    memcpy(h->h_t6.p, t6, 6 * sizeof(float));
    CUDA_TRY(cudaMemcpyAsync(h->d_pts.p, h->h_stage.p, n * sizeof(float4), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemcpyAsync(h->d_t6.p, h->h_t6.p, 6 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    loam::k_loam_init<<<1, 32, 0, h->stream>>>(h->d_ctl, h->d_t6.p, max_iter);
    LAUNCH_COUNT(1);
    return B200_OK;
}

// the device-resident twin of pack_xyz_float4: (x, y, z, 0)
__global__ void k_loam_stage_device(const float4* __restrict__ c, int64_t nc, const float4* __restrict__ s, int64_t n, float4* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = i < nc ? c[i] : s[i - nc];
    out[i] = make_float4(p.x, p.y, p.z, 0.0f);
}
static int32_t loam_stage_device(b200_loam* h, const float4* corner, int64_t nc, const float4* surf, int64_t ns, const float* t6, int max_iter) {
    const int64_t n = nc + ns;
    CUDA_TRY(h->d_pts.reserve(n)); CUDA_TRY(h->d_nb.reserve(n * 5)); CUDA_TRY(h->d_cnt.reserve(n));
    CUDA_TRY(h->d_t6.reserve(8)); CUDA_TRY(h->h_t6.reserve(8));
    memcpy(h->h_t6.p, t6, 6 * sizeof(float));
    k_loam_stage_device<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(corner, nc, surf, n, h->d_pts.p);
    CUDA_TRY(cudaMemcpyAsync(h->d_t6.p, h->h_t6.p, 6 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    loam::k_loam_init<<<1, 32, 0, h->stream>>>(h->d_ctl, h->d_t6.p, max_iter);
    LAUNCH_COUNT(2);
    return B200_OK;
}

static int32_t loam_iterate(b200_loam* h, int64_t n_corner, int64_t n_surf, float* t6, int32_t iter_num, b200_loam_stats* stats);

static void loam_search(b200_loam* h, int64_t nc, int64_t ns) {
    using namespace loam;
    if (nc) {
        const unsigned grid = (unsigned)((nc * G + 255) / 256);
        if (h->corner.knn_mode_g8() >= 5) k_loam_search<5><<<grid, 256, 0, h->stream>>>(h->corner.view(), h->d_pts.p, (int)nc, h->d_ctl, h->d_nb.p, h->d_cnt.p);
        else if (h->corner.knn_mode_g8() == 1) k_loam_search<1><<<grid, 256, 0, h->stream>>>(h->corner.view(), h->d_pts.p, (int)nc, h->d_ctl, h->d_nb.p, h->d_cnt.p);
        else k_loam_search<0><<<grid, 256, 0, h->stream>>>(h->corner.view(), h->d_pts.p, (int)nc, h->d_ctl, h->d_nb.p, h->d_cnt.p);
    }
    if (ns) {
        const unsigned grid = (unsigned)((ns * G + 255) / 256);
        if (h->surf.knn_mode_g8() >= 5) k_loam_search<5><<<grid, 256, 0, h->stream>>>(h->surf.view(), h->d_pts.p + nc, (int)ns, h->d_ctl, h->d_nb.p + nc * 5, h->d_cnt.p + nc);
        else if (h->surf.knn_mode_g8() == 1) k_loam_search<1><<<grid, 256, 0, h->stream>>>(h->surf.view(), h->d_pts.p + nc, (int)ns, h->d_ctl, h->d_nb.p + nc * 5, h->d_cnt.p + nc);
        else k_loam_search<0><<<grid, 256, 0, h->stream>>>(h->surf.view(), h->d_pts.p + nc, (int)ns, h->d_ctl, h->d_nb.p + nc * 5, h->d_cnt.p + nc);
    }
    LAUNCH_COUNT((nc ? 1 : 0) + (ns ? 1 : 0));
}

extern "C" {

/* max_map_points: upper bound on the size of either feature map (laserCloud{Corner,Surf}FromMapDS) */
int32_t b200_loam_create(int64_t max_map_points, int32_t device, b200_loam** out) {
    if (!out || max_map_points < 16) B200_FAIL(B200_ERR_ARG, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) B200_FAIL(B200_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) B200_FAIL(B200_ERR_ARG, "bad device ordinal");
    b200_loam* h = new b200_loam();
    h->device = device;
    b200_map_params p{};
    p.resolution = 1.0f;   // the gate pointSearchSqDis[4] < 1.0 (mapOptmization.cpp:1276,1375)
    p.nearby = 26;
    p.capacity_voxels = (uint64_t)max_map_points + 1024;
    p.max_range = 1.0f;
    p.max_points = (uint64_t)max_map_points;
    int32_t rc = h->corner.init(&p, device);
    if (rc == B200_OK) rc = h->surf.init(&p, device);
    if (rc != B200_OK) { h->corner.destroy(); h->surf.destroy(); delete h; return rc; }
    h->inited = true;
    h->stream = h->corner.stream;
    CUDA_TRY(cudaMalloc(&h->d_ctl, sizeof(loam::Ctl)));
    CUDA_TRY(cudaMemset(h->d_ctl, 0, sizeof(loam::Ctl)));
    CUDA_TRY(h->h_ctl.reserve(1));
    CUDA_TRY(h->d_partials.reserve((size_t)loam::NSUM * loam::MAXB));
    CUDA_TRY(cudaEventCreate(&h->ev0)); CUDA_TRY(cudaEventCreate(&h->ev1)); CUDA_TRY(cudaEventCreate(&h->ev_map));
    *out = h;
    return B200_OK;
}
int32_t b200_loam_destroy(b200_loam* h) {
    if (!h) return B200_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->d_ctl);
    h->d_pts.release(); h->d_nb.release(); h->d_coeff.release(); h->d_cnt.release(); h->d_flags.release(); h->d_partials.release(); h->d_t6.release();
    h->h_stage.release(); h->h_ctl.release(); h->h_t6.release();
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev_map) cudaEventDestroy(h->ev_map);
    if (h->inited) { h->corner.destroy(); h->surf.destroy(); }
    delete h;
    return B200_OK;
}
/* kdtreeCornerFromMap->setInputCloud(laserCloudCornerFromMapDS); kdtreeSurfFromMap->setInputCloud(laserCloudSurfFromMapDS)
 * (mapOptmization.cpp:1568-1569): replaces both feature maps */
int32_t b200_loam_set_map(b200_loam* h, const float* corner_xyz, int64_t n_corner, int64_t stride_corner, const float* surf_xyz, int64_t n_surf,
                          int64_t stride_surf) {
    if (!h || n_corner < 0 || n_surf < 0 || (n_corner && (!corner_xyz || stride_corner < 12)) || (n_surf && (!surf_xyz || stride_surf < 12)))
        B200_FAIL(B200_ERR_ARG, "bad argument");
    // a feature map larger than the handle was created for would make the voxel table evict (LRU) map points silently
    if ((uint64_t)n_corner > h->corner.prm.max_points || (uint64_t)n_surf > h->surf.prm.max_points)
        B200_FAIL(B200_ERR_CAPACITY, "feature map larger than max_map_points of b200_loam_create");
    CUDA_SET_DEVICE(h->device);
    int32_t rc = h->corner.clear();
    if (rc == B200_OK) rc = h->surf.clear();
    if (rc == B200_OK && n_corner) rc = h->corner.insert_host(corner_xyz, n_corner, stride_corner);
    if (rc == B200_OK && n_surf) rc = h->surf.insert_host(surf_xyz, n_surf, stride_surf);
    if (rc != B200_OK) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->corner.stream));
    CUDA_TRY(cudaStreamSynchronize(h->surf.stream));
    h->have_maps = true;
    return B200_OK;
}
/* The loop of scan2MapOptimization (mapOptmization.cpp:1571-1583) for one scan: corner / surf = laserCloud{Corner,Surf}LastDS in
 * the lidar frame; t6 = transformTobeMapped (roll, pitch, yaw, x, y, z), updated in place.  Returns B200_NOT_CONVERGED when
 * iter_num passes ran without LMOptimization reporting convergence (the reference carries on with the transform it has). */
int32_t b200_loam_optimize(b200_loam* h, const float* corner_xyz, int64_t n_corner, int64_t stride_corner, const float* surf_xyz, int64_t n_surf,
                           int64_t stride_surf, float* t6, int32_t iter_num, b200_loam_stats* stats) {
    if (!h || !t6 || n_corner < 0 || n_surf < 0 || n_corner + n_surf < 1 || iter_num < 1 || iter_num > 1000 || n_corner + n_surf > (1 << 26))
        B200_FAIL(B200_ERR_ARG, "bad argument");
    if (!h->have_maps) B200_FAIL(B200_ERR_ARG, "no feature maps set");
    CUDA_SET_DEVICE(h->device);
    int32_t rc = loam_stage(h, corner_xyz, n_corner, stride_corner, surf_xyz, n_surf, stride_surf, t6, iter_num);
    if (rc) return rc;
    return loam_iterate(h, n_corner, n_surf, t6, iter_num, stats);
}
int32_t b200_loam_optimize_device(b200_loam* h, const void* d_corner, int64_t n_corner, const void* d_surf, int64_t n_surf, float* t6, int32_t iter_num,
                                  b200_loam_stats* stats) {
    if (!h || !t6 || n_corner < 0 || n_surf < 0 || n_corner + n_surf < 1 || iter_num < 1 || iter_num > 1000 || n_corner + n_surf > (1 << 26))
        B200_FAIL(B200_ERR_ARG, "bad argument");
    if (!h->have_maps) B200_FAIL(B200_ERR_ARG, "no feature maps set");
    CUDA_SET_DEVICE(h->device);
    if (const int32_t rc = check_device_buffer(d_corner, n_corner, h->device)) return rc;
    if (const int32_t rc = check_device_buffer(d_surf, n_surf, h->device)) return rc;
    const int32_t rc = loam_stage_device(h, (const float4*)d_corner, n_corner, (const float4*)d_surf, n_surf, t6, iter_num);
    if (rc) return rc;
    return loam_iterate(h, n_corner, n_surf, t6, iter_num, stats);
}
}  // extern "C"

// the loop of scan2MapOptimization on the staged scan
static int32_t loam_iterate(b200_loam* h, int64_t n_corner, int64_t n_surf, float* t6, int32_t iter_num, b200_loam_stats* stats) {
    const int64_t n = n_corner + n_surf;
    const int nbx = (int)std::min<int64_t>((n + loam::ACC_THREADS - 1) / loam::ACC_THREADS, loam::MAXB);
    CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
    int launches = 0, it = 0;
    while (it < iter_num) {
        const int batch = std::min(it == 0 ? 6 : 4, iter_num - it);  // typical scans converge in 5-6 iterations: one poll
        for (int b = 0; b < batch; ++b) {
            loam_search(h, n_corner, n_surf);
            loam::k_loam_accum<<<nbx, loam::ACC_THREADS, 0, h->stream>>>(h->d_pts.p, h->d_nb.p, h->d_cnt.p, (int)n_corner, (int)n, h->d_ctl, h->d_partials.p, 0,
                                                                          nullptr, nullptr);
            LAUNCH_COUNT(1);
            launches += 3;
        }
        it += batch;
        CUDA_TRY(cudaMemcpyAsync(h->h_ctl.p, h->d_ctl, sizeof(loam::Ctl), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        if (h->h_ctl.p->done) break;
    }
    CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    CUDA_TRY(cudaGetLastError());
    cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1);
    h->last_launches = launches;
    const loam::Ctl& c = *h->h_ctl.p;
    memcpy(t6, c.t6, 6 * sizeof(float));
    if (stats) {
        stats->iters = c.iter; stats->n_sel = c.n_sel; stats->converged = c.converged; stats->degenerate = c.degenerate; stats->gpu_ms = h->last_ms;
        memcpy(stats->AtA_first, c.AtA_first, sizeof c.AtA_first);
    }
    return c.converged ? B200_OK : B200_NOT_CONVERGED;
}

extern "C" {
/* one cornerOptimization + surfOptimization pass at t6 (parity probe): flags[n_corner + n_surf], coeff4[(n_corner + n_surf) * 4];
 * *n_sel = number of selected features */
int32_t b200_loam_features(b200_loam* h, const float* corner_xyz, int64_t n_corner, int64_t stride_corner, const float* surf_xyz, int64_t n_surf,
                           int64_t stride_surf, const float* t6, uint8_t* flags, float* coeff4, int32_t* n_sel) {
    if (!h || !t6 || !flags || !coeff4 || n_corner < 0 || n_surf < 0 || n_corner + n_surf < 1) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (!h->have_maps) B200_FAIL(B200_ERR_ARG, "no feature maps set");
    CUDA_SET_DEVICE(h->device);
    int32_t rc = loam_stage(h, corner_xyz, n_corner, stride_corner, surf_xyz, n_surf, stride_surf, t6, 1);
    if (rc) return rc;
    const int64_t n = n_corner + n_surf;
    CUDA_TRY(h->d_flags.reserve(n)); CUDA_TRY(h->d_coeff.reserve(n));
    const int nbx = (int)std::min<int64_t>((n + loam::ACC_THREADS - 1) / loam::ACC_THREADS, loam::MAXB);
    loam_search(h, n_corner, n_surf);
    loam::k_loam_accum<<<nbx, loam::ACC_THREADS, 0, h->stream>>>(h->d_pts.p, h->d_nb.p, h->d_cnt.p, (int)n_corner, (int)n, h->d_ctl, h->d_partials.p, 1,
                                                                  h->d_flags.p, h->d_coeff.p);
    LAUNCH_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(flags, h->d_flags.p, n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaMemcpyAsync(coeff4, h->d_coeff.p, n * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    CUDA_TRY(cudaGetLastError());
    if (n_sel) { int s = 0; for (int64_t i = 0; i < n; ++i) s += flags[i]; *n_sel = s; }
    return B200_OK;
}

/* extractSurroundingKeyFrames from the store + setInputCloud of both maps, the points staying on the device.  Host syncs: the
 * keyframe list, the per-segment min / max, the run ranges (loop::surrounding), then one insert counter read per map. */
int32_t b200_loam_set_map_from_keyframes(b200_loam* h, b200_keyframes* store, int64_t cur, double time_cur, const b200_surround_params* prm,
                                         b200_surround_info* info) {
    if (!h || !store) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (const int32_t rc = loop::check_surround(store, cur, time_cur, prm)) return rc;
    if (loop::device_of(store) != h->device) B200_FAIL(B200_ERR_ARG, "keyframe store and LOAM handle are on different devices");
    CUDA_SET_DEVICE(h->device);
    cudaStream_t ss = loop::stream_of(store);
    CUDA_TRY(cudaEventRecord(h->ev0, ss));
    loop::Surround sr;
    if (const int32_t rc = loop::surrounding(store, cur, time_cur, *prm, sr)) return rc;
    const int64_t nc = sr.sm.count[0], ns = sr.sm.count[1];
    if ((uint64_t)nc > h->corner.prm.max_points || (uint64_t)ns > h->surf.prm.max_points)
        B200_FAIL(B200_ERR_CAPACITY, "feature map larger than max_map_points of b200_loam_create");
    // the centroids are written on the store's stream; both maps read them on their own streams
    CUDA_TRY(cudaEventRecord(h->ev_map, ss));
    CUDA_TRY(cudaStreamWaitEvent(h->corner.stream, h->ev_map, 0));
    CUDA_TRY(cudaStreamWaitEvent(h->surf.stream, h->ev_map, 0));
    int32_t rc = h->corner.clear();
    if (rc == B200_OK) rc = h->surf.clear();
    if (rc == B200_OK && nc) rc = h->corner.insert_device(sr.sm.pts + sr.sm.first[0], nc);
    if (rc == B200_OK && ns) rc = h->surf.insert_device(sr.sm.pts + sr.sm.first[1], ns);
    if (rc != B200_OK) return rc;
    CUDA_TRY(cudaEventRecord(h->ev_map, h->surf.stream));
    CUDA_TRY(cudaStreamWaitEvent(h->corner.stream, h->ev_map, 0));
    CUDA_TRY(cudaEventRecord(h->ev1, h->corner.stream));
    CUDA_TRY(cudaStreamSynchronize(h->corner.stream));
    CUDA_TRY(cudaStreamSynchronize(h->surf.stream));
    h->have_maps = true;
    if (info) {
        info->n_list = sr.n_list;
        info->n_kept = (int64_t)sr.keys.size();
        info->n_corner_raw = sr.raw[0];
        info->n_surf_raw = sr.raw[1];
        info->n_corner = nc;
        info->n_surf = ns;
        info->gpu_ms = 0.f;
        cudaEventElapsedTime(&info->gpu_ms, h->ev0, h->ev1);
        info->pad = 0;
    }
    return B200_OK;
}

}  // extern "C"
