// b200reg — NDT registration: device data layout and per-(point, voxel) arithmetic.
//
// Replaces (paths relative to the reference's src/pointcloud_match/ndt_omp/include/pclomp):
//   VoxelGridCovariance::applyFilter / Leaf            voxel_grid_covariance_omp_impl.hpp:49-370
//   getNeighborhoodAtPoint{,7,1}                       voxel_grid_covariance_omp_impl.hpp:374-442
//   computeAngleDerivatives                            ndt_omp_impl.hpp:271-366
//   computePointDerivatives + updateDerivatives        ndt_omp_impl.hpp:370-409,452-495   (float path)
//   computePointDerivatives(double) + updateHessian    ndt_omp_impl.hpp:413-449,565-590   (double path)
//   calculateScore                                     ndt_omp_impl.hpp:836-880
//
// Layout in HBM
//   cell2leaf[div_x*div_y*div_z] int32   dense voxel grid over the target's bounding box (the reference's own
//                                        leaf id = (ijk - min_b) . divb_mul indexes it directly): leaf slot or -1.
//                                        One 4-byte load resolves a neighbourhood probe; 10M-pt / 1 m maps need a few MB.
//   leafF[L]  64 B   {double mean[3]; float icov[9]; pad}   what the float derivative path reads (4 x 16-byte loads)
//   leafD[L]  96 B   {double mean[3]; double icov[9]}        what computeHessian reads (6 x 16-byte loads)
//   score store, 72 B per leaf in three arrays (what calculateScore reads: two 32-byte loads and one 8-byte load)
//     sA[L]   32 B   {mean_x, mean_y, mean_z, icov00}
//     sB[L]   32 B   {icov01 + icov10, icov02 + icov20, icov11, icov12 + icov21}
//     sC[L]    8 B   icov22
//   fp32 screen store, 36 B per leaf, the same numbers narrowed (what the relocalization screen reads; 8 leaves per line)
//     fA[L]   16 B   {m_x, m_y, m_z, icov00}      m = fp32(mean - o), o = corner of the leaf's cell (cell_origin)
//     fB[L]   16 B   {s01, s02, icov11, s12}
//     fC[L]    4 B   icov22
//   cov[L] 72 B, npts[L], ids[L], valid[L]                   only read back by b200_ndt_leaves
// The TU is compiled with -fmad=false: every fp32/fp64 operation below is individually rounded, in the
// evaluation order of the reference C++ (Eigen fixed-size products accumulate k = 0..3 left to right).
#pragma once
#include "common.cuh"
#include <math_constants.h>

namespace b200 {
namespace ndt {

struct __align__(16) LeafF {
    double mean[3];
    float icov[9];
    float pad;
};
struct __align__(16) LeafD {
    double mean[3];
    double icov[9];
};
static_assert(sizeof(LeafF) == 64 && sizeof(LeafD) == 96, "leaf records are read with 16-byte loads");

// Score store of one leaf (built by k_ndt_score_store).  Split into arrays so that the same 32-byte piece of four
// consecutive leaves shares a 128-byte line: a warp's load of neighbouring leaves touches fewer lines than the 96-byte
// records, whose pieces of neighbouring leaves almost never share one.
struct __align__(32) Dbl4 {
    double x, y, z, w;
};
// One 256-bit load (sm_100: ld.global.nc.v4.f64 -> LDG.E.256): the L1 wavefronts of a warp request go with the number of
// load instructions and the distinct lines they touch.  Dbl4 arrays are cudaMalloc'ed, so no piece straddles a line.
__device__ __forceinline__ Dbl4 load_dbl4_256(const Dbl4* p) {
    Dbl4 r;
    asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=d"(r.w) : "l"(p));
    return r;
}

struct AngleTables {   // computeAngleDerivatives: j_ang_a_..h_ / h_ang_a2_..f3_ (double) and j_ang / h_ang (float)
    double jd[8][3];
    double hd[15][3];
    float jf[8][3];
    float hf[15][3];
};

struct View {
    const float4* src;
    int n_src;
    const int* cell2leaf;
    const float* centroid;  // [leaves][3] fp32 centroids (leaf.centroid, the cloud the reference's kd-tree indexes); KDTREE mode only
    int kdtree;        // neighbourhood = radiusSearch(point, resolution) over the centroids (ndt_omp_impl.hpp:217-219)
    float kd_r2;       // its squared radius as FLANN sees it: (float)(resolution * resolution)
    const int* nbr7;   // [cells][8]: leaf slot (or -1) of the DIRECT7 neighbourhood cells of every grid cell, [7] = how many exist
    const LeafF* leafF;
    const LeafD* leafD;
    const Dbl4* sA;    // score store (see the layout above); set_target builds it, the batched pairs target does not
    const Dbl4* sB;
    const double* sC;
    int min_b[3], max_b[3], mul[3];
    float leaf;
    int nst;   // 1, 7, 27
    double d1, d2, d3;
};

// Corner of grid cell i along one axis, as the screen store and the screen kernel both compute it (same bits on both sides)
__device__ __forceinline__ float cell_origin(int i, float leaf) { return __fmul_rn((float)i, leaf); }

// DIRECT7 order (voxel_grid_covariance_omp_impl.hpp:423-430); DIRECT26 = pcl::getAllNeighborCellIndices()
// (27 cells, x slowest); DIRECT1 = the cell itself.
__device__ __forceinline__ void nbr_offset(int nst, int s, int& dx, int& dy, int& dz) {
    if (nst == 27) {
        dx = s / 9 - 1;
        dy = (s / 3) % 3 - 1;
        dz = s % 3 - 1;
    } else {
        // s: 0 c, 1 +x, 2 -x, 3 +y, 4 -y, 5 +z, 6 -z
        const int a = (s + 1) >> 1;               // 0,1,1,2,2,3,3
        const int sg = (s & 1) ? 1 : -1;          // odd -> +, even -> -
        dx = (a == 1) ? sg : 0;
        dy = (a == 2) ? sg : 0;
        dz = (a == 3) ? sg : 0;
    }
}

// leaf slot of the s-th neighbourhood cell of the point (tx,ty,tz), or -1 (getNeighborhoodAtPoint, :374-404)
__device__ __forceinline__ int nbr_leaf(const View& v, float tx, float ty, float tz, int s) {
    const int ix = (int)floorf(tx / v.leaf), iy = (int)floorf(ty / v.leaf), iz = (int)floorf(tz / v.leaf);
    int dx, dy, dz;
    nbr_offset(v.nst, s, dx, dy, dz);
    if (!(v.min_b[0] - ix <= dx && v.max_b[0] - ix >= dx && v.min_b[1] - iy <= dy && v.max_b[1] - iy >= dy &&
          v.min_b[2] - iz <= dz && v.max_b[2] - iz >= dz))
        return -1;
    const int id = (ix + dx - v.min_b[0]) * v.mul[0] + (iy + dy - v.min_b[1]) * v.mul[1] + (iz + dz - v.min_b[2]) * v.mul[2];
    int lf = __ldg(v.cell2leaf + id);
    if (v.kdtree && lf >= 0) {
        // VoxelGridCovariance::radiusSearch (voxel_grid_covariance_omp.h:477-505): the kd-tree holds the fp32 centroids of the
        // leaves; FLANN's L2_Simple adds the squared differences in x, y, z order in fp32 and its radius result set keeps
        // dist < radius^2.  A centroid lies inside its own cell, so every hit is in the 27-cell block around the point.
        const float cx = __ldg(v.centroid + 3 * lf), cy = __ldg(v.centroid + 3 * lf + 1), cz = __ldg(v.centroid + 3 * lf + 2);
        const float ax = tx - cx, ay = ty - cy, az = tz - cz;
        const float d = (ax * ax + ay * ay) + az * az;
        if (!(d < v.kd_r2)) lf = -1;
    }
    return lf;
}

// pcl::transformPointCloud (PCL 1.7/1.8 scalar form) with a row-major 3x4 float matrix
__device__ __forceinline__ void xform(const float* M, float x, float y, float z, float& tx, float& ty, float& tz) {
    tx = ((M[0] * x + M[1] * y) + M[2] * z) + M[3];
    ty = ((M[4] * x + M[5] * y) + M[6] * z) + M[7];
    tz = ((M[8] * x + M[9] * y) + M[10] * z) + M[11];
}

// Translation * AngleAxis(x) * AngleAxis(y) * AngleAxis(z) in float (ndt_omp_impl.hpp:129,749-753); float sin/cos
// evaluated as the correctly rounded value (double evaluation, narrowed)
// The sines / cosines of a requested pose: cf / sf = correctly rounded floats of the float-narrowed angles (pose_matrix),
// cd / sd = doubles with computeAngleDerivatives' small-angle snap (angle_tables).  Six independent evaluations: the
// evaluation kernel computes them on six lanes instead of one after the other.
struct Trig {
    double cd[3], sd[3];
    float cf[3], sf[3];
};
__device__ inline void trig_of_angle(const double* p, int which /*0..5*/, Trig& t) {
    const int a = which % 3;
    if (which < 3) {
        if (fabs(p[3 + a]) < 10e-5) { t.cd[a] = 1.0; t.sd[a] = 0.0; }
        else { t.cd[a] = cos(p[3 + a]); t.sd[a] = sin(p[3 + a]); }
    } else {
        const float r = (float)p[3 + a];
        t.cf[a] = (float)cos((double)r);
        t.sf[a] = (float)sin((double)r);
    }
}
__device__ inline void pose_matrix_core(const double* p, float cx, float sx, float cy, float sy, float cz, float sz, float* M);
__device__ inline void pose_matrix(const double* p, float* M /*row-major 4x4*/) {
    const float rx = (float)p[3], ry = (float)p[4], rz = (float)p[5];
    const float cx = (float)cos((double)rx), sx = (float)sin((double)rx), cy = (float)cos((double)ry), sy = (float)sin((double)ry),
                cz = (float)cos((double)rz), sz = (float)sin((double)rz);
    pose_matrix_core(p, cx, sx, cy, sy, cz, sz, M);
}
__device__ inline void pose_matrix_core(const double* p, float cx, float sx, float cy, float sy, float cz, float sz, float* M) {
    const float Rx[9] = {1, 0, 0, 0, cx, -sx, 0, sx, cx};
    const float Ry[9] = {cy, 0, sy, 0, 1, 0, -sy, 0, cy};
    const float Rz[9] = {cz, -sz, 0, sz, cz, 0, 0, 0, 1};
    float T1[9], T2[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) T1[i * 3 + j] = (Rx[i * 3] * Ry[j] + Rx[i * 3 + 1] * Ry[3 + j]) + Rx[i * 3 + 2] * Ry[6 + j];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) T2[i * 3 + j] = (T1[i * 3] * Rz[j] + T1[i * 3 + 1] * Rz[3 + j]) + T1[i * 3 + 2] * Rz[6 + j];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) M[i * 4 + j] = T2[i * 3 + j];
        M[i * 4 + 3] = (float)p[i];
    }
    M[12] = M[13] = M[14] = 0.0f;
    M[15] = 1.0f;
}

// Matrix3f::eulerAngles(0,1,2) (Eigen 3.3 EulerAngles.h); R row-major 3x3.  atan2/sin/cos as correctly
// rounded floats.
__device__ inline void euler_012(const float* R, float* res) {
    const float pi = 3.14159265358979323846f;
    auto C = [&](int r, int c) { return R[r * 3 + c]; };
    res[0] = (float)atan2((double)C(1, 2), (double)C(2, 2));
    const float c2 = sqrtf(C(0, 0) * C(0, 0) + C(0, 1) * C(0, 1));
    if (res[0] > 0.0f) {
        res[0] -= pi;
        res[1] = (float)atan2((double)-C(0, 2), (double)-c2);
    } else {
        res[1] = (float)atan2((double)-C(0, 2), (double)c2);
    }
    const float s1 = (float)sin((double)res[0]), c1 = (float)cos((double)res[0]);
    res[2] = (float)atan2((double)(s1 * C(2, 0) - c1 * C(1, 0)), (double)(c1 * C(1, 1) - s1 * C(2, 1)));
    res[0] = -res[0];
    res[1] = -res[1];
    res[2] = -res[2];
}

// computeAngleDerivatives (ndt_omp_impl.hpp:271-366), including the small-angle snap and the float
// table's +sy entry in row d1 (:354) where the double table has -sy (:332).
__device__ inline void angle_tables_core(double cx, double sx, double cy, double sy, double cz, double sz, AngleTables& t);
__device__ inline void angle_tables(const double* p, AngleTables& t) {
    double cx, cy, cz, sx, sy, sz;
    if (fabs(p[3]) < 10e-5) { cx = 1.0; sx = 0.0; } else { cx = cos(p[3]); sx = sin(p[3]); }
    if (fabs(p[4]) < 10e-5) { cy = 1.0; sy = 0.0; } else { cy = cos(p[4]); sy = sin(p[4]); }
    if (fabs(p[5]) < 10e-5) { cz = 1.0; sz = 0.0; } else { cz = cos(p[5]); sz = sin(p[5]); }
    angle_tables_core(cx, sx, cy, sy, cz, sz, t);
}
__device__ inline void angle_tables_core(double cx, double sx, double cy, double sy, double cz, double sz, AngleTables& t) {
    const double J[8][3] = {{(-sx * sz + cx * sy * cz), (-sx * cz - cx * sy * sz), (-cx * cy)},
                            {(cx * sz + sx * sy * cz), (cx * cz - sx * sy * sz), (-sx * cy)},
                            {(-sy * cz), sy * sz, cy},
                            {sx * cy * cz, (-sx * cy * sz), sx * sy},
                            {(-cx * cy * cz), cx * cy * sz, (-cx * sy)},
                            {(-cy * sz), (-cy * cz), 0},
                            {(cx * cz - sx * sy * sz), (-cx * sz - sx * sy * cz), 0},
                            {(sx * cz + cx * sy * sz), (cx * sy * cz - sx * sz), 0}};
    const double Hh[15][3] = {{(-cx * sz - sx * sy * cz), (-cx * cz + sx * sy * sz), sx * cy},
                              {(-sx * sz + cx * sy * cz), (-cx * sy * sz - sx * cz), (-cx * cy)},
                              {(cx * cy * cz), (-cx * cy * sz), (cx * sy)},
                              {(sx * cy * cz), (-sx * cy * sz), (sx * sy)},
                              {(-sx * cz - cx * sy * sz), (sx * sz - cx * sy * cz), 0},
                              {(cx * cz - sx * sy * sz), (-sx * sy * cz - cx * sz), 0},
                              {(-cy * cz), (cy * sz), (-sy)},
                              {(-sx * sy * cz), (sx * sy * sz), (sx * cy)},
                              {(cx * sy * cz), (-cx * sy * sz), (-cx * cy)},
                              {(sy * sz), (sy * cz), 0},
                              {(-sx * cy * sz), (-sx * cy * cz), 0},
                              {(cx * cy * sz), (cx * cy * cz), 0},
                              {(-cy * cz), (cy * sz), 0},
                              {(-cx * sz - sx * sy * cz), (-cx * cz + sx * sy * sz), 0},
                              {(-sx * sz + cx * sy * cz), (-cx * sy * sz - sx * cz), 0}};
    for (int r = 0; r < 8; ++r)
        for (int c = 0; c < 3; ++c) { t.jd[r][c] = J[r][c]; t.jf[r][c] = (float)J[r][c]; }
    for (int r = 0; r < 15; ++r)
        for (int c = 0; c < 3; ++c) { t.hd[r][c] = Hh[r][c]; t.hf[r][c] = (float)Hh[r][c]; }
    t.hf[6][2] = (float)sy;
}

constexpr int NACC = 43;  // score, g[6], H[36]

// Float path for one (point, voxel) pair: computePointDerivatives (ndt_omp_impl.hpp:370-409) followed by
// updateDerivatives (:452-495).  x = source point, (tx,ty,tz) = transformed point, acc += {score, g, H}.
// Products with the structural zeros / ones of point_gradient_ and point_hessian_ are exact and elided.
__device__ __forceinline__ void deriv_pair_f(const View& v, const AngleTables& t, const LeafF& L, float x0, float x1, float x2,
                                             float tx, float ty, float tz, bool hess, double (&acc)[NACC]) {
    const float xt0 = (float)((double)tx - L.mean[0]), xt1 = (float)((double)ty - L.mean[1]), xt2 = (float)((double)tz - L.mean[2]);
    const float* ci = L.icov;  // row-major 3x3 (c_inv.cast<float>())
    float xc[3];               // x_trans4 * c_inv4
#pragma unroll
    for (int c = 0; c < 3; ++c) xc[c] = (xt0 * ci[c] + xt1 * ci[3 + c]) + xt2 * ci[6 + c];
    const float q = (xt0 * xc[0] + xt1 * xc[1]) + xt2 * xc[2];
    const float gd2 = (float)v.d2;
    const float arg = -gd2 * q * 0.5f;
    float e = (float)exp((double)arg);
    const float score_inc = (float)(-v.d1 * (double)e);
    e = gd2 * e;
    if (e > 1 || e < 0 || e != e) return;
    e = (float)((double)e * v.d1);
    float xj[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) xj[r] = (t.jf[r][0] * x0 + t.jf[r][1] * x1) + t.jf[r][2] * x2;
    // c_inv4 * point_gradient4: columns 0..2 are c_inv itself; 3: (.,xj0,xj1); 4: (xj2,xj3,xj4); 5: (xj5,xj6,xj7)
    float cg[3][6];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        cg[r][0] = ci[r * 3];
        cg[r][1] = ci[r * 3 + 1];
        cg[r][2] = ci[r * 3 + 2];
        cg[r][3] = (ci[r * 3] * 0.0f + ci[r * 3 + 1] * xj[0]) + ci[r * 3 + 2] * xj[1];
        cg[r][4] = (ci[r * 3] * xj[2] + ci[r * 3 + 1] * xj[3]) + ci[r * 3 + 2] * xj[4];
        cg[r][5] = (ci[r * 3] * xj[5] + ci[r * 3 + 1] * xj[6]) + ci[r * 3 + 2] * xj[7];
    }
    float xg[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) xg[c] = (xt0 * cg[0][c] + xt1 * cg[1][c]) + xt2 * cg[2][c];
    acc[0] += (double)score_inc;
#pragma unroll
    for (int c = 0; c < 6; ++c) acc[1 + c] += (double)(e * xg[c]);
    if (!hess) return;
    float xh[15];
#pragma unroll
    for (int r = 0; r < 15; ++r) xh[r] = (t.hf[r][0] * x0 + t.hf[r][1] * x1) + t.hf[r][2] * x2;
    // point_gradient4 rows 0..2 as columns: pgc[k][r] = point_gradient(k, r)
    const float pg3[3] = {0.0f, xj[0], xj[1]}, pg4[3] = {xj[2], xj[3], xj[4]}, pg5[3] = {xj[5], xj[6], xj[7]};
    // blocks of point_hessian_: a = (0,xh0,xh1) b = (0,xh2,xh3) c = (0,xh4,xh5) d = (xh6,xh7,xh8) e = (xh9..11) f = (xh12..14)
    const float ha[3] = {0.0f, xh[0], xh[1]}, hb[3] = {0.0f, xh[2], xh[3]}, hc[3] = {0.0f, xh[4], xh[5]};
    const float hd[3] = {xh[6], xh[7], xh[8]}, he[3] = {xh[9], xh[10], xh[11]}, hf[3] = {xh[12], xh[13], xh[14]};
    auto dot_xc = [&](const float* h) { return (xc[0] * h[0] + xc[1] * h[1]) + xc[2] * h[2]; };
    // x_trans4_x_c_inv4 * point_hessian_.block<4,6>(i*4, 0): only i, j >= 3 are non-zero
    const float xa = dot_xc(ha), xb = dot_xc(hb), xcc = dot_xc(hc), xd = dot_xc(hd), xe = dot_xc(he), xf = dot_xc(hf);
    const float xh6[3][3] = {{xa, xb, xcc}, {xb, xd, xe}, {xcc, xe, xf}};
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            // gg(j, i) = point_gradient4.col(j) . (c_inv4 * point_gradient4).col(i)
            float gg;
            if (j < 3) gg = cg[j][i];
            else {
                const float* pc = (j == 3) ? pg3 : (j == 4) ? pg4 : pg5;
                gg = (pc[0] * cg[0][i] + pc[1] * cg[1][i]) + pc[2] * cg[2][i];
            }
            const float hx = (i >= 3 && j >= 3) ? xh6[i - 3][j - 3] : 0.0f;
            acc[7 + i * 6 + j] += (double)(e * ((-gd2 * xg[i] * xg[j] + hx) + gg));
        }
    }
}

// Double path for one (point, voxel) pair: computePointDerivatives(double) (:413-449) + updateHessian (:565-590)
__device__ __forceinline__ void hessian_pair_d(const View& v, const AngleTables& t, const LeafD& L, float fx0, float fx1, float fx2,
                                               float tx, float ty, float tz, double (&H)[36]) {
    const double x[3] = {fx0, fx1, fx2};
    const double xt[3] = {(double)tx - L.mean[0], (double)ty - L.mean[1], (double)tz - L.mean[2]};
    const double* ci = L.icov;
    auto dotx = [&](const double* r) { return x[0] * r[0] + x[1] * r[1] + x[2] * r[2]; };
    double pg[3][6] = {{1, 0, 0, 0, 0, 0}, {0, 1, 0, 0, 0, 0}, {0, 0, 1, 0, 0, 0}};
    pg[1][3] = dotx(t.jd[0]); pg[2][3] = dotx(t.jd[1]);
    pg[0][4] = dotx(t.jd[2]); pg[1][4] = dotx(t.jd[3]); pg[2][4] = dotx(t.jd[4]);
    pg[0][5] = dotx(t.jd[5]); pg[1][5] = dotx(t.jd[6]); pg[2][5] = dotx(t.jd[7]);
    const double a[3] = {0, dotx(t.hd[0]), dotx(t.hd[1])}, b[3] = {0, dotx(t.hd[2]), dotx(t.hd[3])}, c[3] = {0, dotx(t.hd[4]), dotx(t.hd[5])};
    const double d[3] = {dotx(t.hd[6]), dotx(t.hd[7]), dotx(t.hd[8])}, e[3] = {dotx(t.hd[9]), dotx(t.hd[10]), dotx(t.hd[11])},
                 f[3] = {dotx(t.hd[12]), dotx(t.hd[13]), dotx(t.hd[14])};
    const double zero3[3] = {0, 0, 0};
    auto mv = [&](const double* vv, double* r) {
        for (int k = 0; k < 3; ++k) r[k] = ci[k * 3] * vv[0] + ci[k * 3 + 1] * vv[1] + ci[k * 3 + 2] * vv[2];
    };
    double cx[3];
    mv(xt, cx);
    double e_x = v.d2 * exp(-v.d2 * (xt[0] * cx[0] + xt[1] * cx[1] + xt[2] * cx[2]) / 2);
    if (e_x > 1 || e_x < 0 || e_x != e_x) return;
    e_x *= v.d1;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const double col_i[3] = {pg[0][i], pg[1][i], pg[2][i]};
        double cdi[3];
        mv(col_i, cdi);
        const double t1 = xt[0] * cdi[0] + xt[1] * cdi[1] + xt[2] * cdi[2];
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const double col_j[3] = {pg[0][j], pg[1][j], pg[2][j]};
            const double* hij = zero3;
            if (i >= 3 && j >= 3) {
                const int k = (i - 3) * 3 + (j - 3);
                hij = (k == 0) ? a : (k == 1 || k == 3) ? b : (k == 2 || k == 6) ? c : (k == 4) ? d : (k == 5 || k == 7) ? e : f;
            }
            double cj[3], chij[3];
            mv(col_j, cj);
            mv(hij, chij);
            const double t2 = xt[0] * cj[0] + xt[1] * cj[1] + xt[2] * cj[2];
            const double t3 = xt[0] * chij[0] + xt[1] * chij[1] + xt[2] * chij[2];
            const double t4 = col_j[0] * cdi[0] + col_j[1] * cdi[1] + col_j[2] * cdi[2];
            H[i * 6 + j] += e_x * (-v.d2 * t1 * t2 + t3 + t4);
        }
    }
}

// ------------------------------------------------------------------ small dense helpers (leaf finalisation, Newton step)
// 3x3 inverse by cofactors / determinant
__device__ __forceinline__ void inverse3(const double* m, double* inv) {
    const double c00 = m[4] * m[8] - m[5] * m[7];
    const double c10 = m[5] * m[6] - m[3] * m[8];
    const double c20 = m[3] * m[7] - m[4] * m[6];
    const double det = m[0] * c00 + m[1] * c10 + m[2] * c20;
    const double id = 1.0 / det;
    inv[0] = c00 * id;
    inv[1] = (m[2] * m[7] - m[1] * m[8]) * id;
    inv[2] = (m[1] * m[5] - m[2] * m[4]) * id;
    inv[3] = c10 * id;
    inv[4] = (m[0] * m[8] - m[2] * m[6]) * id;
    inv[5] = (m[2] * m[3] - m[0] * m[5]) * id;
    inv[6] = c20 * id;
    inv[7] = (m[1] * m[6] - m[0] * m[7]) * id;
    inv[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}

// ---- Eigen decompositions the reference calls, following the Eigen sources vendored in the reference
// (pointcloud_match/fast_gicp/thirdparty/Eigen/Eigen/src/, "E/" below) operation by operation; this TU is compiled
// with -fmad=false, fp64 sqrt and division are IEEE, so the results are bit-identical to an SSE2 build of Eigen.
// JacobiRotation<double>::makeGivens, real case (E/Jacobi/Jacobi.h:231-267)
__device__ __forceinline__ void make_givens(double p, double q, double& c, double& s) {
    if (q == 0.0) {
        c = p < 0.0 ? -1.0 : 1.0;
        s = 0.0;
    } else if (p == 0.0) {
        c = 0.0;
        s = q < 0.0 ? 1.0 : -1.0;
    } else if (fabs(p) > fabs(q)) {
        const double t = q / p;
        double u = sqrt(1.0 + t * t);
        if (p < 0.0) u = -u;
        c = 1.0 / u;
        s = -t * c;
    } else {
        const double t = p / q;
        double u = sqrt(1.0 + t * t);
        if (q < 0.0) u = -u;
        s = -1.0 / u;
        c = -t * s;
    }
}
// numext::hypot, real case (Eigen 3.4 Core/MathFunctionsImpl.h positive_real_hypot; Core is absent from the snapshot)
__device__ __forceinline__ double eigen_hypot(double x, double y) {
    x = fabs(x);
    y = fabs(y);
    if (isinf(x) || isinf(y)) return CUDART_INF;
    if (isnan(x) || isnan(y)) return CUDART_NAN;
    const double p = x > y ? x : y;
    if (p == 0.0) return 0.0;
    const double qp = (y < x ? y : x) / p;
    return p * sqrt(1.0 + qp * qp);
}
// SelfAdjointEigenSolver<Matrix3d>::compute(A, ComputeEigenvectors) (vgc_impl:333): scaling E/Eigenvalues/SelfAdjointEigenSolver.h:445-449,
// 3x3 tridiagonalisation E/Eigenvalues/Tridiagonalization.h:459-503, deflation + iteration :498-550, implicit QR step with
// Wilkinson shift :823-893, ascending sort :551-567.  Reads the lower triangle of A (row-major); eigenvalues ascending in w,
// eigenvectors in the columns of V (row-major).
__device__ __noinline__ bool eigen_selfadjoint3(const double* A, double* w, double* V) {
    const double dmin = 2.2250738585072014e-308;
    double m00 = A[0], m10 = A[3], m11 = A[4], m20 = A[6], m21 = A[7], m22 = A[8];
    double scale = fabs(m00);
    scale = fmax(scale, fabs(m10)); scale = fmax(scale, fabs(m11)); scale = fmax(scale, fabs(m20));
    scale = fmax(scale, fabs(m21)); scale = fmax(scale, fabs(m22));
    if (scale == 0.0) scale = 1.0;
    m00 /= scale; m10 /= scale; m11 /= scale; m20 /= scale; m21 /= scale; m22 /= scale;
    double diag[3], sub[2], Q[3][3];
    diag[0] = m00;
    const double v1norm2 = m20 * m20;
    if (v1norm2 <= dmin) {
        diag[1] = m11; diag[2] = m22; sub[0] = m10; sub[1] = m21;
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Q[i][j] = i == j ? 1.0 : 0.0;
    } else {
        const double beta = sqrt(m10 * m10 + v1norm2);
        const double invBeta = 1.0 / beta;
        const double m01 = m10 * invBeta, m02 = m20 * invBeta;
        const double q = 2.0 * m01 * m21 + m02 * (m22 - m11);
        diag[1] = m11 + m02 * q;
        diag[2] = m22 - m02 * q;
        sub[0] = beta;
        sub[1] = m21 - m01 * q;
        Q[0][0] = 1; Q[0][1] = 0; Q[0][2] = 0;
        Q[1][0] = 0; Q[1][1] = m01; Q[1][2] = m02;
        Q[2][0] = 0; Q[2][1] = m02; Q[2][2] = -m01;
    }
    const int n = 3, maxIterations = 30;
    int end = n - 1, start = 0, iter = 0;
    const double precision_inv = 1.0 / 2.220446049250313e-16;
    while (end > 0) {
        for (int i = start; i < end; ++i) {
            if (fabs(sub[i]) < dmin) {
                sub[i] = 0.0;
            } else {
                const double scaled = precision_inv * sub[i];
                if (scaled * scaled <= (fabs(diag[i]) + fabs(diag[i + 1]))) sub[i] = 0.0;
            }
        }
        while (end > 0 && sub[end - 1] == 0.0) end--;
        if (end <= 0) break;
        iter++;
        if (iter > maxIterations * n) break;
        start = end - 1;
        while (start > 0 && sub[start - 1] != 0.0) start--;
        const double td = (diag[end - 1] - diag[end]) * 0.5;
        const double e = sub[end - 1];
        double mu = diag[end];
        if (td == 0.0) {
            mu -= fabs(e);
        } else if (e != 0.0) {
            const double e2 = e * e;
            const double h = eigen_hypot(td, e);
            if (e2 == 0.0) mu -= e / ((td + (td > 0.0 ? h : -h)) / e);
            else mu -= e2 / (td + (td > 0.0 ? h : -h));
        }
        double x = diag[start] - mu;
        double z = sub[start];
        for (int k = start; k < end && z != 0.0; ++k) {
            double c, s;
            make_givens(x, z, c, s);
            const double sdk = s * diag[k] + c * sub[k];
            const double dkp1 = s * sub[k] + c * diag[k + 1];
            diag[k] = c * (c * diag[k] - s * sub[k]) - s * (c * sub[k] - s * diag[k + 1]);
            diag[k + 1] = s * sdk + c * dkp1;
            sub[k] = c * sdk - s * dkp1;
            if (k > start) sub[k - 1] = c * sub[k - 1] - s * z;
            x = sub[k];
            if (k < end - 1) {
                z = -s * sub[k + 1];
                sub[k + 1] = c * sub[k + 1];
            }
            if (!(c == 1.0 && s == 0.0)) {  // q.applyOnTheRight(k, k+1, rot) (E/Jacobi/Jacobi.h:312-319, 331-332)
                for (int i = 0; i < 3; ++i) {
                    const double xi = Q[i][k], yi = Q[i][k + 1];
                    Q[i][k] = c * xi - s * yi;
                    Q[i][k + 1] = s * xi + c * yi;
                }
            }
        }
    }
    const bool ok = iter <= maxIterations * n;
    if (ok) {
        for (int i = 0; i < n - 1; ++i) {
            int k = 0;
            for (int j = 1; j < n - i; ++j)
                if (diag[i + j] < diag[i + k]) k = j;
            if (k > 0) {
                const double t = diag[i]; diag[i] = diag[k + i]; diag[k + i] = t;
                for (int r = 0; r < 3; ++r) { const double tv = Q[r][i]; Q[r][i] = Q[r][k + i]; Q[r][k + i] = tv; }
            }
        }
    }
    for (int i = 0; i < 3; ++i) w[i] = diag[i] * scale;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) V[i * 3 + j] = Q[i][j];
    return ok;
}

// Cyclic Jacobi eigen-decomposition of a symmetric NxN matrix (row-major, destroyed): eigenvalues ascending in w,
// eigenvectors in the columns of V.  Fully unrolled so A and V stay in registers.
template <int N>
__device__ __forceinline__ void jacobi_eig(double (&A)[N * N], double (&w)[N], double (&V)[N * N]) {
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) V[i * N + j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0, diag = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            diag += A[i * N + i] * A[i * N + i];
#pragma unroll
            for (int j = i + 1; j < N; ++j) off += A[i * N + j] * A[i * N + j];
        }
        if (off <= 1e-300 || off <= 1e-34 * diag) break;
#pragma unroll
        for (int p = 0; p < N - 1; ++p)
#pragma unroll
            for (int q = p + 1; q < N; ++q) {
                const double apq = A[p * N + q];
                if (apq != 0.0) {
                    const double theta = (A[q * N + q] - A[p * N + p]) / (2.0 * apq);
                    const double tt = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                    const double c = 1.0 / sqrt(tt * tt + 1.0), s = tt * c;
#pragma unroll
                    for (int k = 0; k < N; ++k) {
                        const double akp = A[k * N + p], akq = A[k * N + q];
                        A[k * N + p] = c * akp - s * akq;
                        A[k * N + q] = s * akp + c * akq;
                    }
#pragma unroll
                    for (int k = 0; k < N; ++k) {
                        const double apk = A[p * N + k], aqk = A[q * N + k];
                        A[p * N + k] = c * apk - s * aqk;
                        A[q * N + k] = s * apk + c * aqk;
                    }
#pragma unroll
                    for (int k = 0; k < N; ++k) {
                        const double vkp = V[k * N + p], vkq = V[k * N + q];
                        V[k * N + p] = c * vkp - s * vkq;
                        V[k * N + q] = s * vkp + c * vkq;
                    }
                }
            }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) w[i] = A[i * N + i];
#pragma unroll
    for (int i = 0; i < N - 1; ++i) {  // ascending selection sort; columns of V follow
        int m = i;
#pragma unroll
        for (int j = i + 1; j < N; ++j)
            if (w[j] < w[m]) m = j;
#pragma unroll
        for (int j = i + 1; j < N; ++j) {
            if (m == j) {
                const double tw = w[i]; w[i] = w[j]; w[j] = tw;
#pragma unroll
                for (int k = 0; k < N; ++k) { const double tv = V[k * N + i]; V[k * N + i] = V[k * N + j]; V[k * N + j] = tv; }
            }
        }
    }
}

}  // namespace ndt
}  // namespace b200
