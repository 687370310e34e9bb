// metrics.cu -- pose-accuracy metrics of the reference's Evaluator (lib/utils/evaluation_utils.py:54-141) and the
// nearest-neighbour index search it calls (lib/utils/extend_utils/src/nearest_neighborhood.cu:48-117).
//
// Nearest neighbour.  The index must equal the reference kernel's bit for bit, so the distance is the reference's
// rounding sequence as nvcc 12.9 compiles it for sm_100a (read off its SASS, DESIGN.md §2):
//     d = ref - que (one FADD per axis);  2-D: fma(dx,dx, dy*dy);  3-D: fma(dz,dz, fma(dx,dx, dy*dy))
// and its selection rule: start at (FLT_MAX, 0), replace only on a strict `dist < min_dist` in increasing reference
// index.  So NaN and +inf are never chosen, the lowest index wins a tie, and a query with no finite distance gets 0.
// Layout: a CTA is 8 warps; lane = query (Q queries per lane in registers), warp = a slice of the reference set.  A
// tile of reference points is staged in shared memory and every warp scans its slice of the tile in increasing
// index (a broadcast read: all lanes read the same point).  The 8 per-slice winners are combined as the 64-bit key
// (float_bits(dist) << 32 | idx): dist is >= 0 or NaN, and the slices' winners are < FLT_MAX or the untouched
// (FLT_MAX, 0), so the smallest key is the reference's answer, ties to the lowest index included.  No workspace,
// no atomics: the result does not depend on scheduling.
//
// Metrics.  fp64.  One CTA per image sums the per-point distances in a fixed order (a strided per-thread sum, then
// a fixed shared-memory tree), so two runs give the same bits.  The clouds keep the reference's dtypes: numpy
// computes `model @ R.T + t` in float32 when the pose is float32 (the ground truth, as the data loader yields it),
// so with the PVNET_METRICS_*_F32 flags that cloud is computed in float32 in numpy's order (transform below).
#include "common.cuh"

#include <cfloat>

namespace {

constexpr int NN_WARPS = 8;
constexpr int NN_TILE = 1024;  // reference points staged per tile (float4 each: 16 KB)

template <int DIM>
__device__ __forceinline__ float nn_dist(float4 r, float qx, float qy, float qz)
{
    const float dx = __fadd_rn(r.x, -qx);
    const float dy = __fadd_rn(r.y, -qy);
    float d = __fmaf_rn(dx, dx, __fmul_rn(dy, dy));
    if (DIM == 3) {
        const float dz = __fadd_rn(r.z, -qz);
        d = __fmaf_rn(dz, dz, d);
    }
    return d;
}

template <int DIM, int Q>
__global__ void __launch_bounds__(32 * NN_WARPS) k_nearest_point_idx(const float *__restrict__ ref,
                                                                       const float *__restrict__ que,
                                                                       int32_t *__restrict__ idxs, int pn1, int pn2,
                                                                       int exclude_self)
{
    __shared__ float4 tile[NN_TILE];
    __shared__ unsigned long long keys[NN_WARPS][32 * Q];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long bi = blockIdx.y;
    const float *rb = ref + bi * (long long)pn1 * DIM;
    const float *qb = que + bi * (long long)pn2 * DIM;
    const int q0 = blockIdx.x * (32 * Q);

    float qx[Q], qy[Q], qz[Q], best[Q];
    int qi[Q], bidx[Q];
#pragma unroll
    for (int k = 0; k < Q; ++k) {
        qi[k] = q0 + k * 32 + lane;
        const int j = qi[k] < pn2 ? qi[k] : pn2 - 1;
        qx[k] = qb[(long long)j * DIM];
        qy[k] = qb[(long long)j * DIM + 1];
        qz[k] = DIM == 3 ? qb[(long long)j * DIM + 2] : 0.f;
        best[k] = FLT_MAX;
        bidx[k] = 0;
    }

    constexpr int SLICE = NN_TILE / NN_WARPS;
    for (int t0 = 0; t0 < pn1; t0 += NN_TILE) {
        const int n = min(NN_TILE, pn1 - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const float *p = rb + (long long)(t0 + i) * DIM;
            tile[i] = make_float4(p[0], p[1], DIM == 3 ? p[2] : 0.f, 0.f);
        }
        __syncthreads();
        const int s0 = warp * SLICE, s1 = min(s0 + SLICE, n);
        for (int i = s0; i < s1; ++i) {
            const float4 r = tile[i];
            const int gi = t0 + i;
#pragma unroll
            for (int k = 0; k < Q; ++k) {
                const float d = nn_dist<DIM>(r, qx[k], qy[k], qz[k]);
                if (d < best[k] && !(exclude_self && gi == qi[k])) {
                    best[k] = d;
                    bidx[k] = gi;
                }
            }
        }
    }

#pragma unroll
    for (int k = 0; k < Q; ++k)
        keys[warp][k * 32 + lane] =
            ((unsigned long long)__float_as_uint(best[k]) << 32) | (unsigned)bidx[k];
    __syncthreads();
    for (int j = threadIdx.x; j < 32 * Q; j += blockDim.x) {
        unsigned long long m = keys[0][j];
#pragma unroll
        for (int w = 1; w < NN_WARPS; ++w) m = min(m, keys[w][j]);
        const int q = q0 + j;
        if (q < pn2) idxs[bi * pn2 + q] = (int32_t)(unsigned)(m & 0xffffffffull);
    }
}

// Four queries per lane once there are enough queries to give every SM a few CTAs; one otherwise.
int launch_nearest(const float *ref, const float *que, int32_t *idxs, int b, int pn1, int pn2, int dim,
                   int exclude_self, cudaStream_t st)
{
    const long long ctas4 = (long long)b * ((pn2 + 127) / 128);
    const bool wide = ctas4 >= 2LL * pvnet::sm_count();
    const int per = wide ? 128 : 32;
    const dim3 grid((pn2 + per - 1) / per, b);
    const dim3 block(32 * NN_WARPS);
    if (dim == 3) {
        if (wide) k_nearest_point_idx<3, 4><<<grid, block, 0, st>>>(ref, que, idxs, pn1, pn2, exclude_self);
        else k_nearest_point_idx<3, 1><<<grid, block, 0, st>>>(ref, que, idxs, pn1, pn2, exclude_self);
    } else {
        if (wide) k_nearest_point_idx<2, 4><<<grid, block, 0, st>>>(ref, que, idxs, pn1, pn2, exclude_self);
        else k_nearest_point_idx<2, 1><<<grid, block, 0, st>>>(ref, que, idxs, pn1, pn2, exclude_self);
    }
    PV_LAUNCHED("k_nearest_point_idx");
    return PVNET_OK;
}

struct Cam {
    double k[9];
};

struct PointClouds {
    double pred[3], tgt[3];   // camera-frame points (the reference's model_pred / model_targets)
    double pred2[2], tgt2[2]; // their projections (Projector.project_K)
};

// numpy: np.dot(model, R.T) + t.  A float64 pose gives a float64 cloud; a float32 pose gives a float32 cloud: the
// length-3 product as numpy's float32 matmul (an sgemm) accumulates it, fma(z,R2, fma(y,R1, x*R0)), then the
// float32 sum with t.  That sequence reproduces numpy's cloud bit for bit on every point of the fixtures.
__device__ __forceinline__ void transform(const double *P, float x, float y, float z, bool f32, double out[3])
{
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        if (f32) {
            const float d = __fmaf_rn(z, (float)P[r * 4 + 2], __fmaf_rn(y, (float)P[r * 4 + 1],
                                                                        __fmul_rn(x, (float)P[r * 4])));
            out[r] = (double)__fadd_rn(d, (float)P[r * 4 + 3]);
        } else {
            out[r] = fma(P[r * 4 + 2], (double)z, fma(P[r * 4 + 1], (double)y, P[r * 4] * (double)x)) + P[r * 4 + 3];
        }
    }
}

// base_utils.py:290-294: pts @ K.T, then [:2] / [2:]
__device__ __forceinline__ void project(const double *K, const double p[3], double out[2])
{
    const double u = fma(K[2], p[2], fma(K[1], p[1], K[0] * p[0]));
    const double v = fma(K[5], p[2], fma(K[4], p[1], K[3] * p[0]));
    const double w = fma(K[8], p[2], fma(K[7], p[1], K[6] * p[0]));
    out[0] = u / w;
    out[1] = v / w;
}

__device__ __forceinline__ const double *camera(const Cam &cam, const double *K_img, int bi)
{
    return K_img ? K_img + (size_t)bi * 9 : cam.k;
}

__device__ __forceinline__ void clouds(const double *pp, const double *pg, const double *K, const float *X, int i,
                                       int flags, PointClouds &c)
{
    const float x = X[(size_t)i * 3], y = X[(size_t)i * 3 + 1], z = X[(size_t)i * 3 + 2];
    transform(pp, x, y, z, flags & PVNET_METRICS_PRED_F32, c.pred);
    transform(pg, x, y, z, flags & PVNET_METRICS_GT_F32, c.tgt);
    project(K, c.pred, c.pred2);
    project(K, c.tgt, c.tgt2);
}

// The clouds the symmetric metrics search over, rounded to float32 as find_nearest_point_idx casts them
// (extend_utils.py:50-51): 3-D [b,pn,3] for ADD-S, 2-D [b,pn,2] for the symmetric projection metric.
__global__ void k_metric_clouds(const double *__restrict__ pose_pred, const double *__restrict__ pose_gt,
                                const float *__restrict__ X, Cam cam, const double *__restrict__ K_img, int b, int pn,
                                int flags, float *pred3, float *tgt3, float *pred2, float *tgt2)
{
    const long long n = (long long)b * pn;
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n; g += (long long)gridDim.x * blockDim.x) {
        const int bi = (int)(g / pn), i = (int)(g % pn);
        PointClouds c;
        clouds(pose_pred + bi * 12, pose_gt + bi * 12, camera(cam, K_img, bi), X, i, flags, c);
        if (flags & PVNET_METRICS_SYM_ADD)
            for (int r = 0; r < 3; ++r) {
                pred3[g * 3 + r] = __double2float_rn(c.pred[r]);
                tgt3[g * 3 + r] = __double2float_rn(c.tgt[r]);
            }
        if (flags & PVNET_METRICS_SYM_PROJ)
            for (int r = 0; r < 2; ++r) {
                pred2[g * 2 + r] = __double2float_rn(c.pred2[r]);
                tgt2[g * 2 + r] = __double2float_rn(c.tgt2[r]);
            }
    }
}

constexpr int MT = 256;

__device__ __forceinline__ double norm3(double a, double b, double c) { return sqrt(fma(c, c, fma(b, b, a * a))); }

// One CTA per image.  values [b,4] = (add_dist, proj_mean_diff, trans_cm, rot_deg); ok [b,3] = (add, proj, 5cm5deg).
__global__ void __launch_bounds__(MT) k_pose_metrics(const double *__restrict__ pose_pred,
                                                     const double *__restrict__ pose_gt, const float *__restrict__ X,
                                                     Cam cam, const double *__restrict__ K_img, int pn, int flags,
                                                     const int32_t *__restrict__ nn3, const int32_t *__restrict__ nn2,
                                                     double add_thr, double proj_thr, double cm_thr, double deg_thr,
                                                     double *__restrict__ values, uint8_t *__restrict__ ok)
{
    __shared__ double s_add[MT], s_proj[MT];
    const int bi = blockIdx.x;
    const double *pp = pose_pred + bi * 12, *pg = pose_gt + bi * 12;
    const double *K = camera(cam, K_img, bi);
    double add = 0.0, proj = 0.0;
    for (int i = threadIdx.x; i < pn; i += MT) {
        PointClouds c;
        clouds(pp, pg, K, X, i, flags, c);
        // find_nearest_point_distance(pred, target) (evaluation_utils.py:54-62): every target point against its
        // nearest predicted point, distance on the unrounded values
        double p3[3] = {c.pred[0], c.pred[1], c.pred[2]}, p2[2] = {c.pred2[0], c.pred2[1]};
        if (nn3 || nn2) {
            const int j3 = nn3 ? nn3[(size_t)bi * pn + i] : i, j2 = nn2 ? nn2[(size_t)bi * pn + i] : i;
            PointClouds c3, c2;
            clouds(pp, pg, K, X, j3, flags, c3);
            clouds(pp, pg, K, X, j2, flags, c2);
            for (int r = 0; r < 3; ++r) p3[r] = c3.pred[r];
            for (int r = 0; r < 2; ++r) p2[r] = c2.pred2[r];
        }
        add += norm3(p3[0] - c.tgt[0], p3[1] - c.tgt[1], p3[2] - c.tgt[2]);
        const double du = p2[0] - c.tgt2[0], dv = p2[1] - c.tgt2[1];
        proj += sqrt(fma(dv, dv, du * du));
    }
    s_add[threadIdx.x] = add;
    s_proj[threadIdx.x] = proj;
    __syncthreads();
    for (int s = MT / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            s_add[threadIdx.x] += s_add[threadIdx.x + s];
            s_proj[threadIdx.x] += s_proj[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double add_dist = s_add[0] / pn, proj_diff = s_proj[0] / pn;
        // cm_degree_5_metric (evaluation_utils.py:132-141)
        const double trans = norm3(pp[3] - pg[3], pp[7] - pg[7], pp[11] - pg[11]) * 100.0;
        double tr = 0.0;
        for (int r = 0; r < 3; ++r)
            for (int k = 0; k < 3; ++k) tr = fma(pp[r * 4 + k], pg[r * 4 + k], tr);
        tr = tr <= 3.0 ? tr : 3.0;  // `trace if trace <= 3 else 3`: NaN also becomes 3; no lower clamp
        const double deg = acos((tr - 1.0) / 2.0) * (180.0 / 3.14159265358979323846);
        values[bi * 4 + 0] = add_dist;
        values[bi * 4 + 1] = proj_diff;
        values[bi * 4 + 2] = trans;
        values[bi * 4 + 3] = deg;
        ok[bi * 3 + 0] = add_dist < add_thr;
        ok[bi * 3 + 1] = proj_diff < proj_thr;
        ok[bi * 3 + 2] = trans < cm_thr && deg < deg_thr;
    }
}

struct MetricsWs {
    float *pred3 = nullptr, *tgt3 = nullptr, *pred2 = nullptr, *tgt2 = nullptr;
    int32_t *nn3 = nullptr, *nn2 = nullptr;
    size_t bytes = 0;
};

MetricsWs carve_metrics(void *base, int b, int pn, int flags)
{
    pvnet::Carver c(base);
    MetricsWs w;
    const size_t n = (size_t)b * pn;
    if (flags & PVNET_METRICS_SYM_ADD) {
        w.pred3 = c.take<float>(n * 3);
        w.tgt3 = c.take<float>(n * 3);
        w.nn3 = c.take<int32_t>(n);
    }
    if (flags & PVNET_METRICS_SYM_PROJ) {
        w.pred2 = c.take<float>(n * 2);
        w.tgt2 = c.take<float>(n * 2);
        w.nn2 = c.take<int32_t>(n);
    }
    w.bytes = c.off;
    return w;
}

constexpr int METRICS_FLAGS = PVNET_METRICS_SYM_ADD | PVNET_METRICS_SYM_PROJ | PVNET_METRICS_PRED_F32 |
                              PVNET_METRICS_GT_F32;

}  // namespace

extern "C" {

int pvnet_find_nearest_point_idx(const float *ref, const float *que, int32_t *idxs, int b, int pn1, int pn2, int dim,
                                 int exclude_self, pvnet_stream_t stream)
{
    PV_CHECK_ARG(ref && que && idxs, "null pointer");
    PV_CHECK_ARG(dim == 2 || dim == 3, "dim %d is neither 2 nor 3", dim);
    PV_CHECK_ARG(b >= 1 && pn1 >= 1 && pn2 >= 1, "non-positive size (b %d, pn1 %d, pn2 %d)", b, pn1, pn2);
    PV_CHECK_ARG(b <= 65535, "batch %d above 65535", b);
    return launch_nearest(ref, que, idxs, b, pn1, pn2, dim, exclude_self, (cudaStream_t)stream);
}

int pvnet_pose_metrics_workspace_bytes(int b, int pn, int flags, size_t *bytes)
{
    PV_CHECK_ARG(bytes, "null pointer");
    PV_CHECK_ARG(b >= 1 && pn >= 1, "non-positive size (b %d, pn %d)", b, pn);
    *bytes = carve_metrics(nullptr, b, pn, flags).bytes;
    return PVNET_OK;
}

int pvnet_pose_metrics(const double *pose_pred, const double *pose_gt, const float *model_points,
                       const double camera_matrix[9], const double *camera_matrices, int b, int pn, int flags,
                       double add_threshold, double proj_threshold, double cm_threshold, double deg_threshold,
                       double *values, uint8_t *ok, void *workspace, size_t workspace_bytes, pvnet_stream_t stream)
{
    PV_CHECK_ARG(pose_pred && pose_gt && model_points && values && ok, "null pointer");
    PV_CHECK_ARG((camera_matrix != nullptr) != (camera_matrices != nullptr),
                 "pass exactly one of camera_matrix / camera_matrices");
    PV_CHECK_ARG(b >= 1 && pn >= 1, "non-positive size (b %d, pn %d)", b, pn);
    PV_CHECK_ARG(b <= 65535, "batch %d above 65535", b);
    PV_CHECK_ARG((flags & ~METRICS_FLAGS) == 0, "unknown flag bits 0x%x", flags & ~METRICS_FLAGS);
    const MetricsWs need = carve_metrics(nullptr, b, pn, flags);
    PV_CHECK_ARG(need.bytes == 0 || workspace, "null workspace");
    if (workspace_bytes < need.bytes) {
        pvnet::set_error("workspace %zu bytes < %zu needed", workspace_bytes, need.bytes);
        return PVNET_E_WORKSPACE;
    }
    const MetricsWs w = carve_metrics(workspace, b, pn, flags);
    cudaStream_t st = (cudaStream_t)stream;
    Cam cam{};
    if (camera_matrix)
        for (int i = 0; i < 9; ++i) cam.k[i] = camera_matrix[i];
    if (flags & (PVNET_METRICS_SYM_ADD | PVNET_METRICS_SYM_PROJ)) {
        const long long n = (long long)b * pn;
        const long long cap = 8LL * pvnet::sm_count();
        const int grid = (int)((n + 255) / 256 < cap ? (n + 255) / 256 : cap);
        k_metric_clouds<<<grid, 256, 0, st>>>(pose_pred, pose_gt, model_points, cam, camera_matrices, b, pn, flags,
                                              w.pred3, w.tgt3, w.pred2, w.tgt2);
        PV_LAUNCHED("k_metric_clouds");
        // ref = prediction, query = target (evaluation_utils.py:61: find_nearest_point_idx(pts1, pts2))
        if (flags & PVNET_METRICS_SYM_ADD) {
            int s = launch_nearest(w.pred3, w.tgt3, w.nn3, b, pn, pn, 3, 0, st);
            if (s) return s;
        }
        if (flags & PVNET_METRICS_SYM_PROJ) {
            int s = launch_nearest(w.pred2, w.tgt2, w.nn2, b, pn, pn, 2, 0, st);
            if (s) return s;
        }
    }
    k_pose_metrics<<<b, MT, 0, st>>>(pose_pred, pose_gt, model_points, cam, camera_matrices, pn, flags, w.nn3, w.nn2,
                                     add_threshold, proj_threshold, cm_threshold, deg_threshold, values, ok);
    PV_LAUNCHED("k_pose_metrics");
    return PVNET_OK;
}

}  // extern "C"
