// align.cu -- K14: superposition of trajectory frames (Molecule.align / molRMSD / MetricRmsd).
//
// Replaces the frame loop of moleculekit's _pp_align / _pp_measure_fit (numpy SVD per frame) and util.molRMSD.
//   fit   : per listed frame, float64 sums over the fit selection -> centroids and 3x3 covariance -> optimal proper
//           rotation (Horn's quaternion, cyclic Jacobi on the 4x4 key matrix) -> transform [R row-major | cP | cQ].
//   apply : x' = (x - cP) R^T + cQ for every atom of every listed frame, in float64, rounded once to float32, in place.
//   rmsd  : per listed frame, float64 sum of |x' - r|^2 over the RMSD selection; x' = the float32 value `apply` would
//           store (or the stored coordinate when no transform is given).
//
// Mapping.  A (atom, dim) row of the trajectory is contiguous along frames, so a block is FPB frame lanes x APB atom lanes
// (FPB * APB = 256): for many frames a warp reads 32 consecutive frames of one row; for one frame all 256 threads run over
// atoms.  FPB is the smallest power of two >= n_frames, capped at 32.  The fit and RMSD reductions are split into atom
// chunks whose size depends only on the selection size and FPB: every thread sums its atoms in order, the block folds the
// atom lanes with a fixed tree, and a second kernel adds the chunks in order.  No atomics, so identical calls give
// identical bits, and a frame shard gives the bits of the whole trajectory whenever both use the same FPB.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>

#include "common.cuh"

using namespace mkb;

namespace {

constexpr int K14_THREADS = 256;
constexpr int FIT_K = 15;  // sums of p' (3), q' (3), p' q'^T (9); p' = p - p0, q' = q - q0 (first selected atom)

// smallest power of two >= n_frames, capped at 32
inline int frames_per_block(int64_t n_frames) {
    int f = 1;
    while (f < 32 && f < n_frames) f *= 2;
    return f;
}

// atoms of the selection per chunk: a function of the selection size and FPB only (see the header comment)
inline int64_t chunk_atoms(int64_t n_sel, int fpb) {
    const int64_t apb = K14_THREADS / fpb;
    const int64_t max_chunks = 512 / fpb;
    const int64_t per_lane = std::max<int64_t>(8, cdiv(n_sel, apb * max_chunks));
    return apb * per_lane;
}

__device__ __forceinline__ float ld_row(const float *coords, int64_t fs, int64_t atom, int d, int64_t f) {
    return __ldg(coords + (atom * 3 + d) * fs + f);
}

// Fixed-order fold of the atom lanes: red[al][fl][k], al = 0 ends with the block's sums.
template <int FPB, int K>
__device__ __forceinline__ void fold_lanes(double (*red)[FPB][K], int al, int fl) {
    constexpr int APB = K14_THREADS / FPB;
#pragma unroll
    for (int s = APB / 2; s > 0; s >>= 1) {
        __syncthreads();
        if (al < s) {
#pragma unroll
            for (int k = 0; k < K; ++k) red[al][fl][k] += red[al + s][fl][k];
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------- fit
template <int FPB>
__global__ void __launch_bounds__(K14_THREADS) k14_fit_partial_kernel(
    const float *__restrict__ coords, int64_t fs, const int64_t *__restrict__ frames, int64_t n_frames,
    const uint32_t *__restrict__ sel, int64_t n_sel, const float *__restrict__ ref, int64_t rs, int32_t matching,
    int64_t chunk, double *__restrict__ partial) {
    __shared__ double red[K14_THREADS / FPB][FPB][FIT_K];
    const int fl = threadIdx.x % FPB, al = threadIdx.x / FPB;
    constexpr int APB = K14_THREADS / FPB;
    const int64_t i = (int64_t)blockIdx.x * FPB + fl;
    double acc[FIT_K];
#pragma unroll
    for (int k = 0; k < FIT_K; ++k) acc[k] = 0.0;
    if (i < n_frames) {
        const int64_t f = frames[i], fr = matching ? f : 0;
        const int64_t a0 = sel[0];
        const double p0[3] = {ld_row(coords, fs, a0, 0, f), ld_row(coords, fs, a0, 1, f), ld_row(coords, fs, a0, 2, f)};
        const double q0[3] = {__ldg(ref + fr), __ldg(ref + rs + fr), __ldg(ref + 2 * rs + fr)};
        const int64_t j0 = (int64_t)blockIdx.y * chunk, j1 = j0 + chunk < n_sel ? j0 + chunk : n_sel;
        for (int64_t j = j0 + al; j < j1; j += APB) {
            const int64_t a = sel[j];
            double p[3], q[3];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                p[d] = (double)ld_row(coords, fs, a, d, f) - p0[d];  // exact: both are float32 values
                q[d] = (double)__ldg(ref + (j * 3 + d) * rs + fr) - q0[d];
            }
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                acc[d] += p[d];
                acc[3 + d] += q[d];
            }
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[6 + 3 * r + c] = fma(p[r], q[c], acc[6 + 3 * r + c]);
        }
    }
#pragma unroll
    for (int k = 0; k < FIT_K; ++k) red[al][fl][k] = acc[k];
    fold_lanes<FPB, FIT_K>(red, al, fl);
    if (al == 0 && i < n_frames) {
        double *out = partial + ((int64_t)blockIdx.y * n_frames + i) * FIT_K;
#pragma unroll
        for (int k = 0; k < FIT_K; ++k) out[k] = red[0][fl][k];
    }
}

// Largest-eigenvalue eigenvector of the symmetric 4x4 A (cyclic Jacobi, fixed sweep count).  Ties go to the lowest index,
// so A = 0 gives e0 -- the identity quaternion.
__device__ void top_eigvec4(double A[4][4], double v[4]) {
    double V[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) V[r][c] = r == c ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 12; ++sweep) {
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                const double apq = A[p][q];
                if (apq == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
                double t;
                if (fabs(theta) > 1e150) t = 0.5 / theta;
                else t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - s * akq;
                    A[k][q] = s * akp + c * akq;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - s * aqk;
                    A[q][k] = s * apk + c * aqk;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - s * vkq;
                    V[k][q] = s * vkp + c * vkq;
                }
            }
        }
    }
    int best = 0;
#pragma unroll
    for (int k = 1; k < 4; ++k)
        if (A[k][k] > A[best][best]) best = k;
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = V[k][best];
}

// One thread per listed frame: add the chunks in order, then centroids, covariance and rotation.
__global__ void k14_fit_solve_kernel(const float *__restrict__ coords, int64_t fs, const int64_t *__restrict__ frames,
                                     int64_t n_frames, const uint32_t *__restrict__ sel, int64_t n_sel,
                                     const float *__restrict__ ref, int64_t rs, int32_t matching,
                                     const double *__restrict__ partial, int64_t n_chunks, double *__restrict__ xf) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_frames) return;
    double s[FIT_K];
#pragma unroll
    for (int k = 0; k < FIT_K; ++k) s[k] = 0.0;
    for (int64_t c = 0; c < n_chunks; ++c) {
        const double *pp = partial + (c * n_frames + i) * FIT_K;
#pragma unroll
        for (int k = 0; k < FIT_K; ++k) s[k] += pp[k];
    }
    const int64_t f = frames[i], fr = matching ? f : 0, a0 = sel[0];
    const double inv_n = 1.0 / (double)n_sel;
    double mp[3], mq[3], cP[3], cQ[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        mp[d] = s[d] * inv_n;
        mq[d] = s[3 + d] * inv_n;
        cP[d] = (double)ld_row(coords, fs, a0, d, f) + mp[d];
        cQ[d] = (double)ref[d * rs + fr] + mq[d];
    }
    // H[r][c] = sum (p - cP)_r (q - cQ)_c = sum p'_r q'_c - n mp_r mq_c
    double H[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) H[r][c] = fma(-(double)n_sel * mp[r], mq[c], s[6 + 3 * r + c]);
    // Horn's key matrix: its top eigenvector is the quaternion of the rotation maximising sum q_c . (R p_c)
    const double Sxx = H[0][0], Sxy = H[0][1], Sxz = H[0][2], Syx = H[1][0], Syy = H[1][1], Syz = H[1][2], Szx = H[2][0],
                 Szy = H[2][1], Szz = H[2][2];
    double N[4][4] = {{Sxx + Syy + Szz, Syz - Szy, Szx - Sxz, Sxy - Syx},
                      {Syz - Szy, Sxx - Syy - Szz, Sxy + Syx, Szx + Sxz},
                      {Szx - Sxz, Sxy + Syx, -Sxx + Syy - Szz, Syz + Szy},
                      {Sxy - Syx, Szx + Sxz, Syz + Szy, -Sxx - Syy + Szz}};
    double qv[4];
    top_eigvec4(N, qv);
    const double nrm = 1.0 / sqrt(qv[0] * qv[0] + qv[1] * qv[1] + qv[2] * qv[2] + qv[3] * qv[3]);
    const double w = qv[0] * nrm, x = qv[1] * nrm, y = qv[2] * nrm, z = qv[3] * nrm;
    double *o = xf + i * FIT_K;
    o[0] = w * w + x * x - y * y - z * z;
    o[1] = 2.0 * (x * y - w * z);
    o[2] = 2.0 * (x * z + w * y);
    o[3] = 2.0 * (x * y + w * z);
    o[4] = w * w - x * x + y * y - z * z;
    o[5] = 2.0 * (y * z - w * x);
    o[6] = 2.0 * (x * z - w * y);
    o[7] = 2.0 * (y * z + w * x);
    o[8] = w * w - x * x - y * y + z * z;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        o[9 + d] = cP[d];
        o[12 + d] = cQ[d];
    }
}

struct Xf {
    double R[9], cP[3], cQ[3];
};

__device__ __forceinline__ void load_xf(const double *__restrict__ xf, int64_t i, Xf &t) {
    const double *p = xf + i * FIT_K;
#pragma unroll
    for (int k = 0; k < 9; ++k) t.R[k] = __ldg(p + k);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        t.cP[d] = __ldg(p + 9 + d);
        t.cQ[d] = __ldg(p + 12 + d);
    }
}

// x' = (x - cP) R^T + cQ in float64, rounded once
__device__ __forceinline__ void xf_point(const Xf &t, const float x[3], float y[3]) {
    const double u0 = (double)x[0] - t.cP[0], u1 = (double)x[1] - t.cP[1], u2 = (double)x[2] - t.cP[2];
#pragma unroll
    for (int r = 0; r < 3; ++r) y[r] = (float)(t.R[3 * r] * u0 + t.R[3 * r + 1] * u1 + t.R[3 * r + 2] * u2 + t.cQ[r]);
}

// ---------------------------------------------------------------------------------------------------------- apply
template <int FPB>
__global__ void __launch_bounds__(K14_THREADS) k14_apply_kernel(float *__restrict__ coords, int64_t fs,
                                                                const int64_t *__restrict__ frames, int64_t n_frames,
                                                                int64_t n_atoms, int64_t chunk,
                                                                const double *__restrict__ xf) {
    constexpr int APB = K14_THREADS / FPB;
    const int fl = threadIdx.x % FPB, al = threadIdx.x / FPB;
    const int64_t i = (int64_t)blockIdx.x * FPB + fl;
    if (i >= n_frames) return;
    const int64_t f = frames[i];
    Xf t;
    load_xf(xf, i, t);
    const int64_t a0 = (int64_t)blockIdx.y * chunk, a1 = a0 + chunk < n_atoms ? a0 + chunk : n_atoms;
    int64_t a = a0 + al;
    // two atoms in flight per thread: six independent loads before the first store
    for (; a + APB < a1; a += 2 * APB) {
        float x[3], x2[3], y[3], y2[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            x[d] = coords[(a * 3 + d) * fs + f];
            x2[d] = coords[((a + APB) * 3 + d) * fs + f];
        }
        xf_point(t, x, y);
        xf_point(t, x2, y2);
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            __stcs(coords + (a * 3 + d) * fs + f, y[d]);
            __stcs(coords + ((a + APB) * 3 + d) * fs + f, y2[d]);
        }
    }
    if (a < a1) {
        float x[3], y[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) x[d] = coords[(a * 3 + d) * fs + f];
        xf_point(t, x, y);
#pragma unroll
        for (int d = 0; d < 3; ++d) __stcs(coords + (a * 3 + d) * fs + f, y[d]);
    }
}

// ---------------------------------------------------------------------------------------------------------- rmsd
template <int FPB>
__global__ void __launch_bounds__(K14_THREADS) k14_rmsd_partial_kernel(
    const float *__restrict__ coords, int64_t fs, const int64_t *__restrict__ frames, int64_t n_frames,
    const uint32_t *__restrict__ sel, int64_t n_sel, const float *__restrict__ ref, int64_t rs, int64_t ref_frames,
    const double *__restrict__ xf, int64_t chunk, double *__restrict__ partial) {
    __shared__ double red[K14_THREADS / FPB][FPB][1];
    constexpr int APB = K14_THREADS / FPB;
    const int fl = threadIdx.x % FPB, al = threadIdx.x / FPB;
    const int64_t i = (int64_t)blockIdx.x * FPB + fl;
    double acc = 0.0;
    if (i < n_frames) {
        const int64_t f = frames[i], fr = ref_frames == 1 ? 0 : f;
        Xf t;
        if (xf) load_xf(xf, i, t);
        const int64_t j0 = (int64_t)blockIdx.y * chunk, j1 = j0 + chunk < n_sel ? j0 + chunk : n_sel;
        for (int64_t j = j0 + al; j < j1; j += APB) {
            const int64_t a = sel[j];
            float x[3], y[3];
#pragma unroll
            for (int d = 0; d < 3; ++d) x[d] = ld_row(coords, fs, a, d, f);
            if (xf) xf_point(t, x, y);
            else {
#pragma unroll
                for (int d = 0; d < 3; ++d) y[d] = x[d];
            }
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const double e = (double)y[d] - (double)__ldg(ref + (j * 3 + d) * rs + fr);
                acc = fma(e, e, acc);
            }
        }
    }
    red[al][fl][0] = acc;
    fold_lanes<FPB, 1>(red, al, fl);
    if (al == 0 && i < n_frames) partial[(int64_t)blockIdx.y * n_frames + i] = red[0][fl][0];
}

__global__ void k14_rmsd_finish_kernel(const double *__restrict__ partial, int64_t n_frames, int64_t n_chunks,
                                       int64_t n_sel, float *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_frames) return;
    double s = 0.0;
    for (int64_t c = 0; c < n_chunks; ++c) s += partial[c * n_frames + i];
    out[i] = (float)sqrt(s / (double)n_sel);
}

// ---------------------------------------------------------------------------------------------------------- dispatch
#define K14_DISPATCH(KERNEL, fpb, grid, st, ...)                                          \
    switch (fpb) {                                                                        \
    case 1: KERNEL<1><<<grid, K14_THREADS, 0, st>>>(__VA_ARGS__); break;                  \
    case 2: KERNEL<2><<<grid, K14_THREADS, 0, st>>>(__VA_ARGS__); break;                  \
    case 4: KERNEL<4><<<grid, K14_THREADS, 0, st>>>(__VA_ARGS__); break;                  \
    case 8: KERNEL<8><<<grid, K14_THREADS, 0, st>>>(__VA_ARGS__); break;                  \
    case 16: KERNEL<16><<<grid, K14_THREADS, 0, st>>>(__VA_ARGS__); break;                \
    default: KERNEL<32><<<grid, K14_THREADS, 0, st>>>(__VA_ARGS__); break;                \
    }

int check_traj(mkb_ctx *h, const mkb_traj *t, const int64_t *frames, int64_t n_frames) {
    if (!t) return fail(h, MKB_ERR_BAD_ARG, "null trajectory");
    if (t->n_atoms < 0 || t->n_frames < 0 || n_frames < 0) return fail(h, MKB_ERR_BAD_ARG, "negative size");
    if (n_frames > 0 && (!frames || !t->coords)) return fail(h, MKB_ERR_BAD_ARG, "null argument");
    if (t->n_frames > 1 && t->frame_stride < t->n_frames) return fail(h, MKB_ERR_BAD_ARG, "frame stride < n_frames");
    if (n_frames >= (1ll << 31)) return fail(h, MKB_ERR_BAD_ARG, "too many frames for one launch");
    return MKB_OK;
}

}  // namespace

extern "C" int mkb_align_fit(mkb_handle_t h, void *stream, const mkb_traj *t, const int64_t *frames, int64_t n_frames,
                             const uint32_t *sel, int64_t n_sel, const float *ref, int64_t ref_stride,
                             int32_t matchingframes, double *transforms) {
    MKB_ENTER(h);
    cudaStream_t st = (cudaStream_t)stream;
    MKB_STREAM_ORDER(h, st);
    int rc;
    if ((rc = check_traj(h, t, frames, n_frames))) return rc;
    if (n_frames == 0) return MKB_OK;
    if (n_sel <= 0) return fail(h, MKB_ERR_BAD_ARG, "empty fit selection");
    if (!sel || !ref || !transforms) return fail(h, MKB_ERR_BAD_ARG, "null argument");
    if (ref_stride < 1) return fail(h, MKB_ERR_BAD_ARG, "ref_stride < 1");
    const int fpb = frames_per_block(n_frames);
    const int64_t chunk = chunk_atoms(n_sel, fpb), n_chunks = cdiv(n_sel, chunk);
    double *partial = nullptr;
    if ((rc = scratch_get(h, S_COM, (size_t)(n_chunks * n_frames * FIT_K), &partial))) return rc;
    const dim3 grid((unsigned)cdiv(n_frames, fpb), (unsigned)n_chunks);
    K14_DISPATCH(k14_fit_partial_kernel, fpb, grid, st, t->coords, t->frame_stride, frames, n_frames, sel, n_sel, ref,
                 ref_stride, matchingframes, chunk, partial);
    MKB_LAUNCHED(h);
    k14_fit_solve_kernel<<<(unsigned)cdiv(n_frames, 128), 128, 0, st>>>(t->coords, t->frame_stride, frames, n_frames,
                                                                        sel, n_sel, ref, ref_stride, matchingframes,
                                                                        partial, n_chunks, transforms);
    MKB_LAUNCHED(h);
    h->last_kernel = "k14_fit_partial_kernel";
    return MKB_OK;
}

extern "C" int mkb_align_apply(mkb_handle_t h, void *stream, const mkb_traj *t, const int64_t *frames,
                               int64_t n_frames, const double *transforms) {
    MKB_ENTER(h);
    cudaStream_t st = (cudaStream_t)stream;
    MKB_STREAM_ORDER(h, st);
    int rc;
    if ((rc = check_traj(h, t, frames, n_frames))) return rc;
    if (n_frames == 0 || t->n_atoms == 0) return MKB_OK;
    if (!transforms) return fail(h, MKB_ERR_BAD_ARG, "null transforms");
    const int fpb = frames_per_block(n_frames);
    const int64_t apb = K14_THREADS / fpb, tiles = cdiv(n_frames, fpb);
    // about 16 blocks per SM in all, at least 4 atoms per atom lane
    const int64_t n_chunks = std::max<int64_t>(
        1, std::min<int64_t>(cdiv(t->n_atoms, 4 * apb), std::max<int64_t>(1, 16ll * h->sm_count / tiles)));
    const int64_t chunk = cdiv(t->n_atoms, n_chunks);
    const dim3 grid((unsigned)tiles, (unsigned)cdiv(t->n_atoms, chunk));
    K14_DISPATCH(k14_apply_kernel, fpb, grid, st, const_cast<float *>(t->coords), t->frame_stride, frames, n_frames,
                 t->n_atoms, chunk, transforms);
    MKB_LAUNCHED(h);
    h->last_kernel = "k14_apply_kernel";
    return MKB_OK;
}

extern "C" int mkb_rmsd(mkb_handle_t h, void *stream, const mkb_traj *t, const int64_t *frames, int64_t n_frames,
                        const uint32_t *sel, int64_t n_sel, const float *ref, int64_t ref_stride, int64_t ref_frames,
                        const double *transforms, float *out) {
    MKB_ENTER(h);
    cudaStream_t st = (cudaStream_t)stream;
    MKB_STREAM_ORDER(h, st);
    int rc;
    if ((rc = check_traj(h, t, frames, n_frames))) return rc;
    if (n_frames == 0) return MKB_OK;
    if (n_sel <= 0) return fail(h, MKB_ERR_BAD_ARG, "empty RMSD selection");
    if (!sel || !ref || !out) return fail(h, MKB_ERR_BAD_ARG, "null argument");
    if (ref_stride < 1 || ref_frames < 1) return fail(h, MKB_ERR_BAD_ARG, "ref_stride and ref_frames must be >= 1");
    const int fpb = frames_per_block(n_frames);
    const int64_t chunk = chunk_atoms(n_sel, fpb), n_chunks = cdiv(n_sel, chunk);
    double *partial = nullptr;
    if ((rc = scratch_get(h, S_COM, (size_t)(n_chunks * n_frames), &partial))) return rc;
    const dim3 grid((unsigned)cdiv(n_frames, fpb), (unsigned)n_chunks);
    K14_DISPATCH(k14_rmsd_partial_kernel, fpb, grid, st, t->coords, t->frame_stride, frames, n_frames, sel, n_sel, ref,
                 ref_stride, ref_frames, transforms, chunk, partial);
    MKB_LAUNCHED(h);
    k14_rmsd_finish_kernel<<<(unsigned)cdiv(n_frames, 128), 128, 0, st>>>(partial, n_frames, n_chunks, n_sel, out);
    MKB_LAUNCHED(h);
    h->last_kernel = "k14_rmsd_partial_kernel";
    return MKB_OK;
}
