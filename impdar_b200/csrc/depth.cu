// Time-to-depth conversion of a migrated (snum, tnum) time section with interval-velocity profiles (depthConvert).
//
// Trace x uses profile col_profile[x] of the P interval profiles v (P x snum, m/s).  Its depth curve is the one-way depth
// of every sample (impdar_b200.migrationlib.depth_curves, the same operations in the same order):
//   t = tt_us / 1e6, j0 = the first sample with t >= 0 (the last sample if there is none)
//   z[j0] = v[j0] t[j0] / 2
//   z[i]  = z[i-1] + (v[i-1] + v[i]) / 2 (t[i] - t[i-1]) / 2      i > j0, summed left to right
//   z[i]  = z[i+1] - (v[i] + v[i+1]) / 2 (t[i+1] - t[i]) / 2      i < j0, summed right to left
// and out[k, x] = numpy.interp(zgrid[k], z, image[:, x], left=nan, right=nan) in float64 (interp_rows_kernel's mode-1
// arithmetic: exact hit or last node copies the sample, slope form from the left node, NaN retried from the right node).
// No FMA contraction anywhere: every product and sum is a separately rounded __dmul_rn / __dadd_rn.
//
//   depth_curve_kernel     one thread per profile walks the sequential trapezoid; a warp stages 32 profiles x 32
//                          samples through shared memory so the (P, snum) read and the sample-major (snum, P) write are
//                          both coalesced
//   depth_resample_kernel  one thread per DR_ROWS consecutive output rows of one column: a binary search for its first
//                          row, then a monotone walk; columns across the warp, so neighbouring traces that share a
//                          profile read the same curve addresses and adjacent image / output addresses
#include <cmath>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace impdar {

constexpr int DC_WARPS = 4;     // warps (32 profiles each) per block of the curve kernel
constexpr int DR_ROWS = 32;     // output rows per thread of the resampling kernel
constexpr int DR_THREADS = 128;

__device__ __forceinline__ double dc_step(double va, double vb, double ta, double tb) {
    // (va + vb) / 2 * (tb - ta) / 2, left to right; halving is exact
    return __dmul_rn(__dmul_rn(__dmul_rn(__dadd_rn(va, vb), 0.5), __dsub_rn(tb, ta)), 0.5);
}

// z (snum, P) from v (P, snum).  Forward tiles from the anchor sample's tile upwards, then backward tiles.
__global__ void __launch_bounds__(DC_WARPS * 32) depth_curve_kernel(const double *__restrict__ v,
                                                                    const double *__restrict__ t,
                                                                    double *__restrict__ z, int S, int P, int j0) {
    __shared__ double tile[DC_WARPS][32][33];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p0 = (blockIdx.x * DC_WARPS + w) * 32;
    if (p0 >= P) return;   // whole warps
    const int p = p0 + lane;
    const int np = min(32, P - p0);
    double (*tl)[33] = tile[w];
    // tile c covers samples [c * 32, c * 32 + 32); lane l loads sample c * 32 + l of the warp's 32 profiles
    auto load = [&](int c) {
        const int j = c * 32 + lane;
        __syncwarp();
        if (j < S) {
#pragma unroll 8
            for (int r = 0; r < 32; ++r)
                if (r < np) tl[r][lane] = v[(size_t)(p0 + r) * S + j];
        }
        __syncwarp();
    };
    const int cj = j0 >> 5;
    const int ntile = (S + 31) >> 5;
    double zc = 0.0, vprev = 0.0, tprev = 0.0;
    for (int c = cj; c < ntile; ++c) {
        load(c);
        const int jb = c == cj ? j0 : c * 32, je = min(c * 32 + 32, S);
        for (int j = jb; j < je; ++j) {
            const double vj = tl[lane][j - c * 32], tj = t[j];
            zc = (j == j0) ? __dmul_rn(__dmul_rn(vj, tj), 0.5) : __dadd_rn(zc, dc_step(vprev, vj, tprev, tj));
            vprev = vj;
            tprev = tj;
            if (lane < np) z[(size_t)j * P + p] = zc;
        }
    }
    if (j0 == 0) return;
    // backward, from the anchor (its tile staged again)
    load(cj);
    double vnext = tl[lane][j0 - cj * 32], tnext = t[j0];
    double znext = __dmul_rn(__dmul_rn(vnext, tnext), 0.5);
    for (int c = cj; c >= 0; --c) {
        if (c != cj) load(c);
        const int jb = c == cj ? j0 - 1 : c * 32 + 31;
        for (int j = jb; j >= c * 32; --j) {
            const double vj = tl[lane][j - c * 32], tj = t[j];
            znext = __dsub_rn(znext, dc_step(vj, vnext, tj, tnext));
            vnext = vj;
            tnext = tj;
            if (lane < np) z[(size_t)j * P + p] = znext;
        }
    }
}

template <typename TI>
__device__ __forceinline__ double dr_value(double zq, double zlo, double zhi, TI ylo, TI yhi, bool copy) {
    const double dlo = (double)ylo, dhi = (double)yhi;
    if (copy) return dlo;
    const double slope = __ddiv_rn(__dsub_rn(dhi, dlo), __dsub_rn(zhi, zlo));
    double r = __dadd_rn(__dmul_rn(slope, __dsub_rn(zq, zlo)), dlo);
    if (isnan(r)) {
        r = __dadd_rn(__dmul_rn(slope, __dsub_rn(zq, zhi)), dhi);
        if (isnan(r) && dlo == dhi) r = dlo;
    }
    return r;
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(DR_THREADS) depth_resample_kernel(const TI *__restrict__ x, TO *__restrict__ y,
                                                                    int S, int T, int nz, int P,
                                                                    const double *__restrict__ z,
                                                                    const int *__restrict__ colp,
                                                                    const double *__restrict__ zgrid) {
    const int col = blockIdx.x * DR_THREADS + threadIdx.x;
    if (col >= T) return;
    const TO nanv = (TO)__longlong_as_double(0x7ff8000000000000LL);
    const double *zc = z + colp[col];
    const double zfirst = zc[0], zlast = zc[(size_t)(S - 1) * P];
    for (int k0 = blockIdx.y * DR_ROWS; k0 < nz; k0 += gridDim.y * DR_ROWS) {
        const int k1 = min(k0 + DR_ROWS, nz);
        // j: the last node with z[j] <= zgrid[k0] (0 when zgrid[k0] < z[0]: those rows are NaN and do not move j)
        const double q0 = zgrid[k0];
        int j = 0;
        if (q0 >= zlast) {
            j = S - 1;
        } else if (q0 >= zfirst) {
            int lo = 0, hi = S - 1;   // z[lo] <= q0 < z[hi]
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (zc[(size_t)mid * P] <= q0) lo = mid; else hi = mid;
            }
            j = lo;
        }
        double zlo = zc[(size_t)j * P], zhi = j + 1 < S ? zc[(size_t)(j + 1) * P] : zlo;
        TI ylo = x[(size_t)j * T + col], yhi = j + 1 < S ? x[(size_t)(j + 1) * T + col] : ylo;
        for (int k = k0; k < k1; ++k) {
            const double q = zgrid[k];
            TO out;
            if (q < zfirst || q > zlast) {
                out = nanv;
            } else {
                if (j + 1 < S && zhi <= q) {
                    do {
                        ++j;
                        zlo = zhi;
                        zhi = j + 1 < S ? zc[(size_t)(j + 1) * P] : zlo;
                    } while (j + 1 < S && zhi <= q);
                    ylo = x[(size_t)j * T + col];
                    yhi = j + 1 < S ? x[(size_t)(j + 1) * T + col] : ylo;
                }
                out = (TO)dr_value<TI>(q, zlo, zhi, ylo, yhi, j == S - 1 || zlo == q);
            }
            y[(size_t)k * T + col] = out;
        }
    }
}

static inline size_t dc_align(size_t b) { return (b + 255) & ~(size_t)255; }

struct DepthLayout {
    size_t t, zg, colp, prof, curve, total;
};

static DepthLayout depth_layout(int S, int T, int nz, int P) {
    DepthLayout L;
    L.t = 0;
    L.zg = L.t + dc_align((size_t)S * sizeof(double));
    L.colp = L.zg + dc_align((size_t)nz * sizeof(double));
    L.prof = L.colp + dc_align((size_t)T * sizeof(int));
    L.curve = L.prof + dc_align((size_t)P * S * sizeof(double));
    L.total = L.curve + dc_align((size_t)S * P * sizeof(double)) + 256;
    return L;
}

// Host vectors go up through two page-locked staging buffers per device, in chunks: the memcpy into one buffer runs
// while the previous chunk's copy from the other is in flight, and the caller never waits for the stream to drain
// (a copy from pageable memory would block the host until it had).  A (P, snum) profile table of several GB streams
// through without a page-locked buffer of its size.
constexpr size_t DS_CHUNK = (size_t)32 << 20;
constexpr int DS_SLOTS = 2;
struct DepthStageSlot {
    void *host;
    cudaEvent_t ev;
    bool used;
};
struct DepthStage {
    DepthStageSlot slot[DS_SLOTS];
    int next;
};
static DepthStage g_dstage[IMPDAR_MAX_DEVICES];
static std::mutex g_dstage_mu;

static int depth_upload(DepthStage &sg, void *dst, const void *src, size_t bytes, cudaStream_t st) {
    for (size_t off = 0; off < bytes; off += DS_CHUNK) {
        const size_t n = bytes - off < DS_CHUNK ? bytes - off : DS_CHUNK;
        DepthStageSlot &sl = sg.slot[sg.next];
        sg.next = (sg.next + 1) % DS_SLOTS;
        if (!sl.ev) IMPDAR_CUDA(cudaEventCreateWithFlags(&sl.ev, cudaEventDisableTiming));
        if (!sl.host) IMPDAR_CUDA(cudaHostAlloc(&sl.host, DS_CHUNK, cudaHostAllocDefault));
        if (sl.used) IMPDAR_CUDA(cudaEventSynchronize(sl.ev));   // the copy that last read this slot has run
        memcpy(sl.host, (const char *)src + off, n);
        IMPDAR_CUDA(cudaMemcpyAsync((char *)dst + off, sl.host, n, cudaMemcpyHostToDevice, st));
        IMPDAR_CUDA(cudaEventRecord(sl.ev, st));
        sl.used = true;
    }
    return IMPDAR_B200_OK;
}

template <typename TI, typename TO>
static int depth_convert(const TI *x, TO *y, int S, int T, int nz, const double *tt_us, const double *profiles, int P,
                         const int *col_profile, const double *zgrid, void *workspace, size_t ws_bytes, void *stream) {
    IMPDAR_CHECK_ARG(x && y && tt_us && profiles && col_profile && zgrid && workspace, "depth_convert: null pointer");
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1 && nz >= 1 && P >= 1, "depth_convert: need snum >= 2, tnum >= 1, nz >= 1, nprof >= 1");
    const size_t need = impdar_depth_workspace_bytes(S, T, nz, P);
    IMPDAR_CHECK_ARG(ws_bytes >= need, "depth_convert: workspace too small (%zu < %zu)", ws_bytes, need);
    std::vector<double> t(S);
    for (int i = 0; i < S; ++i) {
        t[i] = tt_us[i] / 1.0e6;
        IMPDAR_CHECK_ARG(std::isfinite(t[i]), "depth_convert: travel_time[%d] = %g is not finite", i, tt_us[i]);
        IMPDAR_CHECK_ARG(i == 0 || t[i] > t[i - 1], "depth_convert: travel_time must be strictly ascending (sample %d)", i);
    }
    const size_t PS = (size_t)P * S;
    for (size_t i = 0; i < PS; ++i)
        IMPDAR_CHECK_ARG(std::isfinite(profiles[i]) && profiles[i] > 0.0,
                         "depth_convert: profile %zu velocity[%zu] = %g must be finite and positive", i / S, i % S,
                         profiles[i]);
    for (int c = 0; c < T; ++c)
        IMPDAR_CHECK_ARG(col_profile[c] >= 0 && col_profile[c] < P,
                         "depth_convert: col_profile[%d] = %d outside [0, %d)", c, col_profile[c], P);
    for (int k = 0; k < nz; ++k) {
        IMPDAR_CHECK_ARG(std::isfinite(zgrid[k]), "depth_convert: zgrid[%d] = %g is not finite", k, zgrid[k]);
        IMPDAR_CHECK_ARG(k == 0 || zgrid[k] > zgrid[k - 1], "depth_convert: zgrid must be strictly ascending (row %d)", k);
    }
    int j0 = S - 1;
    for (int i = 0; i < S; ++i)
        if (t[i] >= 0.0) { j0 = i; break; }
    int dev = 0;
    IMPDAR_CUDA(cudaGetDevice(&dev));
    IMPDAR_CHECK_ARG(dev >= 0 && dev < IMPDAR_MAX_DEVICES, "depth_convert: device index %d out of range", dev);
    const DepthLayout L = depth_layout(S, T, nz, P);
    char *ws = (char *)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    double *d_t = (double *)(ws + L.t), *d_zg = (double *)(ws + L.zg), *d_prof = (double *)(ws + L.prof);
    double *d_curve = (double *)(ws + L.curve);
    int *d_colp = (int *)(ws + L.colp);
    cudaStream_t st = (cudaStream_t)stream;
    {
        std::lock_guard<std::mutex> lk(g_dstage_mu);
        DepthStage &sg = g_dstage[dev];
        if (int rc = depth_upload(sg, d_t, t.data(), (size_t)S * sizeof(double), st)) return rc;
        if (int rc = depth_upload(sg, d_zg, zgrid, (size_t)nz * sizeof(double), st)) return rc;
        if (int rc = depth_upload(sg, d_colp, col_profile, (size_t)T * sizeof(int), st)) return rc;
        if (int rc = depth_upload(sg, d_prof, profiles, PS * sizeof(double), st)) return rc;
    }
    const int warps = (P + 31) / 32;
    ktimer_begin("depth_curve_kernel", st);
    depth_curve_kernel<<<(warps + DC_WARPS - 1) / DC_WARPS, DC_WARPS * 32, 0, st>>>(d_prof, d_t, d_curve, S, P, j0);
    ktimer_end(st);
    IMPDAR_LAUNCH_CHECK();
    const int groups = (nz + DR_ROWS - 1) / DR_ROWS;
    dim3 grid((unsigned)((T + DR_THREADS - 1) / DR_THREADS), (unsigned)(groups < 65535 ? groups : 65535));
    ktimer_begin("depth_resample_kernel", st);
    depth_resample_kernel<TI, TO><<<grid, DR_THREADS, 0, st>>>(x, y, S, T, nz, P, d_curve, d_colp, d_zg);
    ktimer_end(st);
    IMPDAR_LAUNCH_CHECK();
    return IMPDAR_B200_OK;
}

}  // namespace impdar

using namespace impdar;

extern "C" {

size_t impdar_depth_workspace_bytes(int snum, int tnum, int nz, int nprof) {
    if (snum < 2 || tnum < 1 || nz < 1 || nprof < 1) return 0;
    return depth_layout(snum, tnum, nz, nprof).total;
}

int impdar_depth_convert_f32(const float *x, float *y, int snum, int tnum, int nz, const double *tt_us,
                             const double *profiles, int nprof, const int *col_profile, const double *zgrid,
                             void *workspace, size_t workspace_bytes, void *stream) {
    return depth_convert<float, float>(x, y, snum, tnum, nz, tt_us, profiles, nprof, col_profile, zgrid, workspace,
                                       workspace_bytes, stream);
}
int impdar_depth_convert_f32_f64(const float *x, double *y, int snum, int tnum, int nz, const double *tt_us,
                                 const double *profiles, int nprof, const int *col_profile, const double *zgrid,
                                 void *workspace, size_t workspace_bytes, void *stream) {
    return depth_convert<float, double>(x, y, snum, tnum, nz, tt_us, profiles, nprof, col_profile, zgrid, workspace,
                                        workspace_bytes, stream);
}
int impdar_depth_convert_f64(const double *x, double *y, int snum, int tnum, int nz, const double *tt_us,
                             const double *profiles, int nprof, const int *col_profile, const double *zgrid,
                             void *workspace, size_t workspace_bytes, void *stream) {
    return depth_convert<double, double>(x, y, snum, tnum, nz, tt_us, profiles, nprof, col_profile, zgrid, workspace,
                                         workspace_bytes, stream);
}

}  // extern "C"
