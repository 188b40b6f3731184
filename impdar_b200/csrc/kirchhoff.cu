// Kirchhoff diffraction summation (reference: migrationlib/mig_python.py:35-123, C prototype
// migrationlib/mig_cython.h:11).
//
// out[ti, xi] = 1/(2 pi) * nansum_x( gradD[idx(ti,xi,x), x] * cos(theta)/v  [+ data[idx, x] * cos(theta)/r^2] )
//   r = sqrt((dist[x]-dist[xi])^2 + zs[ti]^2), t = 2 r / v, idx = argmin_k |tt[k] - t| (first minimum),
//   terms with t > max(tt) are zeroed (mig_python.py:52), NaN terms are skipped (nansum, :53).
//
// Design (general geometry kernel):
//   * pre-pass: d/dt (np.gradient's stencil, fp64) fused with a transpose to trace-major gradT[x][k],
//     zero-padded past the last sample, so one warp's gather (32 consecutive output samples, one input
//     trace) touches one or two 128-byte lines and is bank/sector conflict free.
//   * main kernel: a warp owns 32 consecutive output samples of one output trace; a CTA owns 8 adjacent
//     output traces, so the 8 warps gather from the same lines.  Per (output sample, input trace) pair the
//     travel time is evaluated in sample units in fp32: q = U^2 + C^2, s = rsqrt(q), f = q*s - U0, the
//     weight U*s/v falls out of the same rsqrt.  The nearest-sample pick round(f) is only trusted when f
//     is further than `delta` from a rounding boundary; the rare ambiguous pairs are queued per warp and
//     re-evaluated with the reference's exact float64 operation sequence (sqrt, div, |tt[k]-t| compares),
//     so the picked sample is the reference's for every pair.
//   * the aperture cut 2r/v > max(tt) is resolved exactly once per output sample (binary search with the
//     float64 predicate over the ascending trace positions), so the inner loop only tests a trace range.
//   * the velocity is one RMS value per output sample, v[ti] (a constant vector is the reference's single vel):
//     every formula above uses v[ti] for the pairs of output row ti.
//   * lateral variant (LAT): V[ti, xi], one of P RMS profiles per output trace (colp[xi]); the warp of trace xi reads
//     its profile's row vectors and its profile's cs / thr, so column xi is the single-profile call bit for bit.
#include <math.h>

#include <cmath>
#include <mutex>
#include <type_traits>
#include <vector>

#include "common.cuh"

namespace impdar {

struct KirchParams {
    const float *gradT;   // (T, SP)
    const float *dataT;   // (T, SP) or null
    float *out;           // (S, ldo)
    const double *dist;   // T  [m]
    const double *tt;     // S  [s]
    const double *zs;     // S  v*tt/2
    const double *zs2;    // S  zs^2
    const double *vs;     // S  RMS velocity of each output row
    const float3 *rowc;   // S  {sigma = (cs_ti / cs)^2, 1/(2 pi v_ti), 4/(v_ti dt)^2/(2 pi)} (kirch_prep_vectors_kernel)
    const int *flags;     // [0] = 1 + the deepest row of the d/dt (or data) image holding a non-finite value, 0 if none
    unsigned long long *stats;  // [0] pairs, [1] exact pairs
    int S, T, SP, ldo, x_begin, x_end;
    unsigned kmax;                         // SP - 1
    double tmax, tt0, inv_dt, cs;          // cs = 2/(vmin*dt_eff): the offset scale of the staged C^2
    float neg_u0, thr;                     // thr = 0.5 - delta; -1 (every pair exact) for non-monotone positions
    int monotone;                       // dist ascending -> per-sample aperture by binary search
    int rowmajor, Tp, Apad;             // table path: gradT/dataT are (S, Tp) row-major, trace x at column Apad + x
    const int *colp;                    // lateral: profile of each output trace (T); zs, zs2, vs, rowc are then (P, S)
    const double2 *pc;                  // lateral: {cs, thr} of each profile
};

#define KIRCH_MAGIC 12582912.0f  // 1.5 * 2^23
#define KIRCH_MAGIC_I 0x4B400000

__device__ __forceinline__ float rsqrt_approx(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// The reference's own float64 sequence for one pair: returns t = 2*sqrt(d^2 + zs2)/vel without contraction
// (vel = v[ti] of the pair's output row).
__device__ __forceinline__ double exact_time(double d, double zs2, double vel, double &rs) {
    rs = __dsqrt_rn(__dadd_rn(__dmul_rn(d, d), zs2));
    return __ddiv_rn(__dmul_rn(2.0, rs), vel);
}

// argmin_k |tt[k] - t| with first-minimum ties, tt ascending.
__device__ __forceinline__ int exact_pick(const double *__restrict__ tt, int S, double t, double tt0,
                                          double inv_dt) {
    double g = (t - tt0) * inv_dt;
    int k = (g < 0.0) ? 0 : ((g > (double)(S - 1)) ? S - 1 : (int)rint(g));
    double dk = fabs(__dsub_rn(tt[k], t));
    while (k > 0) {
        double dm = fabs(__dsub_rn(tt[k - 1], t));
        if (dm <= dk) { dk = dm; --k; } else break;
    }
    while (k < S - 1) {
        double dp = fabs(__dsub_rn(tt[k + 1], t));
        if (dp < dk) { dk = dp; ++k; } else break;
    }
    return k;
}

// roff: offset of the output row's profile in the (P, S) row vectors of the lateral variant (0 otherwise)
template <bool NEAR>
__device__ __forceinline__ float exact_term(const KirchParams &p, int ti, int x, double dxi, size_t roff = 0) {
    const double d = __dsub_rn(p.dist[x], dxi);
    double rs;
    const double vel = (p.vs + roff)[ti];
    const double t = exact_time(d, (p.zs2 + roff)[ti], vel, rs);
    if (t > p.tmax) return 0.f;
    const int k = exact_pick(p.tt, p.S, t, p.tt0, p.inv_dt);
    const double costheta = (p.zs + roff)[ti] / rs;
    const size_t gi = p.rowmajor ? (size_t)k * p.Tp + p.Apad + x : (size_t)x * p.SP + k;
    const double g = (double)p.gradT[gi];
    double term = g * costheta / vel;
    if (term != term) term = 0.0;
    if (NEAR) {
        const double dv = (double)p.dataT[gi];
        double tn = dv * costheta / (rs * rs);
        if (tn == tn) term += tn;
    }
    return (float)(term * 0.15915494309189535);  // 1/(2 pi)
}

#define KQ_CAP 192

// The lateral variant keeps its per-warp profile values in the warp's c2v staging row, after the 32 staged values:
// [32] the fast/exact threshold, [33] the profile index, [34..35] cs (float64).  They are re-read where they are used
// (thr once per group of 4 traces): kept in registers across the trace loop they push the kernel past 64 registers.
constexpr int KL_THR = 32, KL_PROF = 33, KL_CS = 34, KL_ROW = 36;
template <bool LAT>
__device__ __forceinline__ double kirch_cs(const KirchParams &p, const float *sCw) {
    if constexpr (LAT) return *reinterpret_cast<const volatile double *>(sCw + KL_CS);
    else return p.cs;
}

// Fast path over one staged chunk of <= 32 input traces (4 per iteration, straight-line, predicated).
template <bool NEAR, bool STATS, bool HASNAN, bool LAT, typename Flush>
__device__ __forceinline__ void kirch_chunk(Flush &flush, const float *__restrict__ gT, const float *__restrict__ dT,
                                            const float *__restrict__ sCw, int *__restrict__ sQw, int jend,
                                            unsigned rowoff, unsigned SP, unsigned kmax, int rel, unsigned span,
                                            int xb, int lane, float u2, float sigma, float Uw, float Un, float neg_u0, float thr,
                                            float &acc0, float &acc1, int &qn, unsigned &npairs, unsigned &nexact) {
#pragma unroll 1
    for (int j0 = 0; j0 < jend; j0 += 4) {
        if constexpr (LAT) thr = *reinterpret_cast<const volatile float *>(sCw + KL_THR);
        const float4 c4 = *reinterpret_cast<const float4 *>(sCw + j0);
        const float c[4] = {c4.x, c4.y, c4.z, c4.w};
        unsigned amb4 = 0;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            const float q = fmaf(c[jj], sigma, u2);   // u2 + c[jj] exactly when sigma == 1 (constant velocity)
            const float s = rsqrt_approx(q);
            const float f = fmaf(q, s, neg_u0);
            const float r = f + KIRCH_MAGIC;
            const unsigned k = min((unsigned)(__float_as_int(r) - KIRCH_MAGIC_I), kmax);
            const float e = f - (r - KIRCH_MAGIC);
            const bool inr = (unsigned)(rel + j0 + jj) <= span;
            const bool amb = fabsf(e) > thr;
            const unsigned idx = rowoff + (unsigned)jj * SP + k;
            const float g = __ldg(gT + idx);
            const bool ok = inr && !amb;
            if (!HASNAN) {
                // select on the weight so the accumulate is a single FFMA
                const float w = ok ? Uw * s : 0.f;
                if (jj & 1) acc1 = fmaf(g, w, acc1); else acc0 = fmaf(g, w, acc0);
                if (NEAR) {
                    const float dv = __ldg(dT + idx);
                    const float wn = ok ? (Un * s) * (s * s) : 0.f;
                    if (jj & 1) acc1 = fmaf(dv, wn, acc1); else acc0 = fmaf(dv, wn, acc0);
                }
            } else {
                float term = g * (Uw * s);
                if (term != term) term = 0.f;   // nansum skips NaN terms (mig_python.py:53)
                if (NEAR) {
                    const float dv = __ldg(dT + idx);
                    const float tn = dv * ((Un * s) * (s * s));
                    if (tn == tn) term += tn;
                }
                if (jj & 1) acc1 += ok ? term : 0.f; else acc0 += ok ? term : 0.f;
            }
            if (STATS && inr) ++npairs;
            amb4 |= (inr && amb) ? (1u << jj) : 0u;
        }
        rowoff += 4u * SP;
        if (__any_sync(0xffffffffu, amb4 != 0)) {
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const bool a = (amb4 >> jj) & 1u;
                const unsigned m = __ballot_sync(0xffffffffu, a);
                if (a) {
                    sQw[qn + __popc(m & ((1u << lane) - 1u))] = ((xb + j0 + jj) << 5) | lane;
                    ++nexact;
                }
                qn += __popc(m);
            }
            if (qn > 32) {  // keep the queue below KQ_CAP: at most 128 entries are added per group of 4
                __syncwarp();
                flush(qn);
                qn = 0;
            }
        }
    }
}

template <bool NEAR, bool STATS, bool LAT = false>
__global__ void __launch_bounds__(256) kirch_general_kernel(const __grid_constant__ KirchParams p) {
    __shared__ __align__(16) float sC[8][LAT ? KL_ROW : 32];
    __shared__ int sQ[8][KQ_CAP];
    __shared__ float sT[8][32];
    __shared__ int sO[8][32];
    __shared__ float sOut[32][9];

    const int lane = threadIdx.x, warp = threadIdx.y;
    const int ti0 = blockIdx.x * 32;
    const int ti = ti0 + lane;
    const int xi = p.x_begin + blockIdx.y * 8 + warp;
    const bool warp_active = xi < p.x_end;
    const bool active = warp_active && ti < p.S;
    const bool hasnan = p.flags[0] != 0;

    float acc0 = 0.f, acc1 = 0.f, accx = 0.f;
    unsigned npairs = 0, nexact = 0;

    if (warp_active) {
        const double dxi = p.dist[xi];
        // lateral: this trace's profile (its row vectors start at roff); its cs / thr go to shared memory, out of the
        // registers of the trace loop
        const int prof = LAT ? p.colp[xi] : 0;
        const size_t roff = LAT ? (size_t)prof * p.S : 0;
        if constexpr (LAT) {
            if (lane == 0) {
                const double2 pc = p.pc[prof];
                sC[warp][KL_THR] = (float)pc.y;
                reinterpret_cast<int *>(sC[warp])[KL_PROF] = prof;
                *reinterpret_cast<double *>(sC[warp] + KL_CS) = pc.x;
            }
            __syncwarp();
        }
        const int tic = active ? ti : p.S - 1;
        const double Ud = p.tt[tic] * p.inv_dt;
        const float U = (float)Ud;
        const float u2 = fmaxf((float)(Ud * Ud), 1e-30f);  // q == 0 only at the apex of a zero-depth sample (weight 0)

        // exact per-sample aperture [xlo, xhi]: pairs with 2r/v > max(tt) contribute exactly 0
        int xlo = xi + 1, xhi = xi;
        if (active) {
            const double zs2i = (p.zs2 + roff)[ti], vi = (p.vs + roff)[ti];
            double rs;
            if (!(exact_time(0.0, zs2i, vi, rs) > p.tmax)) {
                if (p.monotone) {
                    int a = 0, b = xi;  // smallest x in [0, xi] inside
                    while (a < b) {
                        int m = (a + b) >> 1;
                        if (exact_time(__dsub_rn(p.dist[m], dxi), zs2i, vi, rs) > p.tmax) a = m + 1; else b = m;
                    }
                    xlo = a;
                    a = xi; b = p.T - 1;  // largest x in [xi, T-1] inside
                    while (a < b) {
                        int m = (a + b + 1) >> 1;
                        if (exact_time(__dsub_rn(p.dist[m], dxi), zs2i, vi, rs) > p.tmax) b = m - 1; else a = m;
                    }
                    xhi = a;
                } else {
                    xlo = 0;
                    xhi = p.T - 1;
                }
            }
        }
        int xlo_w = xlo, xhi_w = xhi;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            xlo_w = min(xlo_w, __shfl_xor_sync(0xffffffffu, xlo_w, o));
            xhi_w = max(xhi_w, __shfl_xor_sync(0xffffffffu, xhi_w, o));
        }
        unsigned span = (unsigned)(xhi - xlo);
        if (xhi < xlo) {  // empty aperture: make the range test fail for every x
            span = 0;
            xlo = 0x40000000;
        }
        // Per-row velocity (kirch_prep_vectors_kernel): the staged c2v carries the offset scale cs = 2/(vmin dt) and
        // this row's C^2 is c2v * sigma; the weights are 1/(2 pi v_ti) and 4/(v_ti dt)^2/(2 pi).
        const float3 rc = (p.rowc + roff)[tic];
        const float sigma = rc.x;
        const float Uw = U * rc.y, Un = U * rc.z;
        const unsigned SP = (unsigned)p.SP;
        int qn = 0;

        auto flush = [&](int count) {
            for (int base = 0; base < count; base += 32) {
                float term = 0.f;
                int owner = -1;
                if (base + lane < count) {
                    const int e = sQ[warp][base + lane];
                    owner = e & 31;
                    const size_t ro = LAT ? (size_t)reinterpret_cast<const volatile int *>(sC[warp])[KL_PROF] * p.S : 0;
                    term = exact_term<NEAR>(p, ti0 + owner, e >> 5, dxi, ro);
                }
                sT[warp][lane] = term;
                sO[warp][lane] = owner;
                __syncwarp();
                const int n = min(32, count - base);
                for (int j = 0; j < n; ++j)
                    if (sO[warp][j] == lane) accx += sT[warp][j];
                __syncwarp();
            }
        };

        // One trace loop per variant, chosen once: a non-finite flag kept live across the loop spills a register.
        auto trace_loop = [&](auto nan_variant) {
            for (int xb = xlo_w; xb <= xhi_w; xb += 32) {
                {
                    const int xx = xb + lane;
                    float c2v = 0.f;
                    if (xx <= xhi_w) {
                        const double C = (p.dist[xx] - dxi) * kirch_cs<LAT>(p, sC[warp]);
                        c2v = (float)(C * C);
                    }
                    __syncwarp();
                    sC[warp][lane] = c2v;
                    __syncwarp();
                }
                const int jend = (min(32, xhi_w - xb + 1) + 3) & ~3;   // padded entries fall outside every lane's range
                const unsigned rowoff = (unsigned)xb * SP;
                const int rel = xb - xlo;
                kirch_chunk<NEAR, STATS, decltype(nan_variant)::value, LAT>(
                    flush, p.gradT, p.dataT, sC[warp], sQ[warp], jend, rowoff, SP, p.kmax, rel, span, xb, lane, u2, sigma, Uw,
                    Un, p.neg_u0, LAT ? 0.f : p.thr, acc0, acc1, qn, npairs, nexact);
            }
        };
        if (hasnan) trace_loop(std::true_type{}); else trace_loop(std::false_type{});
        __syncwarp();
        if (qn > 0) flush(qn);
    }

    // transpose the 32x8 tile so that rows of `out` are written in 32-byte runs
    sOut[lane][warp] = acc0 + acc1 + accx;
    __syncthreads();
    {
        const int tid = warp * 32 + lane;
        const int r = tid >> 3, c = tid & 7;
        const int to = ti0 + r, xo = p.x_begin + blockIdx.y * 8 + c;
        if (to < p.S && xo < p.x_end) p.out[(size_t)to * p.ldo + (xo - p.x_begin)] = sOut[r][c];
    }
    if (STATS) {
        unsigned long long np64 = npairs, ne64 = nexact;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            np64 += __shfl_xor_sync(0xffffffffu, np64, o);
            ne64 += __shfl_xor_sync(0xffffffffu, ne64, o);
        }
        if (lane == 0 && np64) {
            atomicAdd(&p.stats[0], np64);
            if (ne64) atomicAdd(&p.stats[1], ne64);
        }
    }
}

// d/dt with np.gradient's stencil (coefficients a,b,c per row; b == 0 in numpy's uniform branch, which
// never touches f[s]) fused with the transpose to trace-major and a non-finite scan.  `data` holds ncols columns
// with row stride ld; gradT / dataT are indexed by the local column.
__global__ void __launch_bounds__(256) grad_transpose_kernel(const float *__restrict__ data,
                                                             float *__restrict__ gradT,
                                                             float *__restrict__ dataT, int S, int ncols, int ld, int SP,
                                                             const double *__restrict__ coef,
                                                             int *__restrict__ flags) {
    __shared__ float tg[32][33];
    __shared__ float td[32][33];
    const int s0 = blockIdx.y * 32, x0 = blockIdx.x * 32;
    int bad = 0;   // 1 + deepest row with a non-finite value
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int s = s0 + r, x = x0 + threadIdx.x;
        float g = 0.f, dv = 0.f;
        if (s < S && x < ncols) {
            const double a = coef[s], b = coef[S + s], c = coef[2 * S + s];
            dv = data[(size_t)s * ld + x];
            double acc = 0.0;
            if (s > 0 && a != 0.0) acc += a * (double)data[(size_t)(s - 1) * ld + x];
            if (b != 0.0) acc += b * (double)dv;
            if (s < S - 1 && c != 0.0) acc += c * (double)data[(size_t)(s + 1) * ld + x];
            g = (float)acc;
            if (!isfinite(g) || !isfinite(dv)) bad = s + 1;
        }
        tg[r][threadIdx.x] = g;
        td[r][threadIdx.x] = dv;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int x = x0 + r, s = s0 + threadIdx.x;
        if (x < ncols && s < S) {
            gradT[(size_t)x * SP + s] = tg[threadIdx.x][r];
            if (dataT) dataT[(size_t)x * SP + s] = td[threadIdx.x][r];
        }
    }
    bad = __reduce_max_sync(0xffffffffu, bad);
    if (bad && threadIdx.x == 0) atomicMax(flags, bad);
}

// Per-row vectors: zs, zs2 (float64, the reference's operation order) and the general kernel's float32 row constants.
// cs_i / cs = 1 exactly when v_ti is the velocity cs was made with, so a constant vector has sigma == 1 and the
// weights are the single-velocity values bit for bit.
__device__ __forceinline__ void kirch_prep_row(int i, const double *__restrict__ tt, const double *__restrict__ vs,
                                               double *__restrict__ zs, double *__restrict__ zs2,
                                               float3 *__restrict__ rowc, double dt_eff, double cs) {
    const double v = vs[i];
    const double z = __ddiv_rn(__dmul_rn(v, tt[i]), 2.0);   // zs = vel * tt_sec / 2.0   (:101)
    zs[i] = z;
    zs2[i] = __dmul_rn(z, z);                                // zs2 = zs**2.              (:102)
    const double vdt = __dmul_rn(v, dt_eff);
    const double sr = __ddiv_rn(__ddiv_rn(2.0, vdt), cs);   // cs_i / cs, cs_i = 2 / (v dt)
    rowc[i] = make_float3((float)__dmul_rn(sr, sr),
                          (float)__ddiv_rn(1.0, __dmul_rn(2.0 * 3.14159265358979323846, v)),
                          (float)__ddiv_rn(__ddiv_rn(4.0, __dmul_rn(vdt, vdt)), 2.0 * 3.14159265358979323846));
}

__global__ void kirch_prep_vectors_kernel(const double *__restrict__ tt, const double *__restrict__ vs,
                                          double *__restrict__ zs, double *__restrict__ zs2, float3 *__restrict__ rowc,
                                          int S, double dt_eff, double cs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < S) kirch_prep_row(i, tt, vs, zs, zs2, rowc, dt_eff, cs);
}

// The same row constants for each of P profiles (lateral variant): profile blockIdx.x, rows of block blockIdx.y, each
// with its own cs = pc[p].x, so a profile's vectors are bit for bit those of a single-profile call.
__global__ void kirch_prep_profiles_kernel(const double *__restrict__ tt, const double *__restrict__ vs,
                                           double *__restrict__ zs, double *__restrict__ zs2, float3 *__restrict__ rowc,
                                           const double2 *__restrict__ pc, int S, double dt_eff) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x;
    const size_t o = (size_t)blockIdx.x * S;
    if (i < S) kirch_prep_row(i, tt, vs + o, zs + o, zs2 + o, rowc + o, dt_eff, pc[blockIdx.x].x);
}

// =====================================================================================================
// Uniform-geometry path.  When traces are equally spaced (after ImpDAR's constant_space interpolation, or any
// synthetic geometry) the travel time of a pair depends only on (output sample ti, trace offset m = |x - xi|),
// so the nearest-sample pick k(ti, m) and the obliquity weight w(ti, m) are the same for every output trace.
// They are tabulated once per call with the reference's float64 sequence (S x aperture entries), and the
// migration becomes out[ti, xi] = sum_m w[ti,m] * (g[k[ti,m], xi-m] + g[k[ti,m], xi+m]): lanes run over
// consecutive output traces, so every gather is a contiguous 128-byte row segment of the (zero-padded,
// row-major) d/dt image and the inner loop is one load + half an FADD/FFMA per pair.
// Table entries whose pick (or aperture cut) could change within the measured deviation of the real trace
// positions from the uniform grid are flagged and re-evaluated per pair by the exact float64 path, so the
// result is again the reference's pick for every pair.
struct KirchTabParams {
    const float *gP;    // (S, Tp): d/dt, trace x at column Apad + x, zero padded
    const float *dP;    // (S, Tp): data (near field) or null
    const int2 *tab;    // [S][A1]: {k or -1 (no contribution) or -2 (ambiguous), bits of the far weight}
    const float *tabn;  // [S][A1]: near-field weight, or null
    const int *nm;      // [S]: number of table entries to visit
    float *out;
    const int *flags;
    unsigned long long *stats;
    int S, T, Tp, Apad, A1, ldo, x_begin, x_end;
    int s_begin, s_end;  // output rows of this launch (the host pipeline runs the image in row chunks)
    const int *only_if;  // non-null: the launch stands in for the tile kernel: every row when *only_if is set (wide
                         // intervals), otherwise only the rows that read non-finite input (ti < flags[0])
};

__global__ void __launch_bounds__(128) kirch_table_build_kernel(int2 *__restrict__ tab, float *__restrict__ tabn,
                                                                int *__restrict__ nm, int S, int A1, double dxm,
                                                                const double *__restrict__ zs,
                                                                const double *__restrict__ zs2,
                                                                const double *__restrict__ tt,
                                                                const double *__restrict__ vs, double tmax,
                                                                double tt0, double inv_dt, double eps_t,
                                                                int *__restrict__ amb_list, int *__restrict__ amb_count) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    const int ti = blockIdx.y;
    if (m >= A1) return;
    const double d = (double)m * dxm;
    const double vel = vs[ti];
    double rs;
    const double t = exact_time(d, zs2[ti], vel, rs);
    int k = -1;
    float w = 0.f, wn = 0.f;
    const bool in_lo = !((t - eps_t) > tmax), in_hi = !((t + eps_t) > tmax);
    if (in_lo) {
        if (!in_hi) {
            k = -2;
        } else {
            const int k_lo = exact_pick(tt, S, t - eps_t, tt0, inv_dt);
            const int k_hi = exact_pick(tt, S, t + eps_t, tt0, inv_dt);
            k = (k_lo == k_hi) ? exact_pick(tt, S, t, tt0, inv_dt) : -2;
        }
        const double costheta = zs[ti] / rs;
        const double wf = costheta / vel * 0.15915494309189535;
        const double wq = costheta / (rs * rs) * 0.15915494309189535;
        if (wf != wf) {
            k = -1;  // 0/0 at the apex of a zero-depth sample: nansum drops the term (mig_python.py:53)
        } else {
            w = (float)wf;
            wn = (float)wq;
        }
    }
    tab[(size_t)ti * A1 + m] = make_int2(k, __float_as_int(w));
    if (tabn) tabn[(size_t)ti * A1 + m] = wn;
    if (k != -1) atomicMax(&nm[ti], m + 1);
    if (k == -2) amb_list[atomicAdd(amb_count, 1)] = ti * A1 + m;  // list has room for every entry
}

// d/dt (np.gradient stencil) into the padded row-major layout; also the non-finite scan, which records the deepest
// row of the padded images holding a non-finite value (flags[0] = 1 + row).  An output row ti reads only rows >= ti
// of those images, so "flags[0] > ti" is known as soon as the rows >= ti are built: a bottom-up sequence of row chunks
// takes every per-row decision that depends on it exactly as one launch over the whole image does.  `data` holds the radargram
// columns [c0, c0 + ncols) with row stride ld (the whole image: c0 = 0, ncols = ld = T); trace x lands at column
// aoff + x of the padded image (aoff = Apad - c0).
__global__ void __launch_bounds__(256) grad_padded_kernel(const float *__restrict__ data, float *__restrict__ gP,
                                                          float *__restrict__ dP, int S, int c0, int ncols, int ld,
                                                          int Tp, int aoff, const double *__restrict__ coef,
                                                          int *__restrict__ flags, int s0, int vec4) {
    const int s = s0 + blockIdx.y;
    const double a = coef[s], b = coef[S + s], c = coef[2 * S + s];
    bool bad = false;
    if (vec4) {
        // four columns per thread through 128-bit accesses (same arithmetic per element); the host checks alignment
        const float4 *__restrict__ r0 = reinterpret_cast<const float4 *>(data + (size_t)s * ld);
        const float4 *__restrict__ rm = reinterpret_cast<const float4 *>(data + (size_t)(s > 0 ? s - 1 : s) * ld);
        const float4 *__restrict__ rp = reinterpret_cast<const float4 *>(data + (size_t)(s < S - 1 ? s + 1 : s) * ld);
        float4 *__restrict__ go = reinterpret_cast<float4 *>(gP + (size_t)s * Tp + aoff + c0);
        float4 *__restrict__ dout = dP ? reinterpret_cast<float4 *>(dP + (size_t)s * Tp + aoff + c0) : nullptr;
        const bool um = s > 0 && a != 0.0, u0 = b != 0.0, up = s < S - 1 && c != 0.0;
        for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < ncols / 4; j += gridDim.x * blockDim.x) {
            const float4 d0 = r0[j];
            const float4 dm = um ? rm[j] : d0, dq = up ? rp[j] : d0;
            const float v0[4] = {d0.x, d0.y, d0.z, d0.w}, vm[4] = {dm.x, dm.y, dm.z, dm.w}, vp[4] = {dq.x, dq.y, dq.z, dq.w};
            float g[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                double acc = 0.0;
                if (um) acc += a * (double)vm[i];
                if (u0) acc += b * (double)v0[i];
                if (up) acc += c * (double)vp[i];
                g[i] = (float)acc;
                if (!isfinite(g[i]) || !isfinite(v0[i])) bad = true;
            }
            go[j] = make_float4(g[0], g[1], g[2], g[3]);
            if (dout) dout[j] = d0;
        }
        if (__syncthreads_or(bad) && threadIdx.x == 0) atomicMax(flags, s + 1);   // deepest non-finite row
        return;
    }
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < ncols; j += gridDim.x * blockDim.x) {
        const float dv = data[(size_t)s * ld + j];
        double acc = 0.0;
        if (s > 0 && a != 0.0) acc += a * (double)data[(size_t)(s - 1) * ld + j];
        if (b != 0.0) acc += b * (double)dv;
        if (s < S - 1 && c != 0.0) acc += c * (double)data[(size_t)(s + 1) * ld + j];
        const float g = (float)acc;
        if (!isfinite(g) || !isfinite(dv)) bad = true;
        gP[(size_t)s * Tp + aoff + c0 + j] = g;
        if (dP) dP[(size_t)s * Tp + aoff + c0 + j] = dv;
    }
    if (__syncthreads_or(bad) && threadIdx.x == 0) atomicMax(flags, s + 1);   // deepest non-finite row
}

constexpr int KT_R = 4;  // output traces per thread (stride 32)

template <bool NEAR, bool HASNAN, bool STATS, bool APEX>
__device__ __forceinline__ void kirch_table_step(const KirchTabParams &p, const float *__restrict__ gbase,
                                                 const float *__restrict__ dbase, int2 e, float wn, int m, int xbase,
                                                 float (&acc)[KT_R], unsigned &npairs) {
    const float w = __int_as_float(e.y);
    const long long row = (long long)e.x * p.Tp;
    const float *__restrict__ pl = gbase + (row - m);
    const float *__restrict__ pr = gbase + (row + m);
    const float *__restrict__ ql = NEAR ? dbase + (row - m) : nullptr;
    const float *__restrict__ qr = NEAR ? dbase + (row + m) : nullptr;
#pragma unroll
    for (int r = 0; r < KT_R; ++r) {
        const float gl = __ldg(pl + 32 * r);
        const float gr = APEX ? 0.f : __ldg(pr + 32 * r);
        if (!HASNAN) {
            acc[r] = fmaf(w, APEX ? gl : gl + gr, acc[r]);
            if (NEAR) {
                const float dl = __ldg(ql + 32 * r);
                const float dr = APEX ? 0.f : __ldg(qr + 32 * r);
                acc[r] = fmaf(wn, APEX ? dl : dl + dr, acc[r]);
            }
        } else {
            const float tl = w * gl, tr = w * gr;   // nansum: NaN terms are skipped one by one
            if (tl == tl) acc[r] += tl;
            if (!APEX && tr == tr) acc[r] += tr;
            if (NEAR) {
                const float ul = wn * __ldg(ql + 32 * r);
                const float ur = APEX ? 0.f : wn * __ldg(qr + 32 * r);
                if (ul == ul) acc[r] += ul;
                if (!APEX && ur == ur) acc[r] += ur;
            }
        }
        if (STATS) {
            const int x = xbase + 32 * r;
            if (x < p.x_end) npairs += (x - m >= 0) + (!APEX && x + m < p.T);
        }
    }
}

template <bool NEAR, bool HASNAN, bool STATS>
__device__ __forceinline__ void kirch_table_loop(const KirchTabParams &p, int ti, int xbase, float (&acc)[KT_R],
                                                 unsigned &npairs) {
    const int n = p.nm[ti];
    const int2 *__restrict__ trow = p.tab + (size_t)ti * p.A1;
    const float *__restrict__ nrow = NEAR ? p.tabn + (size_t)ti * p.A1 : nullptr;
    // lanes past the end of the profile read the zero padding (rows are over-allocated by one tile)
    const float *__restrict__ gbase = p.gP + (p.Apad + xbase);
    const float *__restrict__ dbase = NEAR ? p.dP + (p.Apad + xbase) : nullptr;
    if (n > 0) {
        const int2 e = __ldg(trow);
        if (e.x >= 0)
            kirch_table_step<NEAR, HASNAN, STATS, true>(p, gbase, dbase, e, NEAR ? __ldg(nrow) : 0.f, 0, xbase, acc, npairs);
    }
#pragma unroll 2
    for (int m = 1; m < n; ++m) {
        const int2 e = __ldg(trow + m);
        if (e.x < 0) continue;  // uniform: no contribution, or ambiguous (exact fix-up pass)
        kirch_table_step<NEAR, HASNAN, STATS, false>(p, gbase, dbase, e, NEAR ? __ldg(nrow + m) : 0.f, m, xbase, acc, npairs);
    }
}

template <bool NEAR, bool STATS>
__global__ void __launch_bounds__(128) kirch_table_kernel(const __grid_constant__ KirchTabParams p) {
    // Rows ti < nan_end read a non-finite value somewhere (the nansum variant); the tile kernel leaves them to this one.
    const int nan_end = p.flags[0];
    const int s_end = (p.only_if && !p.only_if[0]) ? min(p.s_end, nan_end) : p.s_end;
    if (s_end <= p.s_begin) return;   // the tile kernel has done these rows
    // Work item = (row, block of 4 x 32 KT_R output traces), rows fastest.  The grid holds every item when this kernel
    // is the one that does the work; as the tile kernel's stand-in it is a small grid that strides over the items
    // (half a million CTAs that only test the flag and leave cost 0.5 ms at 65536 x 8192).
    const int nrows = s_end - p.s_begin;
    const int ntx = (p.x_end - p.x_begin + 4 * 32 * KT_R - 1) / (4 * 32 * KT_R);
    const long long nitems = (long long)nrows * ntx;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (long long it = blockIdx.x; it < nitems; it += gridDim.x) {
        const int ti = p.s_begin + (int)(it % nrows);
        const int xbase = p.x_begin + ((int)(it / nrows) * 4 + warp) * (32 * KT_R) + lane;
        if (xbase - lane >= p.x_end) continue;
        float acc[KT_R];
#pragma unroll
        for (int r = 0; r < KT_R; ++r) acc[r] = 0.f;
        unsigned npairs = 0;
        if (ti < nan_end)
            kirch_table_loop<NEAR, true, STATS>(p, ti, xbase, acc, npairs);
        else
            kirch_table_loop<NEAR, false, STATS>(p, ti, xbase, acc, npairs);
#pragma unroll
        for (int r = 0; r < KT_R; ++r) {
            const int x = xbase + 32 * r;
            if (x < p.x_end) p.out[(size_t)ti * p.ldo + (x - p.x_begin)] = acc[r];
        }
        if (STATS) {
            unsigned long long np64 = npairs;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) np64 += __shfl_xor_sync(0xffffffffu, np64, o);
            if (lane == 0 && np64) atomicAdd(&p.stats[0], np64);
        }
    }
}

// Exact float64 re-evaluation of every pair that uses a flagged table entry (normally a handful: the apex of
// the last sample sits exactly on the aperture cut).  Work item = (flagged entry, block of 32 output traces).
template <bool NEAR>
__global__ void __launch_bounds__(256) kirch_table_fixup_kernel(const __grid_constant__ KirchTabParams tp,
                                                                const __grid_constant__ KirchParams gp,
                                                                const int *__restrict__ amb_list,
                                                                const int *__restrict__ amb_count) {
    const int lane = threadIdx.x & 31;
    const int nblk = (tp.x_end - tp.x_begin + 31) / 32;
    const int count = *amb_count;
    const int wid = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int nwarps = (int)(((long long)gridDim.x * blockDim.x) >> 5);
    // Entries outside this launch's row range are skipped with one load each (row-chunked launches would otherwise
    // walk the whole (entry, block) space every time); an in-range entry is spread over `split` warps (8 when the
    // list is long, up to one warp per block when it is short: one entry x 2048 blocks on 8 warps took 0.42 ms).
    int split = nwarps / (count > 0 ? count : 1);   // a handful of entries (the usual case): all warps share their blocks
    split = split < 8 ? 8 : (split > nblk ? nblk : split);
    if (split < 1) split = 1;
    for (long long it = wid; it < (long long)count * split; it += nwarps) {
        const int e = amb_list[it / split];
        const int ti = e / tp.A1, m = e % tp.A1;
        if (ti < tp.s_begin || ti >= tp.s_end) continue;
        for (int blk = (int)(it % split); blk < nblk; blk += split) {
            const int xi = tp.x_begin + blk * 32 + lane;
            if (xi >= tp.x_end) continue;
            const double dxi = gp.dist[xi];
            float term = 0.f;
            if (xi - m >= 0) term += exact_term<NEAR>(gp, ti, xi - m, dxi);
            if (m != 0 && xi + m < tp.T) term += exact_term<NEAR>(gp, ti, xi + m, dxi);
            if (term != 0.f) atomicAdd(&tp.out[(size_t)ti * tp.ldo + (xi - tp.x_begin)], term);
            if (tp.stats) atomicAdd(&tp.stats[1], 1ull);
        }
    }
}

}  // namespace impdar
#include "kirchhoff_tile.cuh"
namespace impdar {

static inline int kirch_sp(int S) { return ((S + 64 + 31) / 32) * 32; }

// Per-run path of the lateral entry: folds one run's non-finite / stand-down flags and pair counters into the summary
// block (same layout as the flags block: [0] any run left work to the gather kernel, +128 pairs, exact pairs).
__global__ void kirch_run_summary_kernel(const int *__restrict__ flags, int *__restrict__ sum) {
    if (threadIdx.x == 0) {
        if (flags[0] | flags[16]) sum[0] = 1;
        const unsigned long long *st = reinterpret_cast<const unsigned long long *>(flags + 32);
        unsigned long long *acc = reinterpret_cast<unsigned long long *>(sum + 32);
        acc[0] += st[0];
        acc[1] += st[1];
    }
}

// float32 rows -> float64 rows (the reference returns float64, mig_python.py:95/:118); runs on the download stream
__global__ void __launch_bounds__(256) widen_f32_f64_kernel(const float *__restrict__ x, double *__restrict__ y, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        y[i] = (double)x[i];
}

// Host-to-host pipeline state (impdar_kirchhoff_host_pipelined_f64): an output row ti only reads input rows >= ti - 1
// (the diffraction hyperbola runs downwards in time), so the image is processed bottom-up in row chunks:
// upload chunk j-1 | d/dt + diffraction sum of chunk j | widen + download chunk j+1 on three streams.
constexpr int KP_MAX_CHUNKS = 32;
struct KirchPipe {
    const float *h_in;   // host (pinned for a truly asynchronous copy), (S, T)
    double *h_out;       // host, (S, T)
    float *d_in;         // device (S, T)
    double *d_stage;     // device (S, T)
    int nchunks;
    cudaStream_t up, down;
    cudaEvent_t ev_up[KP_MAX_CHUNKS], ev_done[KP_MAX_CHUNKS], ev_entry, ev_exit;
};
// Row-range call (impdar_kirchhoff_rows_f32): output rows [s_begin, s_end) only; d/dt rows [g_hi, snum) are already in
// the workspace from the previous call of the same bottom-up sequence (g_hi == snum: first call, full preparation).
struct KirchRows {
    int s_begin, s_end, g_hi;
};
// Column window of the input (impdar_kirchhoff_window_f32): `data` holds radargram columns [col0, col0 + ncols), row
// stride ld; `out` has row stride ldo.  any_order: the window is the whole image, so trace positions need not ascend.
struct KirchWindow {
    int col0, ncols, ld, ldo;
    bool any_order;
};
// Lateral velocity (impdar_kirchhoff_window_vxz_f32, general-kernel side): P RMS profiles (host, (P, S)), the profile of
// each trace (host, T), each profile's smallest velocity and whether it is constant; `block` is the device area after
// the single-profile workspace (kirch_lateral_block_bytes).
struct KirchLateral {
    const double *profiles;
    int P;
    const int *colp;
    const double *vmin;
    const unsigned char *vconst;
    char *block;
};
static inline size_t kirch_a256(size_t v) { return (v + 255) / 256 * 256; }
static size_t kirch_lateral_block_bytes(int S, int T, int P) {
    const size_t ps = (size_t)P * (size_t)S;
    // run summary (flags | stats) | {cs, thr} per profile | trace -> profile | v, zs, zs2 | float3 row constants
    return 256 + 256 + kirch_a256((size_t)P * sizeof(double2)) + kirch_a256((size_t)T * sizeof(int)) +
           3 * kirch_a256(ps * sizeof(double)) + kirch_a256(ps * sizeof(float3));
}
// Side streams and events of the host pipeline: one set per device, created on first use under a lock.  Selection
// switches and "last call" records are per host thread (SURVEY.md 8b: one host thread - or process - per GPU).
constexpr int KP_MAX_DEVICES = 64;
static KirchPipe g_pipes[KP_MAX_DEVICES];
static bool g_pipe_ready[KP_MAX_DEVICES];
static std::mutex g_pipe_mu;
static int kirch_pipe_streams(KirchPipe **out) {
    int dev = 0;
    IMPDAR_CUDA(cudaGetDevice(&dev));
    IMPDAR_CHECK_ARG(dev >= 0 && dev < KP_MAX_DEVICES, "kirchhoff_host_pipelined: device index %d out of range", dev);
    std::lock_guard<std::mutex> lk(g_pipe_mu);
    KirchPipe &pp = g_pipes[dev];
    if (!g_pipe_ready[dev]) {
        IMPDAR_CUDA(cudaStreamCreateWithFlags(&pp.up, cudaStreamNonBlocking));
        IMPDAR_CUDA(cudaStreamCreateWithFlags(&pp.down, cudaStreamNonBlocking));
        for (int i = 0; i < KP_MAX_CHUNKS; ++i) {
            IMPDAR_CUDA(cudaEventCreateWithFlags(&pp.ev_up[i], cudaEventDisableTiming));
            IMPDAR_CUDA(cudaEventCreateWithFlags(&pp.ev_done[i], cudaEventDisableTiming));
        }
        IMPDAR_CUDA(cudaEventCreateWithFlags(&pp.ev_entry, cudaEventDisableTiming));
        IMPDAR_CUDA(cudaEventCreateWithFlags(&pp.ev_exit, cudaEventDisableTiming));
        g_pipe_ready[dev] = true;
    }
    *out = &pp;
    return IMPDAR_B200_OK;
}

// Geometry vectors (travel times, d/dt coefficients, per-row velocities, trace positions) go up through a small ring of page-locked staging
// buffers per device: an asynchronous copy from pageable memory makes the HOST wait until the stream has drained, which
// kept the caller from enqueueing the next call (or the next step of a multi-GPU pipeline) while this one runs.
constexpr int KV_SLOTS = 4;
struct KirchVecSlot {
    void *host;
    size_t cap;
    cudaEvent_t ev;
    bool used;
};
struct KirchVecRing {
    KirchVecSlot slot[KV_SLOTS];
    int next;
};
static KirchVecRing g_vecs[KP_MAX_DEVICES];
static int kirch_stage_vectors(const double *tt, const double *coef, const double *vel_s, const double *dist, int S, int T,
                               double *d_dst, cudaStream_t st) {
    int dev = 0;
    IMPDAR_CUDA(cudaGetDevice(&dev));
    IMPDAR_CHECK_ARG(dev >= 0 && dev < KP_MAX_DEVICES, "kirchhoff: device index %d out of range", dev);
    const size_t bytes = ((size_t)5 * S + (size_t)T) * sizeof(double);
    std::lock_guard<std::mutex> lk(g_pipe_mu);
    KirchVecRing &ring = g_vecs[dev];
    KirchVecSlot &sl = ring.slot[ring.next];
    ring.next = (ring.next + 1) % KV_SLOTS;
    if (sl.used) IMPDAR_CUDA(cudaEventSynchronize(sl.ev));   // the copy that last read this slot has run
    if (!sl.ev) IMPDAR_CUDA(cudaEventCreateWithFlags(&sl.ev, cudaEventDisableTiming));
    if (sl.cap < bytes) {
        if (sl.host) IMPDAR_CUDA(cudaFreeHost(sl.host));
        sl.host = nullptr;
        sl.cap = 0;
        IMPDAR_CUDA(cudaHostAlloc(&sl.host, bytes, cudaHostAllocDefault));
        sl.cap = bytes;
    }
    double *h = (double *)sl.host;
    memcpy(h, tt, (size_t)S * sizeof(double));
    memcpy(h + S, coef, (size_t)3 * S * sizeof(double));
    memcpy(h + (size_t)4 * S, vel_s, (size_t)S * sizeof(double));
    memcpy(h + (size_t)5 * S, dist, (size_t)T * sizeof(double));
    IMPDAR_CUDA(cudaMemcpyAsync(d_dst, h, bytes, cudaMemcpyHostToDevice, st));
    IMPDAR_CUDA(cudaEventRecord(sl.ev, st));
    sl.used = true;
    return IMPDAR_B200_OK;
}

static thread_local unsigned long long *g_last_stats = nullptr;
static thread_local const int *g_last_flags = nullptr;
static thread_local cudaStream_t g_last_stats_stream = nullptr;
static thread_local int g_stats_enabled = 0;
static thread_local int g_kirch_mode = 0;   // 0 auto, 1 general, 2 table path (tile kernel where it applies), 3 table path, gather kernel only
static thread_local int g_last_path = 0;    // 1 general, 2 table (gather kernel), 3 table (tile kernel launched)

static bool g_tile_attr[KP_MAX_DEVICES];

}  // namespace impdar

using namespace impdar;

extern "C" {

static inline size_t kirch_roundup(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Farthest trace offset a pair can have on a uniform grid of spacing dxm: 2 r / v <= tmax  =>  m dxm <= v tmax / 2
static inline int kirch_amax(int T, double vel, double tmax, double dxm) {
    int Amax = (int)fmin((double)(T - 1), floor(vel * tmax / 2.0 / dxm) + 2.0);
    return Amax < 0 ? 0 : Amax;
}

size_t impdar_kirchhoff_workspace_bytes(int S, int T, int nearfield) {
    const size_t nf = nearfield ? 2 : 1;
    // general path: trace-major d/dt (and data) with padded samples and 32 spare traces
    const size_t general = (size_t)(T + 32) * (size_t)kirch_sp(S) * sizeof(float) * nf;
    // uniform-geometry path, worst case aperture = the whole profile: padded row-major image(s) + tables + schedule
    const size_t tp = kirch_roundup((size_t)T + 2 * kirch_roundup((size_t)T, 32), 32);
    const size_t nblk = (size_t)(S + KT_Q - 1) / KT_Q + KP_MAX_CHUNKS;
    const size_t table = ((size_t)S * tp + 4096) * sizeof(float) * nf + (size_t)S * (size_t)T * (sizeof(int2) + sizeof(int) + (nearfield ? 4 : 0)) +
                         (size_t)S * sizeof(int) + nblk * ((size_t)S * sizeof(int2) + sizeof(int)) + 1024;
    size_t b = general > table ? general : table;
    b += 9 * (size_t)S * sizeof(double);  // zs, zs2, general-kernel row constants, tt, grad coefficients, velocity
    b += (size_t)T * sizeof(double);      // dist
    return b + 4096;
}

// Per-row velocity vectors of the _vz entries: finite and > 0; returns the largest (it bounds the reach of every pair).
static int kirch_vel_range(const double *vel_s, int S, double *vmax) {
    IMPDAR_CHECK_ARG(vel_s, "kirchhoff: null velocity vector");
    double hi = vel_s[0];
    for (int i = 0; i < S; ++i) {
        IMPDAR_CHECK_ARG(std::isfinite(vel_s[i]) && vel_s[i] > 0.0,
                         "kirchhoff: velocity[%d] = %g must be finite and positive", i, vel_s[i]);
        hi = fmax(hi, vel_s[i]);
    }
    *vmax = hi;
    return IMPDAR_B200_OK;
}

int impdar_kirchhoff_input_window(int S, int T, const double *dist_m, const double *tt_s, double vel, int x_begin,
                                  int x_end, int *col0, int *col1) {
    // vel is the largest velocity of the rows (the reach of a pair grows with it)
    IMPDAR_CHECK_ARG(dist_m && tt_s && col0 && col1, "kirchhoff_input_window: null pointer");
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1 && 0 <= x_begin && x_begin < x_end && x_end <= T, "kirchhoff_input_window: bad range");
    double tmax = tt_s[0];
    for (int i = 1; i < S; ++i) tmax = fmax(tmax, tt_s[i]);
    bool monotone = true;
    for (int i = 1; i < T; ++i)
        if (!(dist_m[i] >= dist_m[i - 1])) { monotone = false; break; }
    *col0 = 0;
    *col1 = T;
    if (!monotone || !(tmax > 0.0) || T < 2) return IMPDAR_B200_OK;
    // by distance (any monotone geometry): |d| <= v tmax / 2, with a relative margin and two traces of slack
    const double reach = vel * tmax / 2.0 * (1.0 + 1e-9);
    int lo = x_begin, hi = x_end - 1;
    while (lo > 0 && dist_m[x_begin] - dist_m[lo - 1] <= reach) --lo;
    while (hi < T - 1 && dist_m[hi + 1] - dist_m[x_end - 1] <= reach) ++hi;
    // by trace count on the fitted uniform grid (what the table path reads): Amax offsets each side
    const double dxm = (dist_m[T - 1] - dist_m[0]) / (double)(T - 1);
    if (dxm > 0.0) {
        const int Amax = kirch_amax(T, vel, tmax, dxm);
        lo = lo < x_begin - Amax ? lo : x_begin - Amax;
        hi = hi > x_end - 1 + Amax ? hi : x_end - 1 + Amax;
    }
    lo -= 2;
    hi += 2;
    lo = lo < 0 ? 0 : lo & ~3;                      // whole groups of four columns: the window's rows stay 16-byte
    int end = (hi + 1 + 3) & ~3;                    // aligned in the image and in a packed copy (128-bit d/dt pass)
    *col0 = lo;
    *col1 = end > T ? T : end;
    return IMPDAR_B200_OK;
}

// Uniform trace spacing?  Deviation of the real positions from the fitted grid, in seconds of travel time (vmin: the
// smallest velocity, whose travel time changes most per metre of position error).  uniform_ok admits the table path.
struct KirchSpacing {
    double dxm, eps_t;
    bool uniform_ok;
};
static KirchSpacing kirch_spacing(int S, int T, const double *h_dist, const double *h_tt, double vmin, bool monotone) {
    double tmax = h_tt[0];
    for (int i = 0; i < S; ++i) tmax = fmax(tmax, h_tt[i]);
    const double tt0 = h_tt[0];
    const double dt_eff = (h_tt[S - 1] - h_tt[0]) / (double)(S - 1);
    double dxm = 0.0, maxdev_d = 0.0;
    if (T > 1) {
        dxm = (h_dist[T - 1] - h_dist[0]) / (double)(T - 1);
        for (int i = 0; i < T; ++i) {
            const double dev = fabs(h_dist[i] - (h_dist[0] + i * dxm));
            if (dev > maxdev_d) maxdev_d = dev;
        }
    }
    const double eps_t = (2.0 / vmin) * (2.0 * maxdev_d) + 1e-15 * (fabs(tmax) + fabs(tt0));
    return {dxm, eps_t, monotone && T > 1 && dxm > 0.0 && tmax > 0.0 && eps_t / dt_eff < 1e-5};
}

static bool kirch_monotone(int T, const double *h_dist) {
    for (int i = 1; i < T; ++i)
        if (!(h_dist[i] >= h_dist[i - 1])) return false;
    return true;
}

static int kirchhoff_impl(const float *data, float *out, int S, int T, const double *dist_m, const double *tt_s,
                          const double *grad_coef, const double *vel_s, int nearfield, int x_begin, int x_end,
                          void *workspace, size_t ws_bytes, void *stream, const KirchPipe *pipe,
                          const KirchRows *rows = nullptr, const KirchWindow *win = nullptr,
                          const KirchLateral *lat = nullptr) {
    IMPDAR_CHECK_ARG(data && out && dist_m && tt_s && grad_coef && vel_s, "kirchhoff: null pointer");
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1, "kirchhoff: need snum >= 2, tnum >= 1");
    IMPDAR_CHECK_ARG(0 <= x_begin && x_begin < x_end && x_end <= T, "kirchhoff: bad output range [%d, %d)",
                     x_begin, x_end);
    double vmin = vel_s[0], vmax = vel_s[0];
    for (int i = 0; i < S; ++i) {
        IMPDAR_CHECK_ARG(vel_s[i] > 0.0, "kirchhoff: vel must be positive");
        vmin = fmin(vmin, vel_s[i]);
        vmax = fmax(vmax, vel_s[i]);
    }
    const bool vconst = vmin == vmax;
    IMPDAR_CHECK_ARG(T < (1 << 26), "kirchhoff: tnum too large");
    const size_t need = impdar_kirchhoff_workspace_bytes(S, T, nearfield);
    IMPDAR_CHECK_ARG(workspace && ws_bytes >= need, "kirchhoff: workspace too small (%zu < %zu)", ws_bytes, need);
    cudaStream_t st = (cudaStream_t)stream;
    const int c0 = win ? win->col0 : 0, ncols = win ? win->ncols : T, ld = win ? win->ld : T;
    const int ldo = win ? win->ldo : x_end - x_begin;
    if (win) {
        IMPDAR_CHECK_ARG(c0 >= 0 && ncols >= 1 && c0 + ncols <= T && ld >= ncols && ldo >= x_end - x_begin,
                         "kirchhoff_window: bad column window [%d, %d) / strides", c0, c0 + ncols);
        int need0 = 0, need1 = T;
        int rcw = impdar_kirchhoff_input_window(S, T, dist_m, tt_s, vmax, x_begin, x_end, &need0, &need1);
        if (rcw) return rcw;
        IMPDAR_CHECK_ARG(c0 <= need0 && c0 + ncols >= need1,
                         "kirchhoff_window: output traces [%d, %d) read input columns [%d, %d), the window holds [%d, %d)",
                         x_begin, x_end, need0, need1, c0, c0 + ncols);
    }

    const double *h_tt = tt_s, *h_dist = dist_m;  // HOST vectors (small); device copies live in the workspace
    double tmax = h_tt[0];
    bool ascending = true;
    for (int i = 0; i < S; ++i) {
        if (h_tt[i] > tmax) tmax = h_tt[i];
        if (i > 0 && !(h_tt[i] > h_tt[i - 1])) ascending = false;
    }
    IMPDAR_CHECK_ARG(ascending, "kirchhoff: travel_time must be strictly ascending");
    const double tt0 = h_tt[0];
    const double dt_eff = (h_tt[S - 1] - h_tt[0]) / (double)(S - 1);
    double maxdev = 0.0;
    for (int i = 0; i < S; ++i) {
        const double dev = fabs(h_tt[i] - (tt0 + i * dt_eff));
        if (dev > maxdev) maxdev = dev;
    }
    const int monotone = kirch_monotone(T, h_dist) ? 1 : 0;
    // fp32 error budget of f = sqrt(U^2 + C^2) - U0 (sample units): ~4 ulp relative on a value <= S + |U0|,
    // plus the deviation of tt from a uniform grid.
    const double u0 = tt0 / dt_eff;
    // A per-row velocity adds one rounding: q = fmaf(c2v, sigma, u2) with sigma = (v_min / v_i)^2 rounded to float,
    // i.e. <= 2^-24 more relative error on the C^2 part of q (<= q), <= 2^-25 sqrt(q) <= 3e-8 (S + |U0|) on f after the
    // square root.  A constant vector has sigma == 1 exactly (no extra rounding) and keeps the budget above unchanged.
    const double delta0 = 6e-7 * ((double)S + fabs(u0) + 64.0) + 2.0 * maxdev / dt_eff + 1e-6;
    const double delta_vz = 6e-8 * ((double)S + fabs(u0) + 64.0);   // non-constant velocity only
    auto fast_thr = [&](bool constant_velocity) {
        const double delta = constant_velocity ? delta0 : delta0 + delta_vz;
        return delta > 0.2 ? -1.f : (float)(0.5 - delta);   // irregular sampling: everything through the exact path
    };
    const float thr = fast_thr(vconst);

    const KirchSpacing spacing = kirch_spacing(S, T, h_dist, h_tt, vmin, monotone);
    const double dxm = spacing.dxm, eps_t = spacing.eps_t;
    const bool uniform_ok = spacing.uniform_ok;
    IMPDAR_CHECK_ARG(lat || !(g_kirch_mode >= 2 && !uniform_ok),
                     "kirchhoff: table path forced but trace spacing is not uniform");
    const bool use_table = !lat && ((g_kirch_mode >= 2) || (g_kirch_mode == 0 && uniform_ok));
    IMPDAR_CHECK_ARG(!(win && !monotone && !win->any_order), "kirchhoff_window: trace positions must be ascending");

    // carve workspace: small vectors first
    char *w = (char *)workspace;
    w = (char *)(((uintptr_t)w + 255) & ~(uintptr_t)255);
    double *zs = (double *)w;
    w += (size_t)S * sizeof(double);
    double *zs2 = (double *)w;
    w += (size_t)S * sizeof(double);
    float3 *rowc = (float3 *)w;
    w += (size_t)S * 2 * sizeof(double);
    double *d_tt = (double *)w;
    w += (size_t)S * sizeof(double);
    double *d_coef = (double *)w;
    w += 3 * (size_t)S * sizeof(double);
    double *d_vel = (double *)w;
    w += (size_t)S * sizeof(double);
    double *d_dist = (double *)w;
    w += (size_t)T * sizeof(double);
    int *flags = (int *)w;                         // [0] non-finite input, [8] ambiguous-entry count, [16] tile stand-down
    unsigned long long *stats = (unsigned long long *)(w + 128);
    w += 256;
    w = (char *)(((uintptr_t)w + 255) & ~(uintptr_t)255);
    const bool continuing = rows && rows->g_hi < S;   // later call of a bottom-up row sequence: flags, tables, tile schedule, d/dt rows
    if (!continuing) {                                // and the vectors stay (same workspace, same stream)
        // d_tt | d_coef (3 S) | d_vel | d_dist are contiguous in the workspace: one copy from the page-locked staging slot
        int rcv = kirch_stage_vectors(tt_s, grad_coef, vel_s, dist_m, S, T, d_tt, st);
        if (rcv) return rcv;
        IMPDAR_CUDA(cudaMemsetAsync(flags, 0, 256, st));
        if (!lat) {
            kirch_prep_vectors_kernel<<<(S + 255) / 256, 256, 0, st>>>(d_tt, d_vel, zs, zs2, rowc, S, dt_eff, 2.0 / (vmin * dt_eff));
            IMPDAR_LAUNCH_CHECK();
        }
    }

    KirchParams p;
    memset(&p, 0, sizeof(p));
    p.out = out; p.dist = d_dist; p.tt = d_tt; p.zs = zs; p.zs2 = zs2; p.vs = d_vel; p.rowc = rowc;
    p.flags = flags; p.stats = stats;
    p.S = S; p.T = T; p.ldo = ldo; p.x_begin = x_begin; p.x_end = x_end;
    p.tmax = tmax; p.tt0 = tt0; p.inv_dt = 1.0 / dt_eff; p.cs = 2.0 / (vmin * dt_eff);
    p.neg_u0 = (float)(-u0); p.thr = monotone ? thr : -1.f;   // non-monotone positions: every pair takes the exact path
    p.monotone = monotone;
    int path = 1;

    if (lat) {
        // Per profile: cs and thr exactly as a single-profile call with that profile computes them, then its row
        // vectors (kirch_prep_row): column xi of the lateral kernel is that call's column xi.
        const int P = lat->P;
        std::vector<double2> pc(P);
        for (int q = 0; q < P; ++q)
            pc[q] = make_double2(2.0 / (lat->vmin[q] * dt_eff), monotone ? (double)fast_thr(lat->vconst[q] != 0) : -1.0);
        char *b = lat->block + 256;   // [0, 256): run summary of the per-run path
        double2 *d_pc = (double2 *)b;
        b += kirch_a256((size_t)P * sizeof(double2));
        int *d_colp = (int *)b;
        b += kirch_a256((size_t)T * sizeof(int));
        const size_t ps = (size_t)P * S;
        double *l_vs = (double *)b;
        b += kirch_a256(ps * sizeof(double));
        double *l_zs = (double *)b;
        b += kirch_a256(ps * sizeof(double));
        double *l_zs2 = (double *)b;
        b += kirch_a256(ps * sizeof(double));
        float3 *l_rowc = (float3 *)b;
        // pageable sources: each copy returns once its source has been staged, so the host vectors may go
        IMPDAR_CUDA(cudaMemcpyAsync(d_pc, pc.data(), (size_t)P * sizeof(double2), cudaMemcpyHostToDevice, st));
        IMPDAR_CUDA(cudaMemcpyAsync(d_colp, lat->colp, (size_t)T * sizeof(int), cudaMemcpyHostToDevice, st));
        IMPDAR_CUDA(cudaMemcpyAsync(l_vs, lat->profiles, ps * sizeof(double), cudaMemcpyHostToDevice, st));
        kirch_prep_profiles_kernel<<<dim3(P, (S + 255) / 256), 256, 0, st>>>(d_tt, l_vs, l_zs, l_zs2, l_rowc, d_pc, S, dt_eff);
        IMPDAR_LAUNCH_CHECK();
        p.vs = l_vs; p.zs = l_zs; p.zs2 = l_zs2; p.rowc = l_rowc; p.colp = d_colp; p.pc = d_pc;
        path = 4;
    }

    if (use_table) {
        const int Amax = kirch_amax(T, vmax, tmax, dxm);
        const int A1 = Amax + 1;
        const int Apad = (int)kirch_roundup((size_t)Amax, 32);
        const int Tp = (int)kirch_roundup((size_t)ncols + 2 * (size_t)Apad, 32);
        const int aoff = Apad - c0;                                     // trace x lives at padded column aoff + x
        const size_t img = ((size_t)S * Tp + 4096) * sizeof(float);    // + slack after the last row (tiles overhang)
        float *gP = (float *)w;
        w += img;
        float *dP = nullptr;
        if (nearfield) {
            dP = (float *)w;
            w += img;
        }
        int2 *tab = (int2 *)w;
        w += (size_t)S * A1 * sizeof(int2);
        float *tabn = nullptr;
        if (nearfield) {
            tabn = (float *)w;
            w += (size_t)S * A1 * sizeof(float);
        }
        int *nm = (int *)w;
        w += (size_t)S * sizeof(int);
        int *amb_list = (int *)w;
        w += (size_t)S * A1 * sizeof(int);
        int *amb_count = flags + 8;
        int *sched_flags = flags + 16;
        w = (char *)(((uintptr_t)w + 255) & ~(uintptr_t)255);
        const bool use_tile = !nearfield && g_kirch_mode != 3;
        const int nchunks = pipe ? pipe->nchunks : 1;
        const size_t nblk_img = (size_t)(S + KT_Q - 1) / KT_Q;   // tile blocks of the image (schedule kept across row chunks)
        int2 *seg = (int2 *)w;
        int *nstage = nullptr;
        if (use_tile) {
            w += nblk_img * (size_t)S * sizeof(int2);
            nstage = (int *)w;
            w += nblk_img * sizeof(int);
        }
        IMPDAR_CHECK_ARG((unsigned long long)S * (unsigned long long)A1 < (1ull << 31), "kirchhoff: table too large");
        IMPDAR_CHECK_ARG((size_t)(w - (char *)workspace) <= ws_bytes, "kirchhoff: workspace too small for the table path");
        if (!continuing) {
            IMPDAR_CUDA(cudaMemsetAsync(gP, 0, img * (nearfield ? 2 : 1), st));
            IMPDAR_CUDA(cudaMemsetAsync(nm, 0, (size_t)S * sizeof(int), st));
            dim3 grid((A1 + 127) / 128, S);
            kirch_table_build_kernel<<<grid, 128, 0, st>>>(tab, tabn, nm, S, A1, dxm, zs, zs2, d_tt, d_vel, tmax, tt0,
                                                          1.0 / dt_eff, eps_t, amb_list, amb_count);
            IMPDAR_LAUNCH_CHECK();
        }
        if (use_tile) {
            int dev = 0;
            IMPDAR_CUDA(cudaGetDevice(&dev));
            if (dev >= 0 && dev < KP_MAX_DEVICES && !g_tile_attr[dev]) {
                IMPDAR_CUDA(cudaFuncSetAttribute(kirch_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KT_SMEM));
                g_tile_attr[dev] = true;
            }
        }
        KirchTabParams tp;
        tp.gP = gP; tp.dP = dP; tp.tab = tab; tp.tabn = tabn; tp.nm = nm; tp.out = out; tp.flags = flags;
        tp.stats = stats; tp.S = S; tp.T = T; tp.Tp = Tp; tp.Apad = aoff; tp.A1 = A1; tp.ldo = ldo;
        tp.x_begin = x_begin; tp.x_end = x_end;
        tp.only_if = use_tile ? sched_flags : nullptr;
        p.gradT = gP; p.dataT = dP; p.rowmajor = 1; p.Tp = Tp; p.Apad = aoff;
        path = use_tile ? 3 : 2;
        // Row chunks, bottom-up.  Without a host pipeline this is one chunk covering the whole image.
        int g_hi = rows ? rows->g_hi : S;   // d/dt rows [g_hi, S) are built
        int u_hi = S;   // input rows [u_hi, S) are uploaded
        for (int j = nchunks - 1; j >= 0; --j) {
            const int r0 = rows ? rows->s_begin : (int)((long long)S * j / nchunks);
            const int r1 = rows ? rows->s_end : (int)((long long)S * (j + 1) / nchunks);
            if (r1 <= r0) continue;
            if (pipe) {
                // rows r0 - 1 .. : what the d/dt stencil of rows >= r0 reads
                const int u0 = r0 > 0 ? r0 - 1 : 0;
                if (u0 < u_hi) {
                    IMPDAR_CUDA(cudaMemcpyAsync(pipe->d_in + (size_t)u0 * T, pipe->h_in + (size_t)u0 * T,
                                                (size_t)(u_hi - u0) * T * sizeof(float), cudaMemcpyHostToDevice, pipe->up));
                    u_hi = u0;
                }
                IMPDAR_CUDA(cudaEventRecord(pipe->ev_up[j], pipe->up));
                IMPDAR_CUDA(cudaStreamWaitEvent(st, pipe->ev_up[j], 0));
            }
            {
                const int g0 = r0;   // row r0 - 1 is uploaded (or r0 == 0: one-sided stencil)
                if (g0 < g_hi) {
                    // 128-bit path: data rows and the padded rows 16-byte aligned (aoff + c0 = Apad is a multiple of 32)
                    const int vec4 = (((uintptr_t)data & 15) == 0 && ld % 4 == 0 && ncols % 4 == 0) ? 1 : 0;
                    const int per_row = vec4 ? ncols / 4 : ncols;
                    int gx = (per_row + 255) / 256;
                    if (gx > 64) gx = 64;
                    dim3 grid(gx, g_hi - g0);
                    grad_padded_kernel<<<grid, 256, 0, st>>>(data, gP, dP, S, c0, ncols, ld, Tp, aoff, d_coef, flags, g0, vec4);
                    IMPDAR_LAUNCH_CHECK();
                    g_hi = g0;
                }
            }
            tp.s_begin = r0; tp.s_end = r1;
            if (g_stats_enabled) {
                kirch_table_count_kernel<<<r1 - r0, 256, 0, st>>>(tab, nm, A1, T, x_begin, x_end, r0, stats);
                IMPDAR_LAUNCH_CHECK();
            }
            if (use_tile && !continuing && j == nchunks - 1) {
                // Schedule of every tile block of the image: blocks at absolute multiples of KT_Q rows, so a row chunk
                // runs its part of the same blocks (clipped; a clipped block's intervals lie inside the full block's).
                // The stand-down for wide intervals is decided here, once per image (first chunk of the first call),
                // over all of them: row chunks, the host pipeline and one launch take the same decision.
                kirch_tile_sched_kernel<<<(S + KT_Q - 1) / KT_Q, 256, 0, st>>>(tab, nm, S, A1, 0, S, seg, nstage, sched_flags);
                IMPDAR_LAUNCH_CHECK();
            }
            if (use_tile) {
                const int b0 = r0 / KT_Q, nblk = (r1 - 1) / KT_Q - b0 + 1;   // the image's blocks that meet [r0, r1)
                KirchTileParams tq;
                tq.seg = seg + (size_t)b0 * S;
                tq.nstage = nstage + b0;
                tq.sched_flags = sched_flags;
                tq.t_base = b0 * KT_Q;
                dim3 tgrid(nblk, (x_end - x_begin + KT_X - 1) / KT_X);
                ktimer_begin("kirch_tile_kernel", st);
                kirch_tile_kernel<<<tgrid, KT_THREADS, KT_SMEM, st>>>(tp, tq);
                ktimer_end(st);
                IMPDAR_LAUNCH_CHECK();
            }
            const long long nitems = (long long)(r1 - r0) * ((x_end - x_begin + 4 * 32 * KT_R - 1) / (4 * 32 * KT_R));
            IMPDAR_CHECK_ARG(nitems < (1ll << 31), "kirchhoff: launch too large");
            // stand-in for the tile kernel: a grid that fills the GPU once and strides; otherwise one CTA per item
            const unsigned grid = (unsigned)(use_tile && nitems > (long long)num_sms() * 16 ? num_sms() * 16 : nitems);
            ktimer_begin("kirch_table_kernel", st);
            if (nearfield) kirch_table_kernel<true, false><<<grid, 128, 0, st>>>(tp);
            else kirch_table_kernel<false, false><<<grid, 128, 0, st>>>(tp);
            ktimer_end(st);
            IMPDAR_LAUNCH_CHECK();
            // exact pass over flagged table entries of these rows (reads the same padded row-major images)
            if (nearfield) kirch_table_fixup_kernel<true><<<num_sms() * 2, 256, 0, st>>>(tp, p, amb_list, amb_count);
            else kirch_table_fixup_kernel<false><<<num_sms() * 2, 256, 0, st>>>(tp, p, amb_list, amb_count);
            IMPDAR_LAUNCH_CHECK();
            if (pipe) {
                IMPDAR_CUDA(cudaEventRecord(pipe->ev_done[j], st));
                IMPDAR_CUDA(cudaStreamWaitEvent(pipe->down, pipe->ev_done[j], 0));
                const size_t n = (size_t)(r1 - r0) * T, off = (size_t)r0 * T;
                int blocks = (int)((n + 256 * 8 - 1) / (256 * 8));
                if (blocks > num_sms() * 8) blocks = num_sms() * 8;
                widen_f32_f64_kernel<<<blocks, 256, 0, pipe->down>>>(out + off, pipe->d_stage + off, n);
                IMPDAR_LAUNCH_CHECK();
                IMPDAR_CUDA(cudaMemcpyAsync(pipe->h_out + off, pipe->d_stage + off, n * sizeof(double), cudaMemcpyDeviceToHost,
                                            pipe->down));
            }
        }
    } else {
        IMPDAR_CHECK_ARG(!rows, "kirchhoff_rows: row-range calls need uniform trace spacing (the table path)");
        IMPDAR_CHECK_ARG((unsigned long long)(ncols + 32) * (unsigned long long)kirch_sp(S) < (1ull << 32),
                         "kirchhoff: (tnum + 32) * padded snum must stay below 2^32 elements");
        const int SP = kirch_sp(S);
        const size_t tbytes = (size_t)(ncols + 32) * SP * sizeof(float);  // 32 zero rows: chunks are padded to 4 traces
        float *gradT = (float *)w;
        w += tbytes;
        float *dataT = nullptr;
        if (nearfield) {
            dataT = (float *)w;
            w += tbytes;
        }
        IMPDAR_CUDA(cudaMemsetAsync(gradT, 0, tbytes * (nearfield ? 2 : 1), st));
        if (pipe)  // irregular geometry: no row pipeline, the whole input goes up first
            IMPDAR_CUDA(cudaMemcpyAsync(pipe->d_in, pipe->h_in, (size_t)S * T * sizeof(float), cudaMemcpyHostToDevice, st));
        {
            dim3 grid((ncols + 31) / 32, (S + 31) / 32), block(32, 8);
            grad_transpose_kernel<<<grid, block, 0, st>>>(data, gradT, dataT, S, ncols, ld, SP, d_coef, flags);
            IMPDAR_LAUNCH_CHECK();
        }
        // the kernel indexes traces globally: shift the bases so that trace x reads local column x - c0.  Its loops
        // stay inside the exact aperture, which the window covers (checked above); chunks of 4 traces may run up to 3
        // traces past it into the zero rows / the next traces, with zero weight.
        p.gradT = gradT - (size_t)c0 * SP; p.dataT = dataT ? dataT - (size_t)c0 * SP : nullptr; p.SP = SP;
        p.kmax = (unsigned)SP - 1u;
        dim3 grid((S + 31) / 32, (x_end - x_begin + 7) / 8), block(32, 8);
        if (lat) {
            ktimer_begin("kirch_general_lateral_kernel", st);
            if (nearfield) {
                if (g_stats_enabled) kirch_general_kernel<true, true, true><<<grid, block, 0, st>>>(p);
                else kirch_general_kernel<true, false, true><<<grid, block, 0, st>>>(p);
            } else {
                if (g_stats_enabled) kirch_general_kernel<false, true, true><<<grid, block, 0, st>>>(p);
                else kirch_general_kernel<false, false, true><<<grid, block, 0, st>>>(p);
            }
            ktimer_end(st);
        } else if (g_stats_enabled) {
            if (nearfield) { ktimer_begin("kirch_general_kernel", st); kirch_general_kernel<true, true><<<grid, block, 0, st>>>(p); ktimer_end(st); }
            else { ktimer_begin("kirch_general_kernel", st); kirch_general_kernel<false, true><<<grid, block, 0, st>>>(p); ktimer_end(st); }
        } else {
            if (nearfield) { ktimer_begin("kirch_general_kernel", st); kirch_general_kernel<true, false><<<grid, block, 0, st>>>(p); ktimer_end(st); }
            else { ktimer_begin("kirch_general_kernel", st); kirch_general_kernel<false, false><<<grid, block, 0, st>>>(p); ktimer_end(st); }
        }
        IMPDAR_LAUNCH_CHECK();
        if (pipe) {
            const size_t n = (size_t)S * T;
            widen_f32_f64_kernel<<<num_sms() * 8, 256, 0, st>>>(out, pipe->d_stage, n);
            IMPDAR_LAUNCH_CHECK();
            IMPDAR_CUDA(cudaMemcpyAsync(pipe->h_out, pipe->d_stage, n * sizeof(double), cudaMemcpyDeviceToHost, st));
        }
    }
    g_last_stats = stats;
    g_last_flags = flags;
    g_last_stats_stream = st;
    g_last_path = path;
    return IMPDAR_B200_OK;
}

// The scalar entries run the per-row code path with a constant vector: the same arithmetic as one velocity.
int impdar_kirchhoff_f32(const float *data, float *out, int S, int T, const double *dist_m, const double *tt_s,
                         const double *grad_coef, double vel, int nearfield, int x_begin, int x_end,
                         void *workspace, size_t ws_bytes, void *stream) {
    const std::vector<double> vs(S > 0 ? S : 0, vel);
    return kirchhoff_impl(data, out, S, T, dist_m, tt_s, grad_coef, vs.data(), nearfield, x_begin, x_end, workspace,
                          ws_bytes, stream, nullptr);
}

int impdar_kirchhoff_rows_f32(const float *data, float *out, int S, int T, const double *dist_m, const double *tt_s,
                              const double *grad_coef, double vel, int nearfield, int x_begin, int x_end, int s_begin,
                              int s_end, int g_hi, void *workspace, size_t ws_bytes, void *stream) {
    IMPDAR_CHECK_ARG(0 <= s_begin && s_begin < s_end && s_end <= S && s_end <= g_hi && g_hi <= S,
                     "kirchhoff_rows: need 0 <= s_begin < s_end <= g_hi <= snum, got [%d, %d), g_hi %d", s_begin, s_end, g_hi);
    const std::vector<double> vs(S, vel);
    KirchRows rows = {s_begin, s_end, g_hi};
    return kirchhoff_impl(data, out, S, T, dist_m, tt_s, grad_coef, vs.data(), nearfield, x_begin, x_end, workspace,
                          ws_bytes, stream, nullptr, &rows);
}

static int kirchhoff_window(const float *data, int col0, int ncols, int ld, float *out, int ldo, int S, int T,
                            const double *dist_m, const double *tt_s, const double *grad_coef, const double *vel_s,
                            int nearfield, int x_begin, int x_end, int s_begin, int s_end, int g_hi, void *workspace,
                            size_t ws_bytes, void *stream, bool any_order) {
    KirchWindow win = {col0, ncols, ld, ldo, false};
    if (s_begin == 0 && s_end == S && g_hi == S) {  // whole image: any geometry
        win.any_order = any_order && col0 == 0 && ncols == T;
        return kirchhoff_impl(data, out, S, T, dist_m, tt_s, grad_coef, vel_s, nearfield, x_begin, x_end, workspace,
                              ws_bytes, stream, nullptr, nullptr, &win);
    }
    IMPDAR_CHECK_ARG(0 <= s_begin && s_begin < s_end && s_end <= S && s_end <= g_hi && g_hi <= S,
                     "kirchhoff_window: need 0 <= s_begin < s_end <= g_hi <= snum, got [%d, %d), g_hi %d", s_begin, s_end, g_hi);
    KirchRows rows = {s_begin, s_end, g_hi};
    return kirchhoff_impl(data, out, S, T, dist_m, tt_s, grad_coef, vel_s, nearfield, x_begin, x_end, workspace, ws_bytes,
                          stream, nullptr, &rows, &win);
}

int impdar_kirchhoff_window_f32(const float *data, int col0, int ncols, int ld, float *out, int ldo, int S, int T,
                                const double *dist_m, const double *tt_s, const double *grad_coef, double vel,
                                int nearfield, int x_begin, int x_end, int s_begin, int s_end, int g_hi, void *workspace,
                                size_t ws_bytes, void *stream) {
    const std::vector<double> vs(S > 0 ? S : 0, vel);
    return kirchhoff_window(data, col0, ncols, ld, out, ldo, S, T, dist_m, tt_s, grad_coef, vs.data(), nearfield, x_begin,
                            x_end, s_begin, s_end, g_hi, workspace, ws_bytes, stream, false);
}

int impdar_kirchhoff_window_vz_f32(const float *data, int col0, int ncols, int ld, float *out, int ldo, int S, int T,
                                   const double *dist_m, const double *tt_s, const double *grad_coef, const double *vel_s,
                                   int nearfield, int x_begin, int x_end, int s_begin, int s_end, int g_hi,
                                   void *workspace, size_t ws_bytes, void *stream) {
    IMPDAR_CHECK_ARG(S >= 2, "kirchhoff: need snum >= 2, tnum >= 1");
    double vmax;
    if (int rc = kirch_vel_range(vel_s, S, &vmax)) return rc;
    return kirchhoff_window(data, col0, ncols, ld, out, ldo, S, T, dist_m, tt_s, grad_coef, vel_s, nearfield, x_begin,
                            x_end, s_begin, s_end, g_hi, workspace, ws_bytes, stream, true);
}

int impdar_kirchhoff_input_window_vz(int S, int T, const double *dist_m, const double *tt_s, const double *vel_s,
                                     int x_begin, int x_end, int *col0, int *col1) {
    IMPDAR_CHECK_ARG(S >= 2, "kirchhoff_input_window: bad range");
    double vmax;
    if (int rc = kirch_vel_range(vel_s, S, &vmax)) return rc;
    return impdar_kirchhoff_input_window(S, T, dist_m, tt_s, vmax, x_begin, x_end, col0, col1);
}

size_t impdar_kirchhoff_host_workspace_bytes(int S, int T, int nearfield) {
    const size_t n = (size_t)S * (size_t)T;
    return impdar_kirchhoff_workspace_bytes(S, T, nearfield) + n * (2 * sizeof(float) + sizeof(double)) + 1024;
}

static int kirchhoff_host_pipelined(const float *h_data, double *h_out, int S, int T, const double *dist_m,
                                    const double *tt_s, const double *grad_coef, const double *vel_s, int nearfield,
                                    int nchunks, void *workspace, size_t ws_bytes, void *stream) {
    IMPDAR_CHECK_ARG(h_data && h_out, "kirchhoff_host_pipelined: null pointer");
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1, "kirchhoff: need snum >= 2, tnum >= 1");
    IMPDAR_CHECK_ARG(nchunks >= 1 && nchunks <= KP_MAX_CHUNKS, "kirchhoff_host_pipelined: nchunks must be in [1, %d]", KP_MAX_CHUNKS);
    const size_t need = impdar_kirchhoff_host_workspace_bytes(S, T, nearfield);
    IMPDAR_CHECK_ARG(workspace && ws_bytes >= need, "kirchhoff_host_pipelined: workspace too small (%zu < %zu)", ws_bytes, need);
    KirchPipe *dev_pipe = nullptr;
    int rc = kirch_pipe_streams(&dev_pipe);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)S * (size_t)T;
    char *w = (char *)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    KirchPipe pipe = *dev_pipe;
    pipe.h_in = h_data;
    pipe.h_out = h_out;
    pipe.d_stage = (double *)w;
    w += n * sizeof(double);
    pipe.d_in = (float *)w;
    w += n * sizeof(float);
    float *d_out = (float *)w;
    w += n * sizeof(float);
    pipe.nchunks = nchunks;
    // the side streams start after whatever the caller's stream has queued on this workspace ...
    IMPDAR_CUDA(cudaEventRecord(pipe.ev_entry, st));
    IMPDAR_CUDA(cudaStreamWaitEvent(pipe.up, pipe.ev_entry, 0));
    IMPDAR_CUDA(cudaStreamWaitEvent(pipe.down, pipe.ev_entry, 0));
    rc = kirchhoff_impl(pipe.d_in, d_out, S, T, dist_m, tt_s, grad_coef, vel_s, nearfield, 0, T, w,
                        ws_bytes - (size_t)(w - (char *)workspace), stream, &pipe);
    // ... and the caller's stream finishes after them: one synchronisation on `stream` covers the downloads
    cudaEventRecord(pipe.ev_exit, pipe.down);
    cudaStreamWaitEvent(st, pipe.ev_exit, 0);
    cudaEventRecord(pipe.ev_exit, pipe.up);
    cudaStreamWaitEvent(st, pipe.ev_exit, 0);
    return rc;
}

int impdar_kirchhoff_host_pipelined_f64(const float *h_data, double *h_out, int S, int T, const double *dist_m,
                                        const double *tt_s, const double *grad_coef, double vel, int nearfield,
                                        int nchunks, void *workspace, size_t ws_bytes, void *stream) {
    const std::vector<double> vs(S > 0 ? S : 0, vel);
    return kirchhoff_host_pipelined(h_data, h_out, S, T, dist_m, tt_s, grad_coef, vs.data(), nearfield, nchunks, workspace,
                                    ws_bytes, stream);
}

int impdar_kirchhoff_host_pipelined_vz_f64(const float *h_data, double *h_out, int S, int T, const double *dist_m,
                                           const double *tt_s, const double *grad_coef, const double *vel_s,
                                           int nearfield, int nchunks, void *workspace, size_t ws_bytes, void *stream) {
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1, "kirchhoff: need snum >= 2, tnum >= 1");
    double vmax;
    if (int rc = kirch_vel_range(vel_s, S, &vmax)) return rc;
    return kirchhoff_host_pipelined(h_data, h_out, S, T, dist_m, tt_s, grad_coef, vel_s, nearfield, nchunks, workspace,
                                    ws_bytes, stream);
}

size_t impdar_kirchhoff_lateral_workspace_bytes(int S, int T, int P, int nearfield) {
    if (S < 2 || T < 1 || P < 1) return 0;
    return impdar_kirchhoff_workspace_bytes(S, T, nearfield) + kirch_lateral_block_bytes(S, T, P);
}

// Lateral velocity: output trace xi migrates with profile col_profile[xi] of `profiles` (P x S RMS velocities).  Path:
// with uniform spacing and runs (maximal ranges of traces with one profile) at least KIRCH_RUN_MIN traces wide on
// average over the whole profile, one single-profile table / tile call per run of [x_begin, x_end) on its own input
// sub-window; otherwise the lateral general kernel in one launch.  KIRCHHOFF_GENERAL forces the kernel, the table modes
// force the runs.
constexpr int KIRCH_RUN_MIN = 192;

int impdar_kirchhoff_window_vxz_f32(const float *data, int col0, int ncols, int ld, float *out, int ldo, int S, int T,
                                    const double *dist_m, const double *tt_s, const double *grad_coef,
                                    const double *profiles, int P, const int *col_profile, int nearfield, int x_begin,
                                    int x_end, void *workspace, size_t ws_bytes, void *stream) {
    IMPDAR_CHECK_ARG(data && out && dist_m && tt_s && grad_coef && profiles && col_profile, "kirchhoff_vxz: null pointer");
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1 && P >= 1, "kirchhoff_vxz: need snum >= 2, tnum >= 1, nprof >= 1");
    IMPDAR_CHECK_ARG(T < (1 << 26), "kirchhoff: tnum too large");
    IMPDAR_CHECK_ARG(0 <= x_begin && x_begin < x_end && x_end <= T, "kirchhoff: bad output range [%d, %d)", x_begin, x_end);
    const size_t base = impdar_kirchhoff_workspace_bytes(S, T, nearfield);
    const size_t need = impdar_kirchhoff_lateral_workspace_bytes(S, T, P, nearfield);
    IMPDAR_CHECK_ARG(workspace && ws_bytes >= need, "kirchhoff_vxz: workspace too small (%zu < %zu)", ws_bytes, need);
    std::vector<double> vmin(P), vmax(P), vrow(S, 0.0);   // vrow: largest velocity of each row (the reach of a pair)
    std::vector<unsigned char> vconst(P);
    for (int q = 0; q < P; ++q) {
        const double *v = profiles + (size_t)q * S;
        double lo = v[0], hi = v[0];
        for (int i = 0; i < S; ++i) {
            IMPDAR_CHECK_ARG(std::isfinite(v[i]) && v[i] > 0.0,
                             "kirchhoff_vxz: profile %d velocity[%d] = %g must be finite and positive", q, i, v[i]);
            lo = fmin(lo, v[i]);
            hi = fmax(hi, v[i]);
            vrow[i] = fmax(vrow[i], v[i]);
        }
        vmin[q] = lo;
        vmax[q] = hi;
        vconst[q] = lo == hi;
    }
    for (int x = 0; x < T; ++x)
        IMPDAR_CHECK_ARG(col_profile[x] >= 0 && col_profile[x] < P, "kirchhoff_vxz: col_profile[%d] = %d outside [0, %d)",
                         x, col_profile[x], P);
    // The path depends on the whole trace -> profile map (not on [x_begin, x_end) or the window), so sub-ranges and
    // windows take the whole image's path.
    long long runs_all = 1;
    for (int x = 1; x < T; ++x) runs_all += col_profile[x] != col_profile[x - 1];
    std::vector<int> run0;   // first output trace of each run of [x_begin, x_end)
    for (int x = x_begin; x < x_end; ++x)
        if (x == x_begin || col_profile[x] != col_profile[x - 1]) run0.push_back(x);
    const int nruns = (int)run0.size();
    run0.push_back(x_end);
    double vmin_all = vmin[0];
    for (int q = 1; q < P; ++q) vmin_all = fmin(vmin_all, vmin[q]);
    // a run's own spacing test (its vmin >= vmin_all) passes whenever this one does
    const bool uniform_ok = kirch_spacing(S, T, dist_m, tt_s, vmin_all, kirch_monotone(T, dist_m)).uniform_ok;
    IMPDAR_CHECK_ARG(!(g_kirch_mode >= 2 && !uniform_ok), "kirchhoff: table path forced but trace spacing is not uniform");
    const bool per_run = g_kirch_mode >= 2 ||
                         (g_kirch_mode == 0 && uniform_ok && (long long)T >= (long long)KIRCH_RUN_MIN * runs_all);
    char *block = (char *)(((uintptr_t)workspace + base + 255) & ~(uintptr_t)255);
    cudaStream_t st = (cudaStream_t)stream;
    if (!per_run) {
        KirchLateral lat = {profiles, P, col_profile, vmin.data(), vconst.data(), block};
        KirchWindow win = {col0, ncols, ld, ldo, col0 == 0 && ncols == T};
        return kirchhoff_impl(data, out, S, T, dist_m, tt_s, grad_coef, vrow.data(), nearfield, x_begin, x_end, workspace,
                              base, stream, nullptr, nullptr, &win, &lat);
    }
    IMPDAR_CHECK_ARG(col0 >= 0 && ncols >= 1 && col0 + ncols <= T && ld >= ncols,
                     "kirchhoff_window: bad column window [%d, %d) / strides", col0, col0 + ncols);
    int *sum = (int *)block;
    IMPDAR_CUDA(cudaMemsetAsync(sum, 0, 256, st));
    int path = 0;
    for (int r = 0; r < nruns; ++r) {
        const int a = run0[r], b = run0[r + 1], q = col_profile[a];
        // the run's input window, inside the caller's, cut at multiples of 4 columns from col0 (128-bit d/dt pass)
        int w0 = 0, w1 = T;
        if (int rc = impdar_kirchhoff_input_window(S, T, dist_m, tt_s, vmax[q], a, b, &w0, &w1)) return rc;
        w0 = w0 > col0 ? w0 : col0;
        w1 = w1 < col0 + ncols ? w1 : col0 + ncols;
        w0 = col0 + ((w0 - col0) & ~3);
        w1 = col0 + ((w1 - col0 + 3) & ~3);
        if (w1 > col0 + ncols) w1 = col0 + ncols;
        KirchWindow win = {w0, w1 - w0, ld, ldo, false};
        int rc = kirchhoff_impl(data + (w0 - col0), out + (a - x_begin), S, T, dist_m, tt_s, grad_coef,
                                profiles + (size_t)q * S, nearfield, a, b, workspace, base, stream, nullptr, nullptr, &win);
        if (rc) return rc;
        kirch_run_summary_kernel<<<1, 32, 0, st>>>(g_last_flags, sum);
        IMPDAR_LAUNCH_CHECK();
        path = g_last_path;
    }
    g_last_flags = sum;
    g_last_stats = (unsigned long long *)(sum + 32);
    g_last_path = path;
    return IMPDAR_B200_OK;
}

int impdar_kirchhoff_set_mode(int mode) {
    IMPDAR_CHECK_ARG(mode >= 0 && mode <= 3, "kirchhoff_set_mode: 0 auto, 1 general kernel, 2 uniform-geometry table path, "
                                             "3 table path with the global-gather kernel only");
    g_kirch_mode = mode;
    return IMPDAR_B200_OK;
}

int impdar_kirchhoff_last_path(void) { return g_last_path; }

int impdar_kirchhoff_enable_stats(int on) {
    g_stats_enabled = on ? 1 : 0;
    return IMPDAR_B200_OK;
}

int impdar_kirchhoff_last_stats(unsigned long long *pairs, unsigned long long *exact_pairs) {
    IMPDAR_CHECK_ARG(g_last_stats, "kirchhoff_last_stats: no previous call");
    unsigned long long h[2];
    IMPDAR_CUDA(cudaMemcpyAsync(h, g_last_stats, sizeof(h), cudaMemcpyDeviceToHost, g_last_stats_stream));
    IMPDAR_CUDA(cudaStreamSynchronize(g_last_stats_stream));
    if (pairs) *pairs = h[0];
    if (exact_pairs) *exact_pairs = h[1];
    return IMPDAR_B200_OK;
}

int impdar_kirchhoff_last_tile_standdown(int *stood_down) {
    IMPDAR_CHECK_ARG(stood_down && g_last_flags, "kirchhoff_last_tile_standdown: no previous call");
    int h[17] = {0};
    IMPDAR_CUDA(cudaMemcpyAsync(h, g_last_flags, sizeof(h), cudaMemcpyDeviceToHost, g_last_stats_stream));
    IMPDAR_CUDA(cudaStreamSynchronize(g_last_stats_stream));
    *stood_down = (g_last_path != 3) ? -1 : ((h[0] | h[16]) ? 1 : 0);
    return IMPDAR_B200_OK;
}

}  // extern "C"
