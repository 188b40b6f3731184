// Stolt f-k migration (reference: migrationlib/mig_python.py:126-208).
//
//   taper -> rfft2(axes=(1,0)) -> for every (kz_j, kx): KK = lin-interp_w FK[:, kx] at w' = sqrt(w_j^2 + (v kx/2)^2)
//   (clamped to the Nyquist row, FITPACK k=1 semantics) * w_j/w' -> KK[0,0] = 0 -> irfft2(axes=(1,0)).
//
// Device pipeline per profile (HBM-bound, five sweeps):
//   1 taper (fp32, vectorised)            2 cuFFT R2C along time (stride = tnum, batch = tnum)
//   3 cuFFT C2C along traces, in place    4 remap + obliquity + 1/(S'T) scale kernel (this file)
//   5 cuFFT C2C inverse along traces      6 cuFFT C2R along time
// Even snum and tnum take the paired-trace pipeline instead (three sweeps fewer, no real-transform wrappers):
//   adjacent traces are one complex signal z[s][j] = d[s][2j] + i d[s][2j+1] (a reinterpretation of the same
//   memory), transformed by plain in-place 2-D C2C FFTs; stolt_remap_paired_kernel recovers
//   FK[w][kx] = E[w][kx mod T/2] + e^{-2 pi i kx/T} O[w][kx mod T/2] from Zh = E + iO and its Hermitian partner
//   Zh[-w][-k] on the fly, applies the remap to the two columns kx and kx + T/2, and writes the spectrum of the
//   output image in the same paired form (plus its Hermitian mirror row), so the inverse C2C lands the real
//   result directly in the output layout.
// The remap coordinate f = w'/dw = sqrt(j^2 + beta^2) is evaluated in fp64 (f reaches ~snum/2 and the
// interpolation weight is its fractional part); the interpolation itself is fp32 complex FMA.
#include <cufft.h>

#include <cmath>
#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"

extern "C" int impdar_taper_f32(const float *x, float *y, int S, int T, int batch, double htaper, double vtaper,
                                int trunc_int, void *stream);

namespace impdar {

#define IMPDAR_CUFFT(call)                                                                  \
    do {                                                                                    \
        cufftResult r__ = (call);                                                           \
        if (r__ != CUFFT_SUCCESS) {                                                         \
            impdar::set_error("%s:%d %s -> cufft error %d", __FILE__, __LINE__, #call, (int)r__); \
            return IMPDAR_B200_ECUFFT;                                                      \
        }                                                                                   \
    } while (0)

struct StoltRemapParams {
    const float2 *FK;  // (M, T)
    float2 *KK;        // (M, T)
    int M, T, nz;
    double beta_unit;  // beta = beta_unit * kxi   (kxi = signed fft index of the column)
    float norm;        // 1 / (S' * T)
};

__global__ void __launch_bounds__(128) stolt_remap_kernel(const __grid_constant__ StoltRemapParams p, int rows_per_cta) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= p.T) return;
    const int kxi = (x <= (p.T - 1) / 2) ? x : x - p.T;  // np.fft.fftfreq ordering
    const double beta = p.beta_unit * (double)kxi;
    const double beta2 = beta * beta;
    const int j0 = blockIdx.y * rows_per_cta;
    const int j1 = min(p.M, j0 + rows_per_cta);
    const double fmax = (double)(p.M - 1);
    int cur = -2;
    float2 v0 = make_float2(0.f, 0.f), v1 = v0;
    for (int j = j0; j < j1; ++j) {
        float2 o = make_float2(0.f, 0.f);
        if (j < p.nz && p.M > 1) {
            const double f = sqrt((double)j * (double)j + beta2);
            const double fq = fmin(f, fmax);
            int i0 = (int)fq;
            i0 = min(i0, p.M - 2);
            const float a = (float)(fq - (double)i0);
            if (i0 != cur) {
                if (i0 == cur + 1) {
                    v0 = v1;
                } else {
                    v0 = p.FK[(size_t)i0 * p.T + x];
                }
                v1 = p.FK[(size_t)(i0 + 1) * p.T + x];
                cur = i0;
            }
            // scaling = kZ / sqrt(kX^2 + kZ^2) = j / f ; (0,0) is 0/0 in the reference and then set to 0
            const float sc = (f > 0.0) ? (float)((double)j / f) * p.norm : 0.f;
            const float w0 = (1.f - a) * sc, w1 = a * sc;
            o.x = fmaf(v0.x, w0, v1.x * w1);
            o.y = fmaf(v0.y, w0, v1.y * w1);
        }
        p.KK[(size_t)j * p.T + x] = o;
    }
}


struct StoltPairedParams {
    const float2 *Zh;  // (S, Th) forward 2-D spectrum of the paired image
    float2 *Zq;        // (S, Th) spectrum of the paired output image
    int S, Th, T, nz;
    double beta_unit;
    float norm;        // 1 / (S * T)
};

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}

// FK[i][kap] and FK[i][kap + Th] from the paired spectrum: E = (Z + conj(Zp))/2, O = (Z - conj(Zp))/(2i),
// FK = E +- w O with w = exp(-2 pi i kap / T).
__device__ __forceinline__ void paired_row(const StoltPairedParams &p, int i, int kap, int kapm, float2 w, float2 &fa,
                                           float2 &fb) {
    const float2 z = p.Zh[(size_t)i * p.Th + kap];
    const int im = (i == 0) ? 0 : p.S - i;
    const float2 zp = p.Zh[(size_t)im * p.Th + kapm];
    const float2 e = make_float2(0.5f * (z.x + zp.x), 0.5f * (z.y - zp.y));
    const float2 o = make_float2(0.5f * (z.y + zp.y), -0.5f * (z.x - zp.x));
    const float2 wo = cmul(w, o);
    fa = cadd(e, wo);
    fb = csub(e, wo);
}

__global__ void __launch_bounds__(128) stolt_remap_paired_kernel(const __grid_constant__ StoltPairedParams p,
                                                                 int rows_per_cta) {
    const int kap = blockIdx.x * blockDim.x + threadIdx.x;
    if (kap >= p.Th) return;
    const int kapm = (kap == 0) ? 0 : p.Th - kap;
    double sn, cs;
    sincospi(-2.0 * (double)kap / (double)p.T, &sn, &cs);
    const float2 w = make_float2((float)cs, (float)sn);
    const float2 wc = make_float2(w.x, -w.y);
    const double betaA = p.beta_unit * (double)kap, betaB = p.beta_unit * (double)(p.Th - kap);
    const double bA2 = betaA * betaA, bB2 = betaB * betaB;
    const double fmax = (double)p.nz;  // last rfft row index M - 1 = S/2
    const int j0 = blockIdx.y * rows_per_cta;
    const int j1 = min(p.nz, j0 + rows_per_cta);
    int curA = -2, curB = -2;
    float2 a0 = make_float2(0.f, 0.f), a1 = a0, b0 = a0, b1 = a0, tmp;
    for (int j = j0; j < j1; ++j) {
        if (j == 0) {  // kz = 0 row: scaling is 0 (and KK[0,0] = 0); its mirror is itself; also clear the Nyquist row
            p.Zq[kap] = make_float2(0.f, 0.f);
            p.Zq[(size_t)p.nz * p.Th + kap] = make_float2(0.f, 0.f);
            continue;
        }
        const double jj = (double)j * (double)j;
        // ---- column kx = kap
        const double fA = sqrt(jj + bA2);
        {
            const double fq = fmin(fA, fmax);
            const int i0 = min((int)fq, p.nz - 1);
            if (i0 != curA) {
                if (i0 == curA + 1) a0 = a1; else paired_row(p, i0, kap, kapm, w, a0, tmp);
                paired_row(p, i0 + 1, kap, kapm, w, a1, tmp);
                curA = i0;
            }
        }
        const double fqA = fmin(fA, fmax);
        const float aA = (float)(fqA - (double)curA);
        const float scA = (float)((double)j / fA) * p.norm;
        const float2 gA = make_float2(fmaf(a0.x, (1.f - aA) * scA, a1.x * (aA * scA)),
                                      fmaf(a0.y, (1.f - aA) * scA, a1.y * (aA * scA)));
        // ---- column kx = kap + Th
        const double fB = sqrt(jj + bB2);
        {
            const double fq = fmin(fB, fmax);
            const int i0 = min((int)fq, p.nz - 1);
            if (i0 != curB) {
                if (i0 == curB + 1) b0 = b1; else paired_row(p, i0, kap, kapm, w, tmp, b0);
                paired_row(p, i0 + 1, kap, kapm, w, tmp, b1);
                curB = i0;
            }
        }
        const double fqB = fmin(fB, fmax);
        const float aB = (float)(fqB - (double)curB);
        const float scB = (float)((double)j / fB) * p.norm;
        const float2 gB = make_float2(fmaf(b0.x, (1.f - aB) * scB, b1.x * (aB * scB)),
                                      fmaf(b0.y, (1.f - aB) * scB, b1.y * (aB * scB)));
        // ---- paired output spectrum and its Hermitian mirror
        const float2 e = cadd(gA, gB);
        const float2 o = cmul(csub(gA, gB), wc);
        p.Zq[(size_t)j * p.Th + kap] = make_float2(e.x - o.y, e.y + o.x);              // E' + i O'
        p.Zq[(size_t)(p.S - j) * p.Th + kapm] = make_float2(e.x + o.y, o.x - e.y);     // conj(E') + i conj(O')
    }
}

struct StoltPlans {
    cufftHandle r2c = 0, c2c = 0, c2r = 0, c2c2d = 0;
    bool paired = false;
};
static std::map<std::tuple<int, int, int, long long>, StoltPlans> g_plans;  // (device, S, T, stream): a cuFFT plan owns one
// work area, so calls that may overlap on different streams get their own plans
static std::mutex g_plans_mu;

// 0 auto (five-pass kernels of stolt_fft.cu for the power-of-two shapes they cover, else the cuFFT paired-trace
// pipeline for even shapes, else cuFFT R2C/C2R); 1 force cuFFT R2C/C2R; 2 force cuFFT paired; 3 force five-pass.
static int g_stolt_mode = 0;
static int g_stolt_stop_after = 0;
static int g_stolt_last = 0;
static inline bool stolt_use_paired(int S, int T) {
    return g_stolt_mode != 1 && (S % 2 == 0) && (T % 2 == 0) && S >= 4 && T >= 4;
}

bool stolt_fft_supported(int S, int T);
size_t stolt_fft_workspace_bytes(int S, int T);
int stolt_fft_run(const float *data, float *out, int S, int T, int batch, double dt, double dx, double vel, double htaper,
                  double vtaper, int trunc_int, void *workspace, int stop_after, cudaStream_t st);

int stolt_fft_scan_forward(const float *data, float *W1, float *W2, int S, int T, double htaper, double vtaper,
                           int trunc_int, cudaStream_t st);
int stolt_fft_scan_velocity(const float *W2, float *W3, float *img, int S, int T, double dt, double dx, double vel,
                            cudaStream_t st);
size_t stolt_focus_workspace_bytes(int rows, int cols);
int stolt_focus_run(const float *img, int rows, int cols, int ws, int wt, double *focus, void *part, cudaStream_t st);

static int get_plans(int S, int T, cudaStream_t st, StoltPlans &out) {
    int dev = 0;
    IMPDAR_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_plans_mu);
    auto key = std::make_tuple(dev, S, stolt_use_paired(S, T) ? T : -T, (long long)(intptr_t)st);
    auto it = g_plans.find(key);
    if (it != g_plans.end()) {
        out = it->second;
        return IMPDAR_B200_OK;
    }
    StoltPlans pl;
    const int M = S / 2 + 1;
    const int S2 = 2 * (M - 1);
    pl.paired = stolt_use_paired(S, T);
    if (pl.paired) {
        int n[2] = {S, T / 2};
        IMPDAR_CUFFT(cufftPlanMany(&pl.c2c2d, 2, n, nullptr, 1, 0, nullptr, 1, 0, CUFFT_C2C, 1));
        g_plans[key] = pl;
        out = pl;
        return IMPDAR_B200_OK;
    }
    {
        int n[1] = {S}, inembed[1] = {S}, onembed[1] = {M};
        IMPDAR_CUFFT(cufftPlanMany(&pl.r2c, 1, n, inembed, T, 1, onembed, T, 1, CUFFT_R2C, T));
    }
    {
        int n[1] = {T};
        IMPDAR_CUFFT(cufftPlanMany(&pl.c2c, 1, n, nullptr, 1, T, nullptr, 1, T, CUFFT_C2C, M));
    }
    if (S2 >= 1) {
        int n[1] = {S2}, inembed[1] = {M}, onembed[1] = {S2};
        IMPDAR_CUFFT(cufftPlanMany(&pl.c2r, 1, n, inembed, T, 1, onembed, T, 1, CUFFT_C2R, T));
    }
    g_plans[key] = pl;
    out = pl;
    return IMPDAR_B200_OK;
}

}  // namespace impdar

using namespace impdar;

extern "C" {

size_t impdar_stolt_workspace_bytes(int S, int T, int batch) {
    // cuFFT pipelines: profiles go one at a time through the same buffers.  Five-pass pipeline: one transposed
    // half spectrum per profile of a launch, up to 4 GiB (larger batches are processed in chunks).
    if (g_stolt_mode != 1 && g_stolt_mode != 2 && stolt_fft_supported(S, T)) {
        const size_t per = stolt_fft_workspace_bytes(S, T) - 256;
        size_t nb = (size_t)(batch < 1 ? 1 : batch);
        const size_t cap = ((size_t)4 << 30) / per;
        if (nb > cap) nb = cap < 1 ? 1 : cap;
        const size_t five = nb * per + 256;
        const size_t M5 = (size_t)(S / 2 + 1);
        const size_t generic = 2 * M5 * (size_t)T * sizeof(float2) + 1024;
        return five > generic ? five : generic;
    }
    const size_t M = (size_t)(S / 2 + 1);
    const size_t cplx = M * (size_t)T * sizeof(float2);
    const size_t real = (size_t)S * (size_t)T * sizeof(float);
    const size_t a = cplx > real ? cplx : real;
    return a + cplx + 1024;
}

int impdar_stolt_f32(const float *data, float *out, int S, int T, int batch, double dt, double dx, double vel,
                     double htaper, double vtaper, int trunc_int, void *workspace, size_t ws_bytes,
                     void *stream) {
    IMPDAR_CHECK_ARG(data && out, "stolt: null pointer");
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1 && batch >= 1, "stolt: need snum >= 2, tnum >= 1, batch >= 1");
    IMPDAR_CHECK_ARG(dt > 0.0 && vel > 0.0 && dx != 0.0, "stolt: dt, vel must be positive and dx non-zero");
    const size_t need = impdar_stolt_workspace_bytes(S, T, batch);
    IMPDAR_CHECK_ARG(workspace && ws_bytes >= need, "stolt: workspace too small (%zu < %zu)", ws_bytes, need);
    cudaStream_t st = (cudaStream_t)stream;
    const int M = S / 2 + 1;
    const int S2 = 2 * (M - 1);
    const size_t cplx = (size_t)M * T * sizeof(float2);
    const size_t real = (size_t)S * T * sizeof(float);
    char *w = (char *)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    float *bufA = (float *)w;              // tapered input, later the remapped spectrum KK
    float2 *bufKK = (float2 *)w;
    float2 *bufFK = (float2 *)(w + (((cplx > real ? cplx : real) + 255) & ~(size_t)255));

    IMPDAR_CHECK_ARG(!(g_stolt_mode == 3 && !stolt_fft_supported(S, T)),
                     "stolt: the five-pass pipeline does not cover snum = %d, tnum = %d", S, T);
    if ((g_stolt_mode == 0 || g_stolt_mode == 3) && stolt_fft_supported(S, T)) {
        // as many profiles per launch as the workspace holds (grid.z <= 65535, batch * T/2 columns fit an int)
        size_t per = stolt_fft_workspace_bytes(S, T) - 256;
        int nb_max = (int)((ws_bytes - 256) / per);
        if (nb_max > 4096) nb_max = 4096;
        for (int b = 0; b < batch; b += nb_max) {
            const int nb = (batch - b < nb_max) ? batch - b : nb_max;
            int rcf = stolt_fft_run(data + (size_t)b * S * T, out + (size_t)b * S * T, S, T, nb, dt, dx, vel, htaper, vtaper,
                                    trunc_int, workspace, g_stolt_stop_after, st);
            if (rcf) return rcf;
        }
        g_stolt_last = 3;
        return IMPDAR_B200_OK;
    }
    StoltPlans pl;
    int rc = get_plans(S, T, st, pl);
    if (rc) return rc;
    g_stolt_last = pl.paired ? 2 : 1;
    if (pl.paired) {
        IMPDAR_CUFFT(cufftSetStream(pl.c2c2d, st));
        StoltPairedParams pp;
        pp.S = S; pp.Th = T / 2; pp.T = T; pp.nz = S / 2;
        pp.beta_unit = vel * (double)S * dt / (2.0 * (double)T * dx);
        pp.norm = (float)(1.0 / ((double)S * (double)T));
        for (int b = 0; b < batch; ++b) {
            const float *din = data + (size_t)b * S * T;
            float *dout = out + (size_t)b * S * T;
            rc = impdar_taper_f32(din, bufA, S, T, 1, htaper, vtaper, trunc_int, stream);
            if (rc) return rc;
            IMPDAR_CUFFT(cufftExecC2C(pl.c2c2d, (cufftComplex *)bufA, (cufftComplex *)bufA, CUFFT_FORWARD));
            pp.Zh = (const float2 *)bufA;
            pp.Zq = (float2 *)dout;
            const int rows_per_cta = 32;
            dim3 grid((pp.Th + 127) / 128, (pp.nz + rows_per_cta - 1) / rows_per_cta);
            ktimer_begin("stolt_remap_paired_kernel", st);
            stolt_remap_paired_kernel<<<grid, 128, 0, st>>>(pp, rows_per_cta);
            ktimer_end(st);
            IMPDAR_LAUNCH_CHECK();
            IMPDAR_CUFFT(cufftExecC2C(pl.c2c2d, (cufftComplex *)dout, (cufftComplex *)dout, CUFFT_INVERSE));
            count_launch(2);
        }
        return IMPDAR_B200_OK;
    }
    IMPDAR_CUFFT(cufftSetStream(pl.r2c, st));
    IMPDAR_CUFFT(cufftSetStream(pl.c2c, st));
    IMPDAR_CUFFT(cufftSetStream(pl.c2r, st));

    StoltRemapParams rp;
    rp.M = M; rp.T = T; rp.nz = S / 2;
    // beta = (vel * kx / 2) / dw,  kx = 2 pi kxi / (T dx),  dw = 2 pi / (S dt)
    rp.beta_unit = vel * (double)S * dt / (2.0 * (double)T * dx);
    rp.norm = (float)(1.0 / ((double)S2 * (double)T));

    for (int b = 0; b < batch; ++b) {
        const float *din = data + (size_t)b * S * T;
        float *dout = out + (size_t)b * S2 * T;
        rc = impdar_taper_f32(din, bufA, S, T, 1, htaper, vtaper, trunc_int, stream);
        if (rc) return rc;
        IMPDAR_CUFFT(cufftExecR2C(pl.r2c, bufA, (cufftComplex *)bufFK));
        IMPDAR_CUFFT(cufftExecC2C(pl.c2c, (cufftComplex *)bufFK, (cufftComplex *)bufFK, CUFFT_FORWARD));
        count_launch(2);
        rp.FK = bufFK;
        rp.KK = bufKK;
        const int rows_per_cta = 32;
        dim3 grid((T + 127) / 128, (M + rows_per_cta - 1) / rows_per_cta);
        ktimer_begin("stolt_remap_kernel", st);
        stolt_remap_kernel<<<grid, 128, 0, st>>>(rp, rows_per_cta);
        ktimer_end(st);
        IMPDAR_LAUNCH_CHECK();
        IMPDAR_CUFFT(cufftExecC2C(pl.c2c, (cufftComplex *)bufKK, (cufftComplex *)bufKK, CUFFT_INVERSE));
        IMPDAR_CUFFT(cufftExecC2R(pl.c2r, (cufftComplex *)bufKK, dout));
        count_launch(2);
    }
    return IMPDAR_B200_OK;
}

static inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// Velocities run one after another through the same buffers, so the scratch does not grow with nvel.
size_t impdar_stolt_scan_workspace_bytes(int S, int T, int nvel) {
    (void)nvel;
    if (S < 2 || T < 1) return 0;
    const size_t M = (size_t)(S / 2 + 1);
    const size_t img = (size_t)S * (size_t)T * sizeof(float);
    const size_t cplx = M * (size_t)T * sizeof(float2);
    // five-pass: W1 (P1 output and the image when the caller keeps none), W2 (forward spectrum), W3 (one velocity's
    // spectrum); cuFFT: the taper / remapped-spectrum buffer, the forward spectrum and the image
    const size_t five = 3 * align256(img);
    const size_t fft = align256(cplx > img ? cplx : img) + align256(cplx) + align256(img);
    return (five > fft ? five : fft) + align256(stolt_focus_workspace_bytes(2 * (S / 2), T)) + 256;
}

int impdar_stolt_scan_f32(const float *data, int S, int T, double dt, double dx, const double *vels, int nvel,
                          double htaper, double vtaper, int trunc_int, int win_s, int win_t, double *focus,
                          float *images, void *workspace, size_t ws_bytes, void *stream) {
    IMPDAR_CHECK_ARG(data && focus, "stolt_scan: null pointer");
    IMPDAR_CHECK_ARG(S >= 2 && T >= 1, "stolt_scan: need snum >= 2, tnum >= 1");
    IMPDAR_CHECK_ARG(dt > 0.0 && dx != 0.0, "stolt_scan: dt must be positive and dx non-zero");
    IMPDAR_CHECK_ARG(vels && nvel >= 1, "stolt_scan: need at least one velocity");
    for (int v = 0; v < nvel; ++v)
        IMPDAR_CHECK_ARG(std::isfinite(vels[v]) && vels[v] > 0.0, "stolt_scan: velocity %d (%g) must be finite and positive",
                         v, vels[v]);
    IMPDAR_CHECK_ARG(win_s >= 1 && win_t >= 1, "stolt_scan: window (%d, %d) must be at least 1 x 1", win_s, win_t);
    const size_t need = impdar_stolt_scan_workspace_bytes(S, T, nvel);
    IMPDAR_CHECK_ARG(workspace && ws_bytes >= need, "stolt_scan: workspace too small (%zu < %zu)", ws_bytes, need);
    IMPDAR_CHECK_ARG(!(g_stolt_mode == 3 && !stolt_fft_supported(S, T)),
                     "stolt: the five-pass pipeline does not cover snum = %d, tnum = %d", S, T);
    cudaStream_t st = (cudaStream_t)stream;
    const int M = S / 2 + 1;
    const int S2 = 2 * (M - 1);
    const size_t per_img = (size_t)S2 * T;
    const size_t per_focus = (size_t)((S2 + win_s - 1) / win_s) * (size_t)((T + win_t - 1) / win_t);
    const size_t img = (size_t)S * T * sizeof(float);
    const size_t cplx = (size_t)M * T * sizeof(float2);
    char *w = (char *)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    const size_t five = 3 * align256(img);
    const size_t fft = align256(cplx > img ? cplx : img) + align256(cplx) + align256(img);
    void *part = w + (five > fft ? five : fft);
    int rc;

    if ((g_stolt_mode == 0 || g_stolt_mode == 3) && stolt_fft_supported(S, T)) {
        float *W1 = (float *)w, *W2 = (float *)(w + align256(img)), *W3 = (float *)(w + 2 * align256(img));
        if ((rc = stolt_fft_scan_forward(data, W1, W2, S, T, htaper, vtaper, trunc_int, st))) return rc;
        for (int v = 0; v < nvel; ++v) {
            float *dout = images ? images + v * per_img : W1;
            if ((rc = stolt_fft_scan_velocity(W2, W3, dout, S, T, dt, dx, vels[v], st))) return rc;
            if ((rc = stolt_focus_run(dout, S2, T, win_s, win_t, focus + v * per_focus, part, st))) return rc;
        }
        g_stolt_last = 3;
        return IMPDAR_B200_OK;
    }
    StoltPlans pl;
    rc = get_plans(S, T, st, pl);
    if (rc) return rc;
    g_stolt_last = pl.paired ? 2 : 1;
    float *bufA = (float *)w;  // tapered input, later each velocity's remapped spectrum KK
    float2 *bufKK = (float2 *)w;
    float2 *bufFK = (float2 *)(w + align256(cplx > img ? cplx : img));
    float *scratch = (float *)(w + align256(cplx > img ? cplx : img) + align256(cplx));
    rc = impdar_taper_f32(data, bufA, S, T, 1, htaper, vtaper, trunc_int, stream);
    if (rc) return rc;
    if (pl.paired) {
        IMPDAR_CUFFT(cufftSetStream(pl.c2c2d, st));
        IMPDAR_CUFFT(cufftExecC2C(pl.c2c2d, (cufftComplex *)bufA, (cufftComplex *)bufA, CUFFT_FORWARD));
        count_launch(1);
        StoltPairedParams pp;
        pp.S = S; pp.Th = T / 2; pp.T = T; pp.nz = S / 2;
        pp.norm = (float)(1.0 / ((double)S * (double)T));
        pp.Zh = (const float2 *)bufA;
        for (int v = 0; v < nvel; ++v) {
            float *dout = images ? images + v * per_img : scratch;
            pp.beta_unit = vels[v] * (double)S * dt / (2.0 * (double)T * dx);
            pp.Zq = (float2 *)dout;
            const int rows_per_cta = 32;
            dim3 grid((pp.Th + 127) / 128, (pp.nz + rows_per_cta - 1) / rows_per_cta);
            ktimer_begin("stolt_remap_paired_kernel", st);
            stolt_remap_paired_kernel<<<grid, 128, 0, st>>>(pp, rows_per_cta);
            ktimer_end(st);
            IMPDAR_LAUNCH_CHECK();
            IMPDAR_CUFFT(cufftExecC2C(pl.c2c2d, (cufftComplex *)dout, (cufftComplex *)dout, CUFFT_INVERSE));
            count_launch(1);
            if ((rc = stolt_focus_run(dout, S2, T, win_s, win_t, focus + v * per_focus, part, st))) return rc;
        }
        return IMPDAR_B200_OK;
    }
    IMPDAR_CUFFT(cufftSetStream(pl.r2c, st));
    IMPDAR_CUFFT(cufftSetStream(pl.c2c, st));
    IMPDAR_CUFFT(cufftSetStream(pl.c2r, st));
    IMPDAR_CUFFT(cufftExecR2C(pl.r2c, bufA, (cufftComplex *)bufFK));
    IMPDAR_CUFFT(cufftExecC2C(pl.c2c, (cufftComplex *)bufFK, (cufftComplex *)bufFK, CUFFT_FORWARD));
    count_launch(2);
    StoltRemapParams rp;
    rp.M = M; rp.T = T; rp.nz = S / 2;
    rp.norm = (float)(1.0 / ((double)S2 * (double)T));
    rp.FK = bufFK;
    rp.KK = bufKK;
    for (int v = 0; v < nvel; ++v) {
        float *dout = images ? images + v * per_img : scratch;
        rp.beta_unit = vels[v] * (double)S * dt / (2.0 * (double)T * dx);
        const int rows_per_cta = 32;
        dim3 grid((T + 127) / 128, (M + rows_per_cta - 1) / rows_per_cta);
        ktimer_begin("stolt_remap_kernel", st);
        stolt_remap_kernel<<<grid, 128, 0, st>>>(rp, rows_per_cta);
        ktimer_end(st);
        IMPDAR_LAUNCH_CHECK();
        IMPDAR_CUFFT(cufftExecC2C(pl.c2c, (cufftComplex *)bufKK, (cufftComplex *)bufKK, CUFFT_INVERSE));
        IMPDAR_CUFFT(cufftExecC2R(pl.c2r, (cufftComplex *)bufKK, dout));
        count_launch(2);
        if ((rc = stolt_focus_run(dout, S2, T, win_s, win_t, focus + v * per_focus, part, st))) return rc;
    }
    return IMPDAR_B200_OK;
}

/* Testing hook: 1 forces the generic R2C/C2R pipeline even when the paired-trace one applies. */
int impdar_stolt_force_r2c(int on) {
    g_stolt_mode = on ? 1 : 0;
    return IMPDAR_B200_OK;
}

int impdar_stolt_set_pipeline(int mode) {
    IMPDAR_CHECK_ARG(mode >= 0 && mode <= 3, "stolt_set_pipeline: 0 auto, 1 cuFFT R2C/C2R, 2 cuFFT paired C2C, 3 five-pass kernels");
    g_stolt_mode = mode;
    return IMPDAR_B200_OK;
}

int impdar_stolt_last_pipeline(void) { return g_stolt_last; }

int impdar_stolt_debug_stop_after(int stage) {
    IMPDAR_CHECK_ARG(stage >= 0 && stage <= 5, "stolt_debug_stop_after: stage must be in [0, 5]");
    g_stolt_stop_after = stage;
    return IMPDAR_B200_OK;
}

}  // extern "C"
