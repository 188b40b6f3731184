// Stolt f-k migration as five hand-written HBM sweeps (reference: migrationlib/mig_python.py:126-208).
//
// The cuFFT pipeline of stolt.cu moves ~9 sweeps of the radargram through HBM (taper, three transform passes
// forward, remap, three back).  For power-of-two shapes this file does the whole job in five, which is the
// 40 B/sample model of SURVEY.md 8d:
//
//   P1 rows     taper (mig_python.py:152-157) fused into the load; adjacent traces paired into one complex signal
//               z[s][j] = d[s][2j] + i d[s][2j+1], j = n1*N2 + n2 (N2 = 256); FFT over n1; twiddle      -> W1[s][k1*N2+n2]
//   P2 rows     FFT over n2; untangle the paired transform into the half spectrum D[s][kx], kx in [0, T/2);
//               transposed store, so a wavenumber column becomes contiguous in time                     -> Dt[c][s]
//               (memory column c = k1*N2 + k2 holds kx = k1 + N1*k2; column 0 packs the real kx = 0 and T/2 series)
//   P3 columns  one CTA per wavenumber: FFT over s in shared memory, w -> kz remap with complex linear
//               interpolation and obliquity scaling (:171-200) on both frequency halves, inverse FFT       in place
//   P4 rows     transposed load, tangle, inverse FFT over k2                                               -> W1[s][k1*N2+n2]
//   P5 rows     twiddle, inverse FFT over k1, real image written in place of W1 (the caller's `out`)
//
// All transforms are fp32 Stockham / four-step FFTs with radix-16/32 butterflies in registers (fft_regs.cuh)
// and twiddle tables computed in fp64; the remap coordinate sqrt(j^2 + beta^2) is fp64 (one Newton step on
// the fp32 square root).  tests/stolt_stage_model.py restates every stage in numpy with the same indexing.
#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "fft_regs.cuh"

namespace impdar {
namespace sfft {

using namespace fftr;

constexpr int N2 = 256;      // contiguous sub-transform length of a row
constexpr int NC2 = 16;      // n2 values per P1/P5 tile (128-byte runs)

// ------------------------------------------------------------------------------------------- tables
__global__ void twiddle_table_kernel(cf *__restrict__ tab, int n, int count) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= count) return;
    double s, c;
    sincospi(2.0 * (double)m / (double)n, &s, &c);
    tab[m] = mk((float)c, (float)(-s));  // forward twiddle w_n^m = e^{-2 pi i m / n}
}

// ------------------------------------------------------------------ two-step FFT along the slow axis of a tile
// Element (slot, col) lives at sm[slot * PITCH + (SK ? slot >> 4 : 0) + col]; N = RA * RB slots.  Lanes run over
// `col`, so every access is conflict free.  In place; afterwards slot p holds X[k] with k = p / RB + RA * (p % RB).
template <int PITCH, int SK>
FFTR_DI int slot_addr(int slot) { return slot * PITCH + (SK ? (slot >> 4) : 0); }
template <int RA, int RB>
FFTR_DI int slot_to_k(int p) { return (p / RB) + RA * (p % RB); }
template <int RA, int RB>
FFTR_DI int k_to_slot(int k) { return (k % RA) * RB + (k / RA); }

template <int RA, int RB, int DIR, int PITCH, int SK, int NTHREADS>
FFTR_DI void tile_fft(cf *__restrict__ sm, const cf *__restrict__ tw, int tw_stride, int ncols, int tid) {
    // step 1: radix RA over q for every (r, col); twiddle w_N^{r ka}
    for (int item = tid; item < RB * ncols; item += NTHREADS) {
        const int r = item / ncols, col = item - r * ncols;
        cf v[RA];
#pragma unroll
        for (int q = 0; q < RA; ++q) v[q] = sm[slot_addr<PITCH, SK>(q * RB + r) + col];
        fft_reg<RA, DIR>(v);
        if (RB > 1) {
#pragma unroll
            for (int ka = 1; ka < RA; ++ka) v[ka] = cmul_dir<DIR>(v[ka], tw[(r * ka) * tw_stride]);
        }
#pragma unroll
        for (int ka = 0; ka < RA; ++ka) sm[slot_addr<PITCH, SK>(ka * RB + r) + col] = v[ka];
    }
    __syncthreads();
    if (RB > 1) {
        for (int item = tid; item < RA * ncols; item += NTHREADS) {
            const int ka = item / ncols, col = item - ka * ncols;
            cf v[RB];
#pragma unroll
            for (int r = 0; r < RB; ++r) v[r] = sm[slot_addr<PITCH, SK>(ka * RB + r) + col];
            fft_reg<RB, DIR>(v);
#pragma unroll
            for (int kb = 0; kb < RB; ++kb) sm[slot_addr<PITCH, SK>(ka * RB + kb) + col] = v[kb];
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------- taper
// min(i, n-1-i) / len clipped to 1 (mig_python.py:152-156).  `iceil` = ceil(len) as an int (INT_MAX when len is
// not finite), so the interior - where the weight is exactly 1 - is decided without any fp64 work.
FFTR_DI double taper_w(int i, int n, double len, int iceil) {
    const int m = min(i, n - 1 - i);
    if (m > 0 && m >= iceil) return 1.0;
    double w = (double)m / len;  // 0/0 -> NaN, like numpy
    if (w > 1.0) w = 1.0;
    return w;
}

// ------------------------------------------------------------------------------ P1 / P5: strided row sub-transform
struct RowAParams {
    const float *data;  // P1 input (S, T) real
    cf *W1;             // P1 output / P5 input (S, Th) complex; P5 writes the real image in place
    int S, T, Th, N1, rows_per_cta, batch;
    double htaper, vtaper;
    int hceil, vceil;   // ceil(htaper), ceil(vtaper)
    int trunc_int;
    const cf *twTh;     // w_Th^m, m < Th
};

FFTR_DI void cp_async16(void *smem_dst, const void *gsrc) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gsrc) : "memory");
}
FFTR_DI void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
FFTR_DI void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int TILE_A = 4096;  // complex elements per P1/P5 tile (32 KB), double buffered

// Tile = N1 (all strided sub-transform inputs) x NS rows x 16 consecutive n2, laid out [n1][row][n2] so that every
// global run is 128 contiguous bytes and the transform runs along the slow axis with lanes over (row, n2).
// N1 = 16 * RB: step 1 is radix 16, step 2 radix RB; slot p = ka * RB + kb holds index k = ka + 16 kb.
// Loads are cp.async into a double buffer (the next tile streams in while this one is transformed); every
// address is a per-thread base plus a compile-time offset.
template <int N1, int DIR>
__global__ void __launch_bounds__(256, 2) stolt_rowA_kernel(const __grid_constant__ RowAParams p) {
    constexpr int RB = N1 / 16;
    constexpr int NS = TILE_A / (N1 * NC2);  // rows per tile = 16 / RB
    constexpr int COLS = NS * NC2;           // 256 / RB
    static_assert(RB >= 1 && RB <= 16 && NS * RB == 16, "N1 must be 16, 32, 64, 128 or 256");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cf *tiles = reinterpret_cast<cf *>(smem_raw);  // 2 x TILE_A
    cf *tab = tiles + 2 * TILE_A;                  // [N1][NC2]: w_Th^{k1 n2}
    cf *tw = tab + N1 * NC2;                       // [N1]: w_N1^m
    const int tid = threadIdx.x;
    const int n2b = blockIdx.x * NC2;
    for (int i = tid; i < N1 * NC2; i += 256) {
        const int k1 = i / NC2, n2 = n2b + (i % NC2);
        tab[i] = p.twTh[(int)(((long long)k1 * n2) % p.Th)];
    }
    for (int i = tid; i < N1; i += 256) tw[i] = p.twTh[i * N2];

    const int row_begin = blockIdx.y * p.rows_per_cta;
    const int ntiles = (min(p.S, row_begin + p.rows_per_cta) - row_begin) / NS;

    // ---- per-thread constants of the load: 16-byte chunk c = i * 256 + tid -> (n1, row, piece)
    const int l_piece = tid & 7, l_sl = (tid >> 3) % NS, l_n1 = (tid >> 3) / NS;
    const size_t boff = (size_t)blockIdx.z * p.S * p.T;  // profile of the batch (floats)
    const float *gsrc = (DIR < 0 ? p.data : reinterpret_cast<const float *>(p.W1)) + boff + (size_t)(row_begin + l_sl) * p.T +
                        2 * (l_n1 * N2 + n2b) + l_piece * 4;
    constexpr int L_STEP = (32 / NS) * N2 * 2;  // floats between the chunks of consecutive i
    // ---- per-thread constants of the store: element e = i * 256 + tid -> (slot, row, n2l); slot = i * RB + s_pt
    const int s_n2l = tid & 15, s_sl = (tid >> 4) % NS, s_pt = (tid >> 4) / NS;
    cf *gdst = p.W1 + boff / 2 + (size_t)(row_begin + s_sl) * p.Th + (size_t)(16 * s_pt) * N2 + n2b + s_n2l;
    const cf *tabs = tab + (16 * s_pt) * NC2 + s_n2l;
    // ---- taper zones of this CTA's columns (P1): weights differ from 1 only there
    const bool hzone = (2 * n2b < max(p.hceil, 1)) || (p.T - 2 * ((N1 - 1) * N2 + n2b + NC2) < max(p.hceil, 1)) ||
                       p.trunc_int;

    auto issue = [&](int t) {
        cf *dst = tiles + (t & 1) * TILE_A;
        const float *src = gsrc + (size_t)t * NS * p.T;
#pragma unroll
        for (int i = 0; i < TILE_A / 2 / 256; ++i) cp_async16(reinterpret_cast<float4 *>(dst) + i * 256 + tid, src + i * L_STEP);
        cp_async_commit();
    };
    if (ntiles > 0) issue(0);
    __syncthreads();  // tables
    for (int t = 0; t < ntiles; ++t) {
        if (t + 1 < ntiles) {
            issue(t + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        cf *tile = tiles + (t & 1) * TILE_A;
        const int s0 = row_begin + t * NS;
        if (DIR < 0) {
            const bool vzone = (s0 < max(p.vceil, 1)) || (p.S - s0 - NS < max(p.vceil, 1));
            if (hzone || vzone) {  // block-uniform: apply the taper to this tile in shared memory
                for (int e = tid; e < TILE_A; e += 256) {
                    const int n2l = e % NC2, sl = (e / NC2) % NS, n1 = e / COLS;
                    const int s = s0 + sl, x = 2 * (n1 * N2 + n2b + n2l);
                    const double v = taper_w(s, p.S, p.vtaper, p.vceil);
                    const double h0 = taper_w(x, p.T, p.htaper, p.hceil), h1 = taper_w(x + 1, p.T, p.htaper, p.hceil);
                    const cf d = tile[e];
                    double a = (double)d.x * h0 * v, b = (double)d.y * h1 * v;  // (data * H) * V, mig_python.py:157
                    if (p.trunc_int) {
                        a = trunc(a);
                        b = trunc(b);
                    }
                    tile[e] = mk((float)a, (float)b);
                }
                __syncthreads();
            }
        }
        // ---- step 1: radix 16 over q (slots q * RB + r) for every (r, col); P5 first multiplies by conj(w_Th^{k1 n2})
        {
            constexpr int ITEMS = RB * COLS / 256;  // = 1
            static_assert(ITEMS == 1, "one radix-16 item per thread");
            const int r = tid / COLS, col = tid % COLS;
            cf v[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = tile[(q * RB + r) * COLS + col];
            if (DIR > 0) {
                const cf *tq = tab + r * NC2 + (col % NC2);
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = cmul_conj(v[q], tq[q * RB * NC2]);
            }
            fft_reg<16, DIR>(v);
            if (RB > 1) {
#pragma unroll
                for (int ka = 1; ka < 16; ++ka) v[ka] = cmul_dir<DIR>(v[ka], tw[r * ka]);
            }
#pragma unroll
            for (int ka = 0; ka < 16; ++ka) tile[(ka * RB + r) * COLS + col] = v[ka];
        }
        __syncthreads();
        if (RB > 1) {
            constexpr int ITEMS = 16 * COLS / 256;  // = 16 / RB
#pragma unroll
            for (int it = 0; it < ITEMS; ++it) {
                const int item = tid + it * 256;
                const int ka = item / COLS, col = item % COLS;
                cf v[RB];
#pragma unroll
                for (int r = 0; r < RB; ++r) v[r] = tile[(ka * RB + r) * COLS + col];
                fft_reg<RB, DIR>(v);
#pragma unroll
                for (int kb = 0; kb < RB; ++kb) tile[(ka * RB + kb) * COLS + col] = v[kb];
            }
            __syncthreads();
        }
        // ---- store: slot i * RB + s_pt holds index k = i + 16 s_pt
        {
            cf *dst = gdst + (size_t)t * NS * p.Th;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                cf val = tile[i * 256 + tid];
                if (DIR < 0) val = cmul(val, tabs[i * NC2]);
                dst[i * N2] = val;  // P5: (re, im) = (out[s][2j], out[s][2j+1])
            }
        }
        __syncthreads();  // the tile buffer is refilled by the prefetch of the next iteration
    }
}

// --------------------------------------------------------- P2 / P4: contiguous row sub-transform + (un)tangle + transpose
struct RowBParams {
    cf *W1;   // (S, Th)
    cf *Dt;   // (Th, S)
    int S, T, Th, N1, batch;
    const cf *tw512;  // w_512^m
};

constexpr int RB_PITCH = 33;
constexpr int RB_TILE = N2 * RB_PITCH + 16;

// Generic version: handles the self-paired sub-transforms k1 = 0 and k1 = N1/2 (blockIdx.x = 0, 1).
template <int DIR>
__global__ void __launch_bounds__(256) stolt_rowB_self_kernel(const __grid_constant__ RowBParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cf *tile = reinterpret_cast<cf *>(smem_raw);
    cf *tw = tile + RB_TILE;  // [512]
    const int tid = threadIdx.x;
    const int k1a = blockIdx.x * (p.N1 / 2), k1b = (p.N1 - k1a) % p.N1;
    const size_t boff = (size_t)blockIdx.z * p.S * p.Th;  // profile of the batch (complex elements)
    cf *const W1 = p.W1 + boff, *const Dt = p.Dt + boff;
    const int nk = (k1a == k1b) ? 1 : 2;
    const int ncols = nk * 16;
    const int s0 = blockIdx.y * 16;
    for (int i = tid; i < 512; i += 256) tw[i] = p.tw512[i];
    double sn, cs;
    sincospi(2.0 * (double)k1a / (double)p.T, &sn, &cs);
    const cf wA = mk((float)cs, (float)(-sn));  // w_T^{k1a}
    const size_t S = (size_t)p.S;

    if (DIR < 0) {
        for (int e = tid; e < nk * 4096; e += 256) {
            const int n2 = e & 255, sl = (e >> 8) & 15, kidx = e >> 12;
            const int k1 = kidx ? k1b : k1a;
            tile[slot_addr<RB_PITCH, 1>(n2) + kidx * 16 + sl] = W1[(size_t)(s0 + sl) * p.Th + k1 * N2 + n2];
        }
    } else {
        for (int e = tid; e < nk * 4096; e += 256) {
            const int sl = e & 15, k2 = (e >> 4) & 255, kidx = e >> 12;
            const int k1 = kidx ? k1b : k1a;
            tile[slot_addr<RB_PITCH, 1>(k2) + kidx * 16 + sl] = Dt[((size_t)k1 * N2 + k2) * S + s0 + sl];
        }
    }
    __syncthreads();
    if (DIR < 0) tile_fft<16, 16, DIR, RB_PITCH, 1, 256>(tile, tw, 2, ncols, tid);

    // pairs (k1a, k2) <-> (k1b, k2p): the columns holding kx and T/2 - kx
    const int npair_k2 = (nk == 2) ? 256 : (k1a == 0 ? 129 : 128);
    for (int q = tid; q < npair_k2 * 16; q += 256) {
        const int sl = q & 15, k2 = q >> 4;
        const int k2p = (k1a == 0) ? ((256 - k2) & 255) : (255 - k2);
        const int colA = sl, colB = (nk == 2 ? 16 : 0) + sl;
        // forward: the transform output sits in digit-transposed slots; inverse: natural slots (input of the IFFT)
        const int sA = DIR < 0 ? k_to_slot<16, 16>(k2) : k2;
        const int sB = DIR < 0 ? k_to_slot<16, 16>(k2p) : k2p;
        const int aA = slot_addr<RB_PITCH, 1>(sA) + colA, aB = slot_addr<RB_PITCH, 1>(sB) + colB;
        const cf zA = tile[aA], zB = tile[aB];
        const bool self = (nk == 1) && (k2p == k2);
        const cf wk = cmul(wA, tw[k2]);  // w_T^{kx}, kx = k1a + N1 k2
        if (DIR < 0) {
            const size_t oA = ((size_t)k1a * N2 + k2) * S + s0 + sl;
            if (k1a == 0 && k2 == 0) {
                Dt[oA] = mk(zA.x + zA.y, zA.x - zA.y);  // (D[0], D[T/2]), both real
            } else {
                const cf e = mk(0.5f * (zA.x + zB.x), 0.5f * (zA.y - zB.y));    // (zA + conj zB) / 2
                const cf o = mk(0.5f * (zA.y + zB.y), -0.5f * (zA.x - zB.x));   // (zA - conj zB) / (2i)
                Dt[oA] = cadd(e, cmul(wk, o));
                if (!self) {
                    const cf wkb = mk(-wk.x, wk.y);  // w_T^{T/2 - kx} = -conj(w_T^{kx})
                    const size_t oB = ((size_t)k1b * N2 + k2p) * S + s0 + sl;
                    Dt[oB] = cadd(cconj(e), cmul(wkb, cconj(o)));
                }
            }
        } else {
            if (k1a == 0 && k2 == 0) {
                tile[aA] = mk(zA.x + zA.y, zA.x - zA.y);
            } else {
                // Zq[k] = (G[k] + conj G[k']) + i (G[k] - conj G[k']) conj(w_T^k)
                const cf eA = mk(zA.x + zB.x, zA.y - zB.y);
                const cf dA = cmul_dir<1>(mk(zA.x - zB.x, zA.y + zB.y), wk);
                tile[aA] = mk(eA.x - dA.y, eA.y + dA.x);
                if (!self) {
                    const cf wkb = mk(-wk.x, wk.y);
                    const cf eB = mk(zB.x + zA.x, zB.y - zA.y);
                    const cf dB = cmul_dir<1>(mk(zB.x - zA.x, zB.y + zA.y), wkb);
                    tile[aB] = mk(eB.x - dB.y, eB.y + dB.x);
                }
            }
        }
    }
    if (DIR > 0) {
        __syncthreads();
        tile_fft<16, 16, DIR, RB_PITCH, 1, 256>(tile, tw, 2, ncols, tid);
        for (int e = tid; e < nk * 4096; e += 256) {
            const int n2 = e & 255, sl = (e >> 8) & 15, kidx = e >> 12;
            const int k1 = kidx ? k1b : k1a;
            W1[(size_t)(s0 + sl) * p.Th + k1 * N2 + n2] =
                tile[slot_addr<RB_PITCH, 1>(k_to_slot<16, 16>(n2)) + kidx * 16 + sl];
        }
    }
}

FFTR_DI void cp_async8(void *smem_dst, const void *gsrc) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gsrc) : "memory");
}

// Fast version for the sub-transform pairs (k1, N1 - k1), k1 = 1 .. N1/2 - 1 (blockIdx.x + 1): 32 columns
// (2 sub-transforms x 16 rows), every shared-memory address is a per-thread base plus a compile-time offset.
template <int DIR>
__global__ void __launch_bounds__(256, 3) stolt_rowB_kernel(const __grid_constant__ RowBParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cf *tile = reinterpret_cast<cf *>(smem_raw);
    cf *tw = tile + RB_TILE;  // [512]: w_512^m
    const int tid = threadIdx.x;
    const int k1a = blockIdx.x + 1, k1b = p.N1 - k1a;
    const int s0 = blockIdx.y * 16;
    const size_t S = (size_t)p.S;
    const size_t boff = (size_t)blockIdx.z * p.S * p.Th;  // profile of the batch (complex elements)
    cf *const W1 = p.W1 + boff, *const Dt = p.Dt + boff;
    const int h = tid >> 4, sl = tid & 15;
    constexpr int QS = 16 * RB_PITCH + 1;  // address step between slots q*16 + r and (q+1)*16 + r

    if (DIR < 0) {
        // W1[(s0 + row)][k1*256 + n2] -> tile[slot n2][kidx*16 + row]; thread = n2
        const cf *srcA = W1 + (size_t)s0 * p.Th + k1a * N2 + tid;
        const cf *srcB = W1 + (size_t)s0 * p.Th + k1b * N2 + tid;
        cf *dst = tile + slot_addr<RB_PITCH, 1>(tid);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            cp_async8(dst + i, srcA + (size_t)i * p.Th);
            cp_async8(dst + 16 + i, srcB + (size_t)i * p.Th);
        }
    } else {
        // Dt[k1*256 + k2][s0 + row] -> tile[slot k2][kidx*16 + row]; thread = (k2 mod 16 = h, row = sl)
        const cf *srcA = Dt + ((size_t)k1a * N2 + h) * S + s0 + sl;
        const cf *srcB = Dt + ((size_t)k1b * N2 + h) * S + s0 + sl;
        cf *dst = tile + h * RB_PITCH + sl;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            cp_async8(dst + i * QS, srcA + (size_t)i * 16 * S);
            cp_async8(dst + i * QS + 16, srcB + (size_t)i * 16 * S);
        }
    }
    cp_async_commit();
    for (int i = tid; i < 512; i += 256) tw[i] = p.tw512[i];
    double sn, cs;
    sincospi(2.0 * (double)k1a / (double)p.T, &sn, &cs);
    const cf wA = mk((float)cs, (float)(-sn));  // w_T^{k1a}
    cp_async_wait<0>();
    __syncthreads();

    auto fft256 = [&]() {
        // step 1: radix 16 over q (slots q*16 + r), twiddle w_256^{r ka}; items (r, col): col = tid & 31, r = tid>>5 + 8 it
#pragma unroll
        for (int it = 0; it < 2; ++it) {
            const int r = (tid >> 5) + 8 * it, col = tid & 31;
            cf *b = tile + r * RB_PITCH + col;
            cf v[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = b[q * QS];
            fft_reg<16, DIR>(v);
#pragma unroll
            for (int ka = 1; ka < 16; ++ka) v[ka] = cmul_dir<DIR>(v[ka], tw[2 * r * ka]);
#pragma unroll
            for (int ka = 0; ka < 16; ++ka) b[ka * QS] = v[ka];
        }
        __syncthreads();
        // step 2: radix 16 over r (slots ka*16 + r); items (ka, col)
#pragma unroll
        for (int it = 0; it < 2; ++it) {
            const int ka = (tid >> 5) + 8 * it, col = tid & 31;
            cf *b = tile + ka * QS + col;
            cf v[16];
#pragma unroll
            for (int r = 0; r < 16; ++r) v[r] = b[r * RB_PITCH];
            fft_reg<16, DIR>(v);
#pragma unroll
            for (int kb = 0; kb < 16; ++kb) b[kb * RB_PITCH] = v[kb];
        }
        __syncthreads();
    };

    if (DIR < 0) {
        fft256();
        // untangle pairs: A = (k1a, k2), B = (k1b, 255 - k2), k2 = 16 it + h; slot of k2 = h*16 + it
        const cf *tA = tile + (h * 16) * RB_PITCH + h + sl;
        const cf *tB = tile + ((15 - h) * 16 + 15) * RB_PITCH + (15 - h) + 16 + sl;
        cf *gA = Dt + ((size_t)k1a * N2 + h) * S + s0 + sl;
        cf *gB = Dt + ((size_t)k1b * N2 + 255 - h) * S + s0 + sl;
#pragma unroll
        for (int it = 0; it < 16; ++it) {
            const cf zA = tA[it * RB_PITCH], zB = tB[-it * RB_PITCH];
            const cf wk = cmul(wA, tw[h + 16 * it]);  // w_T^{kx}, kx = k1a + N1 k2
            const cf e = cscale(cadd(zA, cconj(zB)), 0.5f);          // (zA + conj zB) / 2
            const cf o = cscale(cmulni(csub(zA, cconj(zB))), 0.5f);   // (zA - conj zB) / (2i)
            gA[(size_t)it * 16 * S] = cadd(e, cmul(wk, o));
            const cf wkb = mk(-wk.x, wk.y);  // w_T^{T/2 - kx} = -conj(w_T^{kx})
            gB[-(ptrdiff_t)((size_t)it * 16 * S)] = cadd(cconj(e), cmul(wkb, cconj(o)));
        }
    } else {
        // tangle pairs in place (natural slots): A at slot k2 = 16 it + h, B at slot 255 - k2
        cf *tA = tile + h * RB_PITCH + sl;
        cf *tB = tile + (255 - h) * RB_PITCH + 15 + 16 + sl;
#pragma unroll
        for (int it = 0; it < 16; ++it) {
            const cf zA = tA[it * QS], zB = tB[-it * QS];
            const cf wk = cmul(wA, tw[h + 16 * it]);
            // Zq[k] = (G[k] + conj G[k']) + i (G[k] - conj G[k']) conj(w_T^k)
            const cf eA = cadd(zA, cconj(zB));
            const cf dA = cmul_conj(csub(zA, cconj(zB)), wk);
            tA[it * QS] = cadd(eA, cmuli(dA));
            const cf wkb = mk(-wk.x, wk.y);
            const cf eB = cadd(zB, cconj(zA));
            const cf dB = cmul_conj(csub(zB, cconj(zA)), wkb);
            tB[-it * QS] = cadd(eB, cmuli(dB));
        }
        __syncthreads();
        fft256();
        // W1[(s0 + row)][k1*256 + n2] <- tile[slot of n2][kidx*16 + row]; thread = n2, slot = (n2 & 15)*16 + (n2 >> 4)
        const cf *src = tile + slot_addr<RB_PITCH, 1>((tid & 15) * 16 + (tid >> 4));
        cf *dA = W1 + (size_t)s0 * p.Th + k1a * N2 + tid;
        cf *dB = W1 + (size_t)s0 * p.Th + k1b * N2 + tid;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            dA[(size_t)i * p.Th] = src[i];
            dB[(size_t)i * p.Th] = src[16 + i];
        }
    }
}

// -------------------------------------------------------------------- P3: column transform + remap + inverse
struct ColParams {
    cf *Dt;  // (Th, S), in place
    int Th, N1, T, ncols;  // ncols = batch * Th
    const cf *twS;  // w_S^k, k < 256
    const cf *tw2;  // w_256^{k t}, [t < 16][k < 16]
    double beta_unit;
    float norm;
};

FFTR_DI int padi(int a) { return a + (a >> 4); }

struct RemapCol {
    int Bi;       // floor(beta^2), saturated at 2^30
    float Bf;     // beta^2 - Bi
    float b2f;    // beta^2
    float norm;
};

// Source row i0, weights w0 = (1 - a) sc, w1 = a sc of output row jj (1 <= jj < NZ) of a column with beta^2 = Bi + Bf:
// f = sqrt(jj^2 + beta^2) (mig_python.py:188), a = f - i0 = (jj^2 + beta^2 - i0^2) / (f + i0) with the numerator in
// exact integer arithmetic (no fp64), sc = jj / f * norm (:197); beyond Nyquist the spline is clamped: i0 = NZ-1, a = 1.
template <int NZ>
FFTR_DI void remap_coord(int jj, float jjf, const RemapCol &rc, int &i0, float &w0, float &w1) {
    const int qi = jj * jj + rc.Bi;
    const float qf = fmaf(jjf, jjf, rc.b2f);
    float rs;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(qf));
    const float r0 = qf * rs;
    const float m = (r0 - 0.5f) + 12582912.0f;             // round(r0 - 0.5): floor(r0) or one off
    int i = __float_as_int(m) - 0x4B400000;
    float fi = m - 12582912.0f;
    if (i * i > qi) {
        --i;
        fi -= 1.0f;
    } else if ((i + 1) * (i + 1) <= qi) {
        ++i;
        fi += 1.0f;
    }
    const float num = (float)(qi - i * i) + rc.Bf;
    float a = __fdividef(num, r0 + fi);
    if (qi >= NZ * NZ) {
        i = NZ - 1;
        a = 1.0f;
    }
    const float sc = jjf * rs * rc.norm;
    i0 = i;
    w1 = a * sc;
    w0 = sc - w1;
}

struct NoHook {
    FFTR_DI void operator()() const {}
};

// 1-D TMA (cp.async.bulk) of one whole column into shared memory, completion counted on an mbarrier.
FFTR_DI void mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
FFTR_DI void bulk_load_column(void *smem_dst, const void *gsrc, unsigned bytes, unsigned long long *bar) {
    const unsigned sd = (unsigned)__cvta_generic_to_shared(smem_dst), sb = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy reads of the buffer are ordered before the copy
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sb), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sd), "l"(gsrc),
                 "r"(bytes), "r"(sb)
                 : "memory");
}
FFTR_DI void mbar_wait(unsigned long long *bar, unsigned parity) {
    const unsigned sb = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(sb),
        "r"(parity)
        : "memory");
}

// One Stockham step of radix R (Ls = 16 or 256) on the padded shared-memory sequence: item j reads x[j + t S/R],
// multiplies by w_{Ls R}^{k t} (k = j mod Ls), transforms, and writes y[(j - k) R + k + t Ls] - to shared memory
// again or, for the last inverse step, to the global column.
template <int S, int R, int LS, int DIR, int NT, bool TO_GLOBAL, class AfterLoad = NoHook>
FFTR_DI void stockham_step(cf *__restrict__ buf, const cf *__restrict__ twS, const cf *__restrict__ tw2, int tid,
                           cf *__restrict__ gdst, AfterLoad after_load = AfterLoad()) {
    constexpr int ITEMS = S / R / NT;
    constexpr int STR = S / R;  // multiple of 16
    static_assert(ITEMS >= 1 && STR % 16 == 0, "shape");
    cf v[ITEMS][R];
#pragma unroll
    for (int it = 0; it < ITEMS; ++it) {
        const int j = tid + it * NT;
        const cf *src = buf + padi(j);
#pragma unroll
        for (int t = 0; t < R; ++t) v[it][t] = src[t * (STR + STR / 16)];
    }
    if (!TO_GLOBAL) __syncthreads();
    after_load();  // every element this thread needs is in registers
#pragma unroll
    for (int it = 0; it < ITEMS; ++it) {
        const int j = tid + it * NT;
        const int k = j & (LS - 1);
        if (LS == 16) {
            const cf *tq = tw2 + k;  // [t][k]: lanes run over k, conflict free
#pragma unroll
            for (int t = 1; t < R; ++t) v[it][t] = cmul_dir<DIR>(v[it][t], tq[t * 16]);
        } else {
            apply_powers<R, DIR>(v[it], twS[k]);
        }
        fft_reg<R, DIR>(v[it]);
        const int base = (j - k) * R + k;
        if (TO_GLOBAL) {
#pragma unroll
            for (int t = 0; t < R; ++t) gdst[base + t * LS] = v[it][t];
        } else {
            cf *dst = buf + padi(base);
#pragma unroll
            for (int t = 0; t < R; ++t) dst[t * (LS + LS / 16)] = v[it][t];
        }
    }
    if (!TO_GLOBAL) __syncthreads();
}

// S = 16 * 16 * R3.  NT = S/32 threads; thread tid owns the first-step items jA, jB (radix 16, elements j + t S/16) with
// jB the frequency mirror of jA: element (jA, t) <-> (jB, 15 - t), so every remap coordinate serves two outputs.
//
// PF (prefetch): the column is brought into the (then idle) transform buffer by one 1-D TMA bulk copy issued as soon as the
// previous column's last step has its operands in registers, so the load overlaps that step's butterflies and global
// stores instead of being waited for at the top of the loop; without PF the first step loads straight from global memory.
//
// SPLIT (velocity scan): the prefetch reads the column from `src` and the last step stores to p.Dt, so the forward
// spectrum in `src` survives for the next velocity.  Without SPLIT the column is transformed in place in p.Dt and `src`
// is unused; those instantiations compile to the same SASS as before SPLIT existed.
#ifndef COL_MINB_8192
#define COL_MINB_8192 2
#define COL_MINB_4096 4
#define COL_MINB_SMALL 8
#endif
#define COL_MINB(S) ((S) >= 8192 ? COL_MINB_8192 : ((S) >= 4096 ? COL_MINB_4096 : COL_MINB_SMALL))
template <int S, int R3, bool PF, bool SPLIT>
__global__ void __launch_bounds__(S / 32, COL_MINB(S)) stolt_col_kernel(const __grid_constant__ ColParams p,
                                                                         const cf *__restrict__ src) {
    constexpr int NT = S / 32, NI = S / 16, NZ = S / 2;
    static_assert(16 * 16 * R3 == S && NT >= 32, "factorisation");
    static_assert(PF || !SPLIT, "the split variant loads through the prefetch");
    const cf *const srcb = SPLIT ? src : p.Dt;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cf *buf = reinterpret_cast<cf *>(smem_raw);
    cf *twS = buf + (S + S / 16);
    cf *tw2 = twS + 256;
    unsigned long long *bar = reinterpret_cast<unsigned long long *>(tw2 + 256);
    const int tid = threadIdx.x;
    for (int i = tid; i < 256; i += NT) {
        twS[i] = p.twS[i];
        tw2[i] = p.tw2[i];
    }
    const int jA = (tid == 0) ? 0 : tid, jB = (tid == 0) ? NI / 2 : NI - tid;
    unsigned phase = 0;
    if (PF && tid == 0) {
        mbar_init(bar, 1);
        if ((int)blockIdx.x < p.ncols) bulk_load_column(buf, srcb + (size_t)blockIdx.x * S, S * (unsigned)sizeof(cf), bar);
    }
    if (PF) __syncthreads();  // the barrier is initialised before anyone waits on it

    for (int cb = blockIdx.x; cb < p.ncols; cb += gridDim.x) {
        const int c = cb % p.Th;  // column within its profile
        cf *col = p.Dt + (size_t)cb * S;
        cf vA[16], vB[16];
        // ---- forward step 1 (radix 16, no twiddle) from the prefetched copy, or straight from global memory
        if (PF) {
            mbar_wait(bar, phase);
            phase ^= 1u;
#pragma unroll
            for (int t = 0; t < 16; ++t) vA[t] = buf[jA + t * NI];
#pragma unroll
            for (int t = 0; t < 16; ++t) vB[t] = buf[jB + t * NI];
        } else {
#pragma unroll
            for (int t = 0; t < 16; ++t) vA[t] = __ldcs(col + jA + t * NI);
#pragma unroll
            for (int t = 0; t < 16; ++t) vB[t] = __ldcs(col + jB + t * NI);
        }
        fft_reg<16, -1>(vA);
        fft_reg<16, -1>(vB);
        __syncthreads();  // the previous column's last shared-memory reads are done (also orders the table fill)
#pragma unroll
        for (int t = 0; t < 16; ++t) buf[17 * jA + t] = vA[t];
#pragma unroll
        for (int t = 0; t < 16; ++t) buf[17 * jB + t] = vB[t];
        __syncthreads();
        stockham_step<S, 16, 16, -1, NT, false>(buf, twS, tw2, tid, nullptr);
        stockham_step<S, R3, 256, -1, NT, false>(buf, twS, tw2, tid, nullptr);
        // buf now holds F[w], natural order (padded)

        // ---- remap fused with inverse step 1
        const int kx = (c / N2) + p.N1 * (c % N2);
        RemapCol rc;
        {
            const double beta = p.beta_unit * (double)(c == 0 ? p.T / 2 : kx);
            const double b2 = beta * beta;
            const double bfl = floor(fmin(b2, 1073741824.0));
            rc.Bi = (int)bfl;
            rc.Bf = (b2 < 1073741824.0) ? (float)(b2 - bfl) : 0.f;
            rc.b2f = (float)b2;
            rc.norm = p.norm;
        }
        // positive-frequency output row jj and its mirror S - jj from one coordinate evaluation
        auto eval = [&](int jj, float jjf, cf &qpos, cf &qneg) {
            int i0;
            float w0, w1;
            remap_coord<NZ>(jj, jjf, rc, i0, w0, w1);
            if (c != 0) {
                qpos = clerp(buf[padi(i0)], w0, buf[padi(i0 + 1)], w1);
                qneg = clerp(buf[padi((S - i0) & (S - 1))], w0, buf[padi(S - i0 - 1)], w1);
            } else {
                // packed column: Z = F0 + i FN with F0 (kx = 0) and FN (kx = T/2) Hermitian in w
                const cf zj = buf[padi(jj)], zjm = cconj(buf[padi((S - jj) & (S - 1))]);
                const cf z0 = buf[padi(i0)], z0m = cconj(buf[padi((S - i0) & (S - 1))]);
                const cf z1 = buf[padi(i0 + 1)], z1m = cconj(buf[padi(S - i0 - 1)]);
                const cf q0 = cscale(cadd(zj, zjm), 0.5f * rc.norm);  // kx = 0: beta = 0, w' = w, scale 1
                const cf n0 = cscale(cmulni(csub(z0, z0m)), 0.5f);    // FN[i0]
                const cf n1 = cscale(cmulni(csub(z1, z1m)), 0.5f);    // FN[i0 + 1]
                const cf qn = clerp(n0, w0, n1, w1);
                qpos = cadd(q0, cmuli(qn));                 // Q0 + i QN
                qneg = cadd(cconj(q0), cmuli(cconj(qn)));   // both Hermitian
            }
        };
        {
            // One code path for every thread (thread 0 owns the self-mirrored items 0 and NI/2; a separate branch for it
            // would make warp 0 run the remap twice while the rest of the CTA waits at the barrier).  nA / nB are the
            // mirror-row outputs of the jA / jB evaluations: element (jA, t) <-> (jB, 15 - t) in general; for thread 0
            // (0, t) <-> (0, 16 - t) and (NI/2, t) <-> (NI/2, 15 - t), and the rows w = 0 and w = S/2 are zero.
            const bool self = (tid == 0);
            const float fA = (float)jA, fB = (float)jB;
            cf nA[8], nB[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                eval(jA + t * NI, fA + (float)(t * NI), vA[t], nA[t]);
                eval(jB + t * NI, fB + (float)(t * NI), vB[t], nB[t]);
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) vB[15 - t] = self ? nB[t] : nA[t];
#pragma unroll
            for (int t = 0; t < 7; ++t) vA[15 - t] = self ? nA[t + 1] : nB[t];
            vA[8] = self ? mk(0.f, 0.f) : nB[7];
            if (self) vA[0] = mk(0.f, 0.f);
        }
        fft_reg<16, 1>(vA);
        fft_reg<16, 1>(vB);
        __syncthreads();
#pragma unroll
        for (int t = 0; t < 16; ++t) buf[17 * jA + t] = vA[t];
#pragma unroll
        for (int t = 0; t < 16; ++t) buf[17 * jB + t] = vB[t];
        __syncthreads();
        stockham_step<S, 16, 16, 1, NT, false>(buf, twS, tw2, tid, nullptr);
        if (PF) {
            const int nxt = cb + gridDim.x;
            stockham_step<S, R3, 256, 1, NT, true>(buf, twS, tw2, tid, col, [&]() {
                __syncthreads();  // nobody reads the buffer any more: the next column may land in it
                if (tid == 0 && nxt < p.ncols) bulk_load_column(buf, srcb + (size_t)nxt * S, S * (unsigned)sizeof(cf), bar);
            });
        } else {
            stockham_step<S, R3, 256, 1, NT, true>(buf, twS, tw2, tid, col);
        }
    }
}

// ---------------------------------------------------------------------------------------- host side
struct Tables {
    cf *twTh = nullptr, *tw512 = nullptr, *twS = nullptr, *tw2 = nullptr;
};

__global__ void twiddle_prod_table_kernel(cf *__restrict__ tab) {  // w_256^{k t}, [t < 16][k < 16]
    const int t = threadIdx.x >> 4, k = threadIdx.x & 15;
    double s, c;
    sincospi(2.0 * (double)(k * t) / 256.0, &s, &c);
    tab[threadIdx.x] = mk((float)c, (float)(-s));
}
static std::map<std::tuple<int, int, int>, Tables> g_tables;  // (device, S, T)
static std::mutex g_tables_mu;


static int get_tables(int S, int T, cudaStream_t st, Tables &out) {
    int dev = 0;
    IMPDAR_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_tables_mu);
    auto key = std::make_tuple(dev, S, T);
    auto it = g_tables.find(key);
    if (it != g_tables.end()) {
        out = it->second;
        return IMPDAR_B200_OK;
    }
    const int Th = T / 2;
    const int nS = 256;
    cf *mem = nullptr;
    IMPDAR_CUDA(cudaMalloc((void **)&mem, (size_t)(Th + 512 + nS + 256) * sizeof(cf)));
    Tables t;
    t.twTh = mem;
    t.tw512 = mem + Th;
    t.twS = mem + Th + 512;
    t.tw2 = mem + Th + 512 + nS;
    twiddle_table_kernel<<<(Th + 255) / 256, 256, 0, st>>>(t.twTh, Th, Th);
    IMPDAR_LAUNCH_CHECK();
    twiddle_table_kernel<<<2, 256, 0, st>>>(t.tw512, 512, 512);
    IMPDAR_LAUNCH_CHECK();
    twiddle_table_kernel<<<(nS + 255) / 256, 256, 0, st>>>(t.twS, S, nS);
    IMPDAR_LAUNCH_CHECK();
    twiddle_prod_table_kernel<<<1, 256, 0, st>>>(t.tw2);
    IMPDAR_LAUNCH_CHECK();
    IMPDAR_CUDA(cudaStreamSynchronize(st));  // once per shape: other streams may use the tables right away
    g_tables[key] = t;
    out = t;
    return IMPDAR_B200_OK;
}

template <int N1, int DIR>
static int launch_rowA(const RowAParams &p, cudaStream_t st) {
    const size_t smem = (size_t)(2 * TILE_A + N1 * NC2 + N1) * sizeof(cf);
    static bool attr_done[IMPDAR_MAX_DEVICES];
    const int dev = current_device_slot();
    if (!attr_done[dev]) {
        IMPDAR_CUDA(cudaFuncSetAttribute(stolt_rowA_kernel<N1, DIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    dim3 grid(N2 / NC2, (p.S + p.rows_per_cta - 1) / p.rows_per_cta, p.batch);
    ktimer_begin("stolt_rowA_kernel", st);
    stolt_rowA_kernel<N1, DIR><<<grid, 256, smem, st>>>(p);
    ktimer_end(st);
    IMPDAR_LAUNCH_CHECK();
    return IMPDAR_B200_OK;
}

template <int DIR>
static int dispatch_rowA(const RowAParams &p, cudaStream_t st) {
    switch (p.N1) {
        case 16: return launch_rowA<16, DIR>(p, st);
        case 32: return launch_rowA<32, DIR>(p, st);
        case 64: return launch_rowA<64, DIR>(p, st);
        case 128: return launch_rowA<128, DIR>(p, st);
        case 256: return launch_rowA<256, DIR>(p, st);
    }
    set_error("stolt: unsupported row split N1 = %d", p.N1);
    return IMPDAR_B200_EINVAL;
}

template <int DIR>
static int launch_rowB(const RowBParams &p, cudaStream_t st) {
    const size_t smem = (size_t)(RB_TILE + 512) * sizeof(cf);
    static bool attr_done[IMPDAR_MAX_DEVICES];
    const int dev = current_device_slot();
    if (!attr_done[dev]) {
        IMPDAR_CUDA(cudaFuncSetAttribute(stolt_rowB_kernel<DIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        IMPDAR_CUDA(cudaFuncSetAttribute(stolt_rowB_self_kernel<DIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    dim3 grid(p.N1 / 2 - 1, p.S / 16, p.batch);
    ktimer_begin("stolt_rowB_kernel", st);
    stolt_rowB_kernel<DIR><<<grid, 256, smem, st>>>(p);
    ktimer_end(st);
    IMPDAR_LAUNCH_CHECK();
    dim3 grid_self(2, p.S / 16, p.batch);  // k1 = 0 and k1 = N1/2
    ktimer_begin("stolt_rowB_self_kernel", st);
    stolt_rowB_self_kernel<DIR><<<grid_self, 256, smem, st>>>(p);
    ktimer_end(st);
    IMPDAR_LAUNCH_CHECK();
    return IMPDAR_B200_OK;
}

template <int S, int R3, bool PF>
static int launch_col(const ColParams &p, cudaStream_t st) {
    constexpr int NT = S / 32;
    const size_t smem = (size_t)(S + S / 16 + 512) * sizeof(cf) + 16;  // + the mbarrier
    static int ctas_per_sm_dev[IMPDAR_MAX_DEVICES];
    int &ctas_per_sm = ctas_per_sm_dev[current_device_slot()];
    if (!ctas_per_sm) {
        IMPDAR_CUDA(cudaFuncSetAttribute(stolt_col_kernel<S, R3, PF, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int n = 0;
        IMPDAR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, stolt_col_kernel<S, R3, PF, false>, NT, smem));
        ctas_per_sm = n > 0 ? n : 1;
    }
    int grid = num_sms() * ctas_per_sm;
    if (grid > p.ncols) grid = p.ncols;
    ktimer_begin("stolt_col_kernel", st);
    stolt_col_kernel<S, R3, PF, false><<<grid, NT, smem, st>>>(p, nullptr);
    ktimer_end(st);
    IMPDAR_LAUNCH_CHECK();
    return IMPDAR_B200_OK;
}

// IMPDAR_STOLT_COL_PREFETCH=0 selects the variant without the TMA prefetch (development A/B switch).
static bool col_prefetch() {
    const char *e = getenv("IMPDAR_STOLT_COL_PREFETCH");
    return !(e && e[0] == '0');
}

static int dispatch_col(int S, const ColParams &p, cudaStream_t st) {
    if (!col_prefetch()) {
        switch (S) {
            case 1024: return launch_col<1024, 4, false>(p, st);
            case 2048: return launch_col<2048, 8, false>(p, st);
            case 4096: return launch_col<4096, 16, false>(p, st);
            case 8192: return launch_col<8192, 32, false>(p, st);
        }
    }
    switch (S) {
        case 1024: return launch_col<1024, 4, true>(p, st);
        case 2048: return launch_col<2048, 8, true>(p, st);
        case 4096: return launch_col<4096, 16, true>(p, st);
        case 8192: return launch_col<8192, 32, true>(p, st);
    }
    set_error("stolt: unsupported column length %d", S);
    return IMPDAR_B200_EINVAL;
}

template <int S, int R3>
static int launch_col_scan(const ColParams &p, const cf *src, cudaStream_t st) {
    constexpr int NT = S / 32;
    const size_t smem = (size_t)(S + S / 16 + 512) * sizeof(cf) + 16;  // + the mbarrier
    static int ctas_per_sm_dev[IMPDAR_MAX_DEVICES];
    int &ctas_per_sm = ctas_per_sm_dev[current_device_slot()];
    if (!ctas_per_sm) {
        IMPDAR_CUDA(cudaFuncSetAttribute(stolt_col_kernel<S, R3, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int n = 0;
        IMPDAR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, stolt_col_kernel<S, R3, true, true>, NT, smem));
        ctas_per_sm = n > 0 ? n : 1;
    }
    int grid = num_sms() * ctas_per_sm;
    if (grid > p.ncols) grid = p.ncols;
    ktimer_begin("stolt_col_scan_kernel", st);
    stolt_col_kernel<S, R3, true, true><<<grid, NT, smem, st>>>(p, src);
    ktimer_end(st);
    IMPDAR_LAUNCH_CHECK();
    return IMPDAR_B200_OK;
}

static int dispatch_col_scan(int S, const ColParams &p, const cf *src, cudaStream_t st) {
    switch (S) {
        case 1024: return launch_col_scan<1024, 4>(p, src, st);
        case 2048: return launch_col_scan<2048, 8>(p, src, st);
        case 4096: return launch_col_scan<4096, 16>(p, src, st);
        case 8192: return launch_col_scan<8192, 32>(p, src, st);
    }
    set_error("stolt: unsupported column length %d", S);
    return IMPDAR_B200_EINVAL;
}

// Parameters of the five passes for one profile (batch 1), as stolt_fft_run sets them.
static void scan_params(int S, int T, const Tables &tb, RowAParams &pa, RowBParams &pb, ColParams &pc) {
    const int Th = T / 2, N1 = Th / N2;
    pa = RowAParams();
    pa.S = S; pa.T = T; pa.Th = Th; pa.N1 = N1; pa.rows_per_cta = 64; pa.batch = 1; pa.twTh = tb.twTh;
    pb = RowBParams();
    pb.S = S; pb.T = T; pb.Th = Th; pb.N1 = N1; pb.batch = 1; pb.tw512 = tb.tw512;
    pc = ColParams();
    pc.Th = Th; pc.N1 = N1; pc.T = T; pc.ncols = Th; pc.twS = tb.twS; pc.tw2 = tb.tw2;
    pc.norm = (float)(1.0 / ((double)S * (double)T));
}

}  // namespace sfft

bool stolt_fft_supported(int S, int T) {
    const bool s_ok = (S == 1024 || S == 2048 || S == 4096 || S == 8192);
    const bool t_ok = (T == 8192 || T == 16384 || T == 32768 || T == 65536 || T == 131072);
    return s_ok && t_ok;
}

size_t stolt_fft_workspace_bytes(int S, int T) { return (size_t)S * (size_t)T * sizeof(float) + 256; }

// Runs passes P1..P5 on `batch` stacked profiles at once (the workspace holds batch * S * T floats);
// stop_after in 1..5 leaves the intermediate buffers in place for the stage tests.
int stolt_fft_run(const float *data, float *out, int S, int T, int batch, double dt, double dx, double vel, double htaper,
                  double vtaper, int trunc_int, void *workspace, int stop_after, cudaStream_t st) {
    using namespace sfft;
    Tables tb;
    int rc = get_tables(S, T, st, tb);
    if (rc) return rc;
    const int Th = T / 2, N1 = Th / N2;
    cf *W1 = reinterpret_cast<cf *>(out);
    cf *W2 = reinterpret_cast<cf *>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);

    RowAParams pa;
    pa.data = data; pa.W1 = W1; pa.S = S; pa.T = T; pa.Th = Th; pa.N1 = N1;
    pa.rows_per_cta = 64;
    pa.batch = batch;
    pa.htaper = htaper; pa.vtaper = vtaper; pa.trunc_int = trunc_int; pa.twTh = tb.twTh;
    pa.hceil = (htaper == htaper && htaper < 2.0e9) ? (int)ceil(htaper) : 0x7fffffff;
    pa.vceil = (vtaper == vtaper && vtaper < 2.0e9) ? (int)ceil(vtaper) : 0x7fffffff;
    RowBParams pb;
    pb.W1 = W1; pb.Dt = W2; pb.S = S; pb.T = T; pb.Th = Th; pb.N1 = N1; pb.batch = batch; pb.tw512 = tb.tw512;
    ColParams pc;
    pc.Dt = W2; pc.Th = Th; pc.N1 = N1; pc.T = T; pc.ncols = batch * Th; pc.twS = tb.twS; pc.tw2 = tb.tw2;
    pc.beta_unit = vel * (double)S * dt / (2.0 * (double)T * dx);
    pc.norm = (float)(1.0 / ((double)S * (double)T));

    if ((rc = dispatch_rowA<-1>(pa, st))) return rc;
    if (stop_after == 1) return IMPDAR_B200_OK;
    if ((rc = launch_rowB<-1>(pb, st))) return rc;
    if (stop_after == 2) return IMPDAR_B200_OK;
    if ((rc = dispatch_col(S, pc, st))) return rc;
    if (stop_after == 3) return IMPDAR_B200_OK;
    if ((rc = launch_rowB<1>(pb, st))) return rc;
    if (stop_after == 4) return IMPDAR_B200_OK;
    return dispatch_rowA<1>(pa, st);
}

// Velocity scan, forward half: P1 (taper, data -> W1) and P2 (W1 -> W2) once.  W1 and W2 hold snum x tnum floats
// each; W2 keeps the transposed half spectrum that every velocity starts from.
int stolt_fft_scan_forward(const float *data, float *W1, float *W2, int S, int T, double htaper, double vtaper,
                           int trunc_int, cudaStream_t st) {
    using namespace sfft;
    Tables tb;
    int rc = get_tables(S, T, st, tb);
    if (rc) return rc;
    RowAParams pa;
    RowBParams pb;
    ColParams pc;
    scan_params(S, T, tb, pa, pb, pc);
    pa.data = data; pa.W1 = reinterpret_cast<cf *>(W1);
    pa.htaper = htaper; pa.vtaper = vtaper; pa.trunc_int = trunc_int;
    pa.hceil = (htaper == htaper && htaper < 2.0e9) ? (int)ceil(htaper) : 0x7fffffff;
    pa.vceil = (vtaper == vtaper && vtaper < 2.0e9) ? (int)ceil(vtaper) : 0x7fffffff;
    pb.W1 = reinterpret_cast<cf *>(W1); pb.Dt = reinterpret_cast<cf *>(W2);
    if ((rc = dispatch_rowA<-1>(pa, st))) return rc;
    return launch_rowB<-1>(pb, st);
}

// Velocity scan, one velocity: P3 from W2 (left intact) into W3, P4 (W3 -> img) and P5 (in place in img), the same
// kernels and arithmetic as stolt_fft_run's P3..P5, so img is stolt_fft_run's output at this velocity bit for bit.
int stolt_fft_scan_velocity(const float *W2, float *W3, float *img, int S, int T, double dt, double dx, double vel,
                            cudaStream_t st) {
    using namespace sfft;
    Tables tb;
    int rc = get_tables(S, T, st, tb);
    if (rc) return rc;
    RowAParams pa;
    RowBParams pb;
    ColParams pc;
    scan_params(S, T, tb, pa, pb, pc);
    pc.Dt = reinterpret_cast<cf *>(W3);
    pc.beta_unit = vel * (double)S * dt / (2.0 * (double)T * dx);
    pb.W1 = reinterpret_cast<cf *>(img); pb.Dt = reinterpret_cast<cf *>(W3);
    pa.W1 = reinterpret_cast<cf *>(img);
    if ((rc = dispatch_col_scan(S, pc, reinterpret_cast<const cf *>(W2), st))) return rc;
    if ((rc = launch_rowB<1>(pb, st))) return rc;
    return dispatch_rowA<1>(pa, st);
}

}  // namespace impdar
