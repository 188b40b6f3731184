// Uniform-geometry Kirchhoff, shared-memory staged form (north-star (a): output traces tiled per CTA, input trace
// windows staged through shared memory by TMA).  Included by kirchhoff.cu after KirchTabParams.
//
// The table form of the sum (kirchhoff.cu) is out[ti, x] = sum_m w[ti, m] (g[k(ti, m), x - m] + g[k(ti, m), x + m]):
// one 4-byte gather per pair.  Gathered from global memory every pair costs an L1 request (misaligned: ~1.3 data-pipe
// wavefronts) and 40 % of them miss to L2 (ncu, profiles/r01g_ncu_full_kirch_table.txt).  Here a CTA owns KT_Q
// consecutive output rows x KT_X output traces.  Rows of one block walk nearly the same hyperbola, so for a source
// row k the offsets m used by ANY row of the block form a short interval [mlo, mhi] (a device-built schedule, exact,
// from the table itself): the two row segments g[k, x0 - mhi .. x0 + X - mlo) and g[k, x0 + mlo .. x0 + X + mhi) are
// bulk-copied (cp.async.bulk, mbarrier complete_tx) ONCE into a ring of shared-memory stages by a producer warp and
// serve every (row, m) of the block that picks row k: each pair is one conflict-free shared-memory read (any
// alignment is one wavefront), L2 traffic drops from ~2 B to ~0.7 B per pair.
//
// Summation order per output sample: m ascending, partial sums flushed into a second accumulator after every
// KT_FLUSH-th stage; stages are windows of KT_W source rows at ABSOLUTE multiples of KT_W (and the flushes at absolute
// window indices), so the order - and therefore the result, bit for bit - does not depend on how the image is cut
// into row chunks, trace ranges or CTAs.  Nor do the decisions about which rows this kernel does: blocks sit at absolute
// multiples of KT_Q rows (a row chunk runs the clipped part of the image's blocks), the stand-down for intervals wider
// than KT_SPAN is taken once per image over all its blocks, and rows that read non-finite input (ti < flags[0], the
// deepest non-finite row + 1) are left to the gather kernel's nansum variant row by row.
#pragma once

namespace impdar {

// tunables (A/B builds: python -m impdar_b200._build -DKT_CFG_NW=16 -DKT_CFG_RW=2 --out=...)
#ifndef KT_CFG_NW
#define KT_CFG_NW 28
#endif
#ifndef KT_CFG_NP
#define KT_CFG_NP 4
#endif
#ifndef KT_CFG_RW
#define KT_CFG_RW 1
#endif
#ifndef KT_CFG_TR
#define KT_CFG_TR 8
#endif
#ifndef KT_CFG_W
#define KT_CFG_W 16
#endif
#ifndef KT_CFG_NST
#define KT_CFG_NST 4
#endif
constexpr int KT_NW = KT_CFG_NW;     // consumer warps per CTA
constexpr int KT_NP = KT_CFG_NP;     // producer warps per CTA (KT_NW + KT_NP <= 32).  cp.async.bulk is a warp-uniform
                                     // instruction: the rows of a stage are issued one after the other (~9 issue slots
                                     // and a few R2UR round trips each), so ONE producer warp feeding 32 copies per stage
                                     // was the kernel's bottleneck (ncu r02c: consumers spun 56 times per stage wait)
constexpr int KT_RW = KT_CFG_RW;     // output rows per consumer warp
constexpr int KT_Q = KT_NW * KT_RW;  // output rows per CTA
constexpr int KT_TR = KT_CFG_TR;     // output traces per lane (stride 32), even
constexpr int KT_X = 32 * KT_TR;     // output traces per CTA
constexpr int KT_W = KT_CFG_W;       // source rows per stage (<= 32: one producer lane per row)
constexpr int KT_NST = KT_CFG_NST;   // stages in the ring
#ifndef KT_CFG_FLUSH
#define KT_CFG_FLUSH 4
#endif
constexpr int KT_FLUSH = KT_CFG_FLUSH;           // stages (absolute index) between second-level accumulator flushes; power of two
constexpr int KT_SPAN = 120;         // widest [mlo, mhi] interval the staged segments hold
constexpr int KT_SEGW = KT_X + KT_SPAN + 8;                   // floats per staged segment (alignment shift <= 3)
constexpr int KT_STAGE_FLOATS = KT_W * 2 * KT_SEGW;
constexpr int KT_RING = 33;           // decoded entries per (warp, row) ring: one chunk of 32, plus the slot that the
                                      // walk's one-ahead read touches after the chunk's last entry
constexpr size_t KT_SMEM = (size_t)KT_NST * KT_STAGE_FLOATS * sizeof(float) +
                           (size_t)KT_NW * KT_RW * KT_RING * sizeof(int4) + 2 * KT_NST * sizeof(unsigned long long) + 16;
constexpr int KT_THREADS = (KT_NW + KT_NP) * 32;
constexpr int KT_RPP = (KT_W + KT_NP - 1) / KT_NP;   // stage rows per producer warp
static_assert(KT_RPP <= 32 && KT_NW + KT_NP <= 32, "tile kernel configuration");

struct KirchTileParams {
    const int2 *seg;     // [nblocks][S]: {mlo, mhi} per source row (mlo > mhi: not used by the block)
    const int *nstage;   // [nblocks]: stages the block walks (from its first row's absolute window)
    int *sched_flags;    // [0] != 0: some interval of the image is wider than KT_SPAN -> this kernel stands down (table kernel runs)
    int t_base;          // first row of block 0: the multiple of KT_Q at or below the launch's first row
};

// Where source row k sits in the staging buffer: stage ring slot `slot`, row j of the stage, for the block's offset
// interval e = {mlo, mhi} = seg[b][k].  The left segment g[k, x0 - mhi ..] and the right segment g[k, x0 + mlo ..] are
// each copied from the 16-byte boundary at or below their first element (cp.async.bulk alignment), so output trace
// x0 + i reads offset m at buf[ol + i - m] (left) and buf[orr + i + m] (right).  The producers copy by it and the
// consumers decode table entries by it: this is the one definition of the layout.
struct KtPlace {
    long long gl, gr;   // first element of the left / right copy in gP (multiples of 4)
    unsigned nl, nr;    // floats per copy (multiples of 4)
    int dl, dr;         // first float of the left / right copy in buf
    int ol, orr;        // buf index of output trace x0's element at m = 0, left / right
};
__device__ __forceinline__ KtPlace kt_place(const KirchTabParams &p, int x0, int k, int slot, int j, int2 e) {
    const int span = e.y - e.x;
    const long long rowoff = (long long)k * p.Tp + p.Apad + x0;
    const long long il = rowoff - e.y, ir = rowoff + e.x;          // first element of the left / right segment
    const int shl = (int)(il & 3), shr = (int)(ir & 3);
    KtPlace r;
    r.gl = il - shl;
    r.gr = ir - shr;
    r.nl = (unsigned)((shl + KT_X + span + 3) & ~3);
    r.nr = (unsigned)((shr + KT_X + span + 3) & ~3);
    r.dl = slot * KT_STAGE_FLOATS + j * 2 * KT_SEGW;
    r.dr = r.dl + KT_SEGW;
    r.ol = r.dl + shl + e.y;
    r.orr = r.dr + shr - e.x;
    return r;
}

__device__ __forceinline__ unsigned kt_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void kt_mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(kt_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void kt_mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(kt_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void kt_mbar_arrive_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(kt_smem_u32(bar)), "r"(bytes) : "memory");
}
#ifndef KT_CFG_SLEEP
#define KT_CFG_SLEEP 0
#endif
__device__ __forceinline__ bool kt_mbar_try(unsigned long long *bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(kt_smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void kt_mbar_wait(unsigned long long *bar, unsigned parity) {
    while (!kt_mbar_try(bar, parity)) {
        if (KT_CFG_SLEEP) __nanosleep(KT_CFG_SLEEP);   // a waiting warp leaves the issue slots to the working ones
    }
}
__device__ __forceinline__ void kt_bulk_load(void *smem_dst, const void *gsrc, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     kt_smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(kt_smem_u32(bar))
                 : "memory");
}

// Schedule: for every block of KT_Q output rows of [s_begin, s_end) and every source row k, the interval of offsets m with
// k(ti, m) == k for some row ti of the block.  One CTA per block; the table rows are walked once (S x A1 entries in all).
__global__ void __launch_bounds__(256) kirch_tile_sched_kernel(const int2 *__restrict__ tab, const int *__restrict__ nm,
                                                               int S, int A1, int s_begin, int s_end, int2 *__restrict__ seg,
                                                               int *__restrict__ nstage, int *__restrict__ sched_flags) {
    __shared__ int s_kmax, s_wide;
    const int b = blockIdx.x;
    const int t0 = s_begin + b * KT_Q, t1 = min(t0 + KT_Q, s_end);
    int2 *__restrict__ sb = seg + (size_t)b * S;
    if (threadIdx.x == 0) { s_kmax = -1; s_wide = 0; }
    for (int k = t0 + threadIdx.x; k < S; k += blockDim.x) sb[k] = make_int2(0x7fffffff, -1);
    __syncthreads();
    int kmax = -1;
    for (int ti = t0; ti < t1; ++ti) {
        const int n = nm[ti];
        const int2 *__restrict__ row = tab + (size_t)ti * A1;
        for (int m = threadIdx.x; m < n; m += blockDim.x) {
            const int k = row[m].x;
            if (k >= 0) {
                atomicMin(&sb[k].x, m);
                atomicMax(&sb[k].y, m);
                kmax = max(kmax, k);
            }
        }
    }
    if (kmax >= 0) atomicMax(&s_kmax, kmax);
    __syncthreads();
    int wide = 0;
    for (int k = t0 + threadIdx.x; k < S; k += blockDim.x) {
        const int2 e = sb[k];
        if (e.y >= e.x && e.y - e.x > KT_SPAN) wide = 1;
    }
    if (wide) atomicOr(&s_wide, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        const int kbase = (t0 / KT_W) * KT_W;
        nstage[b] = s_kmax < 0 ? 0 : (s_kmax - kbase) / KT_W + 1;
        if (s_wide) atomicOr(sched_flags, 1);
    }
}

// (output sample, input trace) pairs of the table rows [s_begin, s_end) for output traces [x_begin, x_end): what the
// STATS variant of the table kernel counts pair by pair, in closed form per table entry.
__global__ void __launch_bounds__(256) kirch_table_count_kernel(const int2 *__restrict__ tab, const int *__restrict__ nm,
                                                                int A1, int T, int x_begin, int x_end, int s_begin,
                                                                unsigned long long *__restrict__ stats) {
    const int ti = s_begin + blockIdx.x;
    const int n = nm[ti];
    const int2 *__restrict__ row = tab + (size_t)ti * A1;
    unsigned long long c = 0;
    for (int m = threadIdx.x; m < n; m += blockDim.x) {
        if (row[m].x < 0) continue;
        c += (unsigned long long)max(0, x_end - max(x_begin, m));                       // x - m >= 0
        if (m) c += (unsigned long long)max(0, min(x_end, T - m) - x_begin);            // x + m < T
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&stats[0], c);
}

__global__ void __launch_bounds__(KT_THREADS, 1) kirch_tile_kernel(const __grid_constant__ KirchTabParams p,
                                                                   const __grid_constant__ KirchTileParams q) {
    extern __shared__ __align__(128) unsigned char kt_smem_raw[];
    if (q.sched_flags[0] != 0) return;              // wide intervals somewhere in the image: the table kernel runs
    const int b = blockIdx.x;                       // row block (fast index: concurrent CTAs share the column window in L2)
    // the image's block at an absolute multiple of KT_Q rows, clipped to this launch's rows [s_begin, s_end)
    const int t0 = q.t_base + b * KT_Q;
    const int r_lo = max(t0, p.flags[0]);           // rows ti < flags[0] read non-finite input: the table kernel does them
    if (min(t0 + KT_Q, p.s_end) <= r_lo) return;
    float *buf = reinterpret_cast<float *>(kt_smem_raw);
    int4 *rings = reinterpret_cast<int4 *>(buf + (size_t)KT_NST * KT_STAGE_FLOATS);
    unsigned long long *full = reinterpret_cast<unsigned long long *>(rings + KT_NW * KT_RW * KT_RING);
    unsigned long long *empty = full + KT_NST;

    const int x0 = p.x_begin + blockIdx.y * KT_X;
    const int nst = q.nstage[b];
    const int kbase = (t0 / KT_W) * KT_W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int2 *__restrict__ sb = q.seg + (size_t)b * p.S;

    if (threadIdx.x == 0) {
        for (int i = 0; i < KT_NST; ++i) {
            kt_mbar_init(&full[i], KT_NP);
            kt_mbar_init(&empty[i], KT_NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= KT_NW) {
        // ------------------------------------------------- producers: warp pw issues rows [pw KT_RPP, (pw + 1) KT_RPP) of a stage
        const int pw = warp - KT_NW;
        for (int s = 0; s < nst; ++s) {
            const int slot = s % KT_NST;
            if (s >= KT_NST) kt_mbar_wait(&empty[slot], (unsigned)((s / KT_NST - 1) & 1));
            unsigned bytes = 0, nl = 0, nr = 0;
            const float *gl = nullptr, *gr = nullptr;
            float *dl = nullptr, *dr = nullptr;
            const int j = pw * KT_RPP + lane;                // row of the stage
            if (lane < KT_RPP && j < KT_W) {
                const int k = kbase + s * KT_W + j;
                int2 e = make_int2(1, 0);
                if (k >= t0 && k < p.S) e = sb[k];
                if (e.y >= e.x) {
                    const KtPlace pl = kt_place(p, x0, k, slot, j, e);
                    nl = pl.nl;
                    nr = pl.nr;
                    gl = p.gP + pl.gl;
                    gr = p.gP + pl.gr;
                    dl = buf + pl.dl;
                    dr = buf + pl.dr;
                    bytes = (nl + nr) * 4u;
                }
            }
            const unsigned total = __reduce_add_sync(0xffffffffu, bytes);
            __syncwarp();
            if (lane == 0) kt_mbar_arrive_tx(&full[slot], total);
            __syncwarp();
            if (bytes) {
                kt_bulk_load(dl, gl, nl * 4u, &full[slot]);
                kt_bulk_load(dr, gr, nr * 4u, &full[slot]);
            }
        }
        return;
    }

    // -------------------------------------------------------------------- consumers: warp = KT_RW output rows x KT_X traces
    // accumulators as fp32x2 pairs: the adds and FMAs issue on the packed pipe (half the instructions, same roundings)
    float2 acc[KT_RW][KT_TR / 2], tot[KT_RW][KT_TR / 2];
    // The table row of an output sample is walked once, front to back, a chunk of 32 entries at a time.  The raw entries
    // {k, w} come with one coalesced load per lane a chunk ahead of their use (the L1 left beside 200 KB of staging
    // buffers does not hold 31 table rows).  Each lane then decodes one entry of the chunk into what the walk needs:
    // the shared-memory offsets of its source row's two segments, already shifted by -m and +m, and the weight.  Skips
    // (k < 0) are compacted away; the rest go into a warp-private ring, one 16-byte broadcast read per entry, issued an
    // entry ahead of its use.  Each lane keeps the stage of the entry it decoded (csk), so one ballot per stage gives
    // the stage's trip count: the walk itself compares nothing but its index.
    int mnext[KT_RW], mend[KT_RW];     // first table entry of the next chunk; entries in the row
    int pos[KT_RW], cnt[KT_RW];        // next ring entry to walk; entries in the ring
    int csk[KT_RW];                    // per lane: stage of the lane's decoded entry (INT_MAX: none)
    bool live[KT_RW];                  // the row is this launch's and this kernel's to write
    const int2 *trow[KT_RW];
    int2 pre[KT_RW];
    int4 *ring[KT_RW];
    int4 cur[KT_RW];                   // ring[pos], read ahead
    const int2 none = make_int2(-1, 0);
    // Chunk mnext of row w into the ring (which the walk has emptied); the next chunk's load goes out.
    auto decode = [&](int w) {
        const int m = mnext[w] + lane;
        const int2 e = pre[w];
        pre[w] = m + 32 < mend[w] ? __ldg(trow[w] + m + 32) : none;
        const unsigned v = __ballot_sync(0xffffffffu, e.x >= 0);
        __syncwarp();                  // every lane has read the previous chunk's entries
        csk[w] = 0x7fffffff;
        if (e.x >= 0) {
            const unsigned rel = (unsigned)(e.x - kbase), sk = rel / KT_W;
            const KtPlace pl = kt_place(p, x0, e.x, (int)(sk % KT_NST), (int)(rel % KT_W), __ldg(sb + e.x));
            // m == 0: left and right segment hold the same element, w/2 (g + g) == w g exactly
            const float wgt = __int_as_float(e.y) * (m == 0 ? 0.5f : 1.0f);
            ring[w][__popc(v & ((1u << lane) - 1u))] =
                make_int4((pl.ol - m) * 4, (pl.orr + m) * 4, __float_as_int(wgt), 0);   // byte offsets
            csk[w] = (int)sk;
        }
        __syncwarp();
        mnext[w] += 32;
        pos[w] = 0;
        cnt[w] = __popc(v);
        cur[w] = ring[w][0];
    };
#pragma unroll
    for (int w = 0; w < KT_RW; ++w) {
        const int ti = t0 + warp + w * KT_NW;
        live[w] = ti >= max(p.s_begin, r_lo) && ti < p.s_end && (x0 < p.x_end);
        mnext[w] = 0;
        mend[w] = live[w] ? p.nm[ti] : 0;
        trow[w] = p.tab + (size_t)(live[w] ? ti : t0) * p.A1;
        ring[w] = rings + (size_t)(warp * KT_RW + w) * KT_RING;
        pre[w] = lane < mend[w] ? __ldg(trow[w] + lane) : none;
        decode(w);
#pragma unroll
        for (int r = 0; r < KT_TR / 2; ++r) acc[w][r] = tot[w][r] = make_float2(0.f, 0.f);
    }
    const char *__restrict__ lbuf = reinterpret_cast<const char *>(buf + lane);
    const int sabs0 = kbase / KT_W;                 // absolute index of this block's first stage window
    for (int s = 0; s < nst; ++s) {
        const int slot = s % KT_NST;
        kt_mbar_wait(&full[slot], (unsigned)((s / KT_NST) & 1));
#pragma unroll
        for (int w = 0; w < KT_RW; ++w) {
            while (true) {
                const int end = __popc(__ballot_sync(0xffffffffu, csk[w] <= s));   // the ring's entries of stages <= s
                int4 d = cur[w];
#pragma unroll 1   // short trips (at rho 0.169, 62 % of warp-stages walk 2-3 entries): unrolled copies measured slower
                for (int i = pos[w]; i < end; ++i) {
                    const int4 nx = ring[w][i + 1];
                    const float *__restrict__ pl = reinterpret_cast<const float *>(lbuf + d.x);
                    const float *__restrict__ pr = reinterpret_cast<const float *>(lbuf + d.y);
                    const float wgt = __int_as_float(d.z);
                    const float2 w2 = make_float2(wgt, wgt);
#pragma unroll
                    for (int r = 0; r < KT_TR / 2; ++r) {
                        const float2 l = make_float2(pl[64 * r], pl[64 * r + 32]);
                        const float2 g = make_float2(pr[64 * r], pr[64 * r + 32]);
                        acc[w][r] = __ffma2_rn(w2, __fadd2_rn(l, g), acc[w][r]);
                    }
                    d = nx;
                }
                cur[w] = d;
                pos[w] = end;
                if (end < cnt[w] || mnext[w] >= mend[w]) break;   // the stage ends inside this chunk, or the row does
                decode(w);
            }
        }
        if (((sabs0 + s) & (KT_FLUSH - 1)) == KT_FLUSH - 1) {     // second-level accumulation at absolute window indices
#pragma unroll
            for (int w = 0; w < KT_RW; ++w)
#pragma unroll
                for (int r = 0; r < KT_TR / 2; ++r) {
                    tot[w][r] = __fadd2_rn(tot[w][r], acc[w][r]);
                    acc[w][r] = make_float2(0.f, 0.f);
                }
        }
        __syncwarp();
        if (lane == 0) kt_mbar_arrive(&empty[slot]);
    }
#pragma unroll
    for (int w = 0; w < KT_RW; ++w) {
        const int ti = t0 + warp + w * KT_NW;
        if (!live[w]) continue;
#pragma unroll
        for (int r = 0; r < KT_TR / 2; ++r) {
            const float2 v = __fadd2_rn(tot[w][r], acc[w][r]);
            const int x = x0 + lane + 64 * r;
            if (x < p.x_end) p.out[(size_t)ti * p.ldo + (x - p.x_begin)] = v.x;
            if (x + 32 < p.x_end) p.out[(size_t)ti * p.ldo + (x + 32 - p.x_begin)] = v.y;
        }
    }
}

}  // namespace impdar
