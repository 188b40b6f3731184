// Focus measure of a migrated image, per window, for the migration velocity scan (impdar_stolt_scan_f32).
//
// Window (i, j) of an S2 x T image covers rows [i ws, min((i+1) ws, S2)) and columns [j wt, min((j+1) wt, T)).  With
// E2 = sum m^2 and E4 = sum m^4 over its n samples (each float32 sample widened to float64),
//   focus = n E4 / E2^2     (the varimax, or normalised fourth moment: 1 for a constant window, n for one spike),
// and 0 where E2 == 0.  A diffraction migrated with the right velocity collapses to its apex, which raises the measure.
//
// Fixed-order two-level reduction, no atomics, so every call gives the same bits:
//   stolt_focus_kernel          one thread per (row chunk, column): the chunk's rows, top down, in float64 -> partials
//   stolt_focus_windows_kernel  one warp per window: its lanes sum the window's partials in a fixed stride order,
//                               then a shuffle butterfly
// Row chunks are at most FOCUS_RC rows and never cross a window row.  The partials of a pass cover as many window rows
// as focus_group_rows() allows, so the scratch stays at 1/8 of the image whatever the window.
#include "common.cuh"

namespace impdar {

constexpr int FOCUS_RC = 128;  // rows per chunk: enough independent loads per thread, few partials

struct FocusParams {
    const float *img;  // (rows, cols)
    int rows, cols, ws, wt, nwt;
    int wr0;           // first window row of this pass
    int cpw;           // chunks per window row
    int nwr;           // window rows in this pass
    double2 *part;     // [(window row - wr0) * cpw + chunk][col] = (E2, E4)
    double *focus;     // (nws, nwt)
};

__global__ void __launch_bounds__(256) stolt_focus_kernel(const __grid_constant__ FocusParams p) {
    const int x = blockIdx.x * 256 + threadIdx.x;
    if (x >= p.cols) return;
    const int wrl = blockIdx.y / p.cpw, q = blockIdx.y - wrl * p.cpw;
    const int wr = p.wr0 + wrl;
    const int wend = min(wr * p.ws + p.ws, p.rows);
    const int r0 = wr * p.ws + q * FOCUS_RC;
    const int r1 = min(r0 + FOCUS_RC, wend);
    const float *src = p.img + (size_t)r0 * p.cols + x;
    double e2 = 0.0, e4 = 0.0;
    int r = r0;
    for (; r + 8 <= r1; r += 8) {
        float m[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) m[k] = __ldcs(src + (size_t)(r - r0 + k) * p.cols);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const double d = (double)m[k];
            const double d2 = d * d;
            e2 += d2;
            e4 = fma(d2, d2, e4);
        }
    }
    for (; r < r1; ++r) {
        const double d = (double)__ldcs(src + (size_t)(r - r0) * p.cols);
        const double d2 = d * d;
        e2 += d2;
        e4 = fma(d2, d2, e4);
    }
    p.part[(size_t)blockIdx.y * p.cols + x] = make_double2(e2, e4);
}

__global__ void __launch_bounds__(256) stolt_focus_windows_kernel(const __grid_constant__ FocusParams p) {
    const int w = (int)((blockIdx.x * 256u + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= p.nwr * p.nwt) return;  // whole warps
    const int wrl = w / p.nwt, j = w - wrl * p.nwt;
    const int wr = p.wr0 + wrl;
    const int c0 = j * p.wt, c1 = min(c0 + p.wt, p.cols);
    const int rows = min(wr * p.ws + p.ws, p.rows) - wr * p.ws;
    const int nch = (rows + FOCUS_RC - 1) / FOCUS_RC;
    double e2 = 0.0, e4 = 0.0;
    for (int q = 0; q < nch; ++q) {
        const double2 *row = p.part + (size_t)(wrl * p.cpw + q) * p.cols;
        for (int x = c0 + lane; x < c1; x += 32) {
            const double2 v = row[x];
            e2 += v.x;
            e4 += v.y;
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        e2 += __shfl_xor_sync(0xffffffffu, e2, o);
        e4 += __shfl_xor_sync(0xffffffffu, e4, o);
    }
    if (lane == 0) {
        const double n = (double)rows * (double)(c1 - c0);
        p.focus[(size_t)wr * p.nwt + j] = (e2 == 0.0) ? 0.0 : n * e4 / (e2 * e2);
    }
}

// Partial rows (chunks) one pass may hold: the scratch is focus_group_rows(rows) * cols double2, 1/8 of the image.
static inline int focus_group_rows(int rows) { return rows / 32 + 1; }

size_t stolt_focus_workspace_bytes(int rows, int cols) {
    return (size_t)focus_group_rows(rows) * (size_t)cols * sizeof(double2);
}

// focus (nws x nwt, device) of the rows x cols float32 image `img`; `part` is stolt_focus_workspace_bytes of scratch.
int stolt_focus_run(const float *img, int rows, int cols, int ws, int wt, double *focus, void *part, cudaStream_t st) {
    if (rows < 1 || cols < 1) return IMPDAR_B200_OK;
    FocusParams p;
    p.img = img; p.rows = rows; p.cols = cols; p.ws = ws; p.wt = wt;
    p.nwt = (cols + wt - 1) / wt;
    p.part = reinterpret_cast<double2 *>(part);
    p.focus = focus;
    const int nws = (rows + ws - 1) / ws;
    const int span = ws < rows ? ws : rows;  // rows of the tallest window
    p.cpw = (span + FOCUS_RC - 1) / FOCUS_RC;
    int group = focus_group_rows(rows) / p.cpw;  // window rows per pass (cpw <= rows / 128 + 1 <= the budget)
    if (group * p.cpw > 65535) group = 65535 / p.cpw;
    if (group < 1) group = 1;
    for (p.wr0 = 0; p.wr0 < nws; p.wr0 += group) {
        p.nwr = nws - p.wr0 < group ? nws - p.wr0 : group;
        dim3 g1((cols + 255) / 256, p.nwr * p.cpw);
        ktimer_begin("stolt_focus_kernel", st);
        stolt_focus_kernel<<<g1, 256, 0, st>>>(p);
        ktimer_end(st);
        IMPDAR_LAUNCH_CHECK();
        const long long warps = (long long)p.nwr * p.nwt;
        ktimer_begin("stolt_focus_windows_kernel", st);
        stolt_focus_windows_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(p);
        ktimer_end(st);
        IMPDAR_LAUNCH_CHECK();
    }
    return IMPDAR_B200_OK;
}

}  // namespace impdar
