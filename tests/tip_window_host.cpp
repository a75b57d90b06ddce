// Host build of the FP32 overlap kernel's cell window + tips (aai_tip_strips_f32, aai_tip_window_ok in aai_cell.cuh),
// for tests/test_tip_window_host.py.  Compiled with g++: the same arithmetic the kernel runs, lane by lane.
#include <math.h>

#include "../area_average_interpolation_b200/csrc/aai_cell.cuh"

namespace {

template <int NW>
void tips(const AaiShapeF &g, float e0, float t0, int (&first)[2], AaiF2 (&area)[3]) {
    aai_tip_strips_f32<NW>(g, e0, t0, first, area);
}

}  // namespace

extern "C" {

int aai_test_tip_window_ok(double c, double s, double L, int nmax) { return aai_tip_window_ok(c, s, L, nmax) ? 1 : 0; }

// For n footprint centres (cx, cy): the kernel's cell box (FP32, as in overlap_body) and, over its first nmax x nmax
// cells, got[k][r][col] = window cells (FP32 Green form, aai_cell_exact_f32) + the tips' strips (aai_tip_strips_f32),
// want[k][r][col] = exact FP64 area (aai_cell_exact_f64), tip[k][0..5] = the six strip areas.  ok[k] = 0 when the box is
// not one the window body evaluates (the kernel redoes such pixels in FP64).
void aai_test_tip_window(double c, double s, double L, int nmax, const double *cx, const double *cy, double *got,
                         double *want, double *tip, int *ok, long long n) {
    const AaiShape g = aai_make_shape(c, s, L);
    const AaiShapeF gf = aai_make_shape_f(c, s, L);
    const float ext32 = (float)(L / 2 * (c + s) + 0.5 + 2e-6);
    const int nw = nmax - 1;
    for (long long k = 0; k < n; ++k) {
        double *gk = got + k * nmax * nmax, *wk = want + k * nmax * nmax;
        for (int q = 0; q < nmax * nmax; ++q) gk[q] = wk[q] = 0.0;
        const int irx = (int)rint(cx[k]), iry = (int)rint(cy[k]);
        const float fx = (float)(cx[k] - irx), fy = (float)(cy[k] - iry);
        const int bx0 = irx + (int)ceilf(fx - ext32), bx1 = irx + (int)floorf(fx + ext32);
        const int by0 = iry + (int)ceilf(fy - ext32), by1 = iry + (int)floorf(fy + ext32);
        const int ncols = bx1 - bx0 + 1, nrows = by1 - by0 + 1;
        ok[k] = ncols >= nw && ncols <= nmax && nrows >= nw && nrows <= nmax;
        if (!ok[k]) continue;
        // exact FP64 areas of the nmax x nmax cells from (bx0, by0)
        for (int r = 0; r < nmax; ++r)
            for (int col = 0; col < nmax; ++col) {
                const double rx = (bx0 + col) - cx[k], ry = (by0 + r) - cy[k];
                double xlT, xrT, xlB, xrB, ytL, ybL, ytR, ybR;
                aai_chord_h(g, ry - 0.5, xlT, xrT);
                aai_chord_h(g, ry + 0.5, xlB, xrB);
                aai_chord_v(g, rx - 0.5, ytL, ybL);
                aai_chord_v(g, rx + 0.5, ytR, ybR);
                wk[r * nmax + col] = aai_cell_exact_f64(g, rx, ry, aai_overlap1(xlT, xrT, rx), aai_overlap1(xlB, xrB, rx),
                                                        aai_overlap1(ytL, ybL, ry), aai_overlap1(ytR, ybR, ry));
            }
        // window cells in FP32, footprint-local coordinates as in the kernel
        const float rx0 = (float)(bx0 - irx) - fx, t0 = ((float)(by0 - iry) - fy) - 0.5f, e0 = rx0 - 0.5f;
        for (int r = 0; r < nw; ++r)
            for (int col = 0; col < nw; ++col) {
                const float rx = rx0 + (float)col, ry = (float)(by0 - iry + r) - fy;
                float xlT, xrT, xlB, xrB, ytL, ybL, ytR, ybR;
                aai_chord_h_f32(gf, ry - 0.5f, xlT, xrT);
                aai_chord_h_f32(gf, ry + 0.5f, xlB, xrB);
                aai_chord_v_f32(gf, rx - 0.5f, ytL, ybL);
                aai_chord_v_f32(gf, rx + 0.5f, ytR, ybR);
                const float ex = rx - 0.5f, ey = ry - 0.5f;
                gk[r * nmax + col] = aai_cell_exact_f32(gf, fmaf(rx, gf.cs, -ry * gf.sn), fmaf(rx, gf.sn, ry * gf.cs),
                                                        aai_overlap1_f32(xlT, xrT, ex), aai_overlap1_f32(xlB, xrB, ex),
                                                        aai_overlap1_f32(ytL, ybL, ey), aai_overlap1_f32(ytR, ybR, ey));
            }
        int first[2];
        AaiF2 a[3];
        switch (nw) {
            case 3: tips<3>(gf, e0, t0, first, a); break;
            case 4: tips<4>(gf, e0, t0, first, a); break;
            case 5: tips<5>(gf, e0, t0, first, a); break;
            default: tips<7>(gf, e0, t0, first, a); break;
        }
        for (int j = 0; j < 3; ++j) {  // right tip in column nw, bottom tip in row nw (strips beyond the grid: dropped)
            const int r = first[0] + j, col = first[1] + j;
            if (r < nmax) gk[r * nmax + nw] += a[j].x;
            if (col < nmax) gk[nw * nmax + col] += a[j].y;
            tip[k * 6 + j] = a[j].x;
            tip[k * 6 + 3 + j] = a[j].y;
        }
    }
}

}  // extern "C"
