// Per-(footprint, unit cell) overlap arithmetic shared by every overlap kernel.
//
// Host+device inline functions, so that the CPU test-suite can exercise exactly the arithmetic the kernels
// run (tests/cell_math_host.cpp compiles this header with g++ for unit tests only; the product path never
// evaluates it on the host).
//
// Geometry (SURVEY.md Appendix A): the footprint of a canvas pixel is the square |u| <= h, |v| <= h with
//   u = (p - C).(c, -s),  v = (p - C).(s, c),  h = L/2,  theta in (0, 90 deg), y pointing down;
// its "left/right" edges u = +-h have direction (s, c) (the reference's "vertical lines", Source.cpp:457-468),
// its "top/bottom" edges v = +-h have direction (c, -s).  A cell is the unit square centred at integer (i, j).
#ifndef AAI_CELL_CUH_
#define AAI_CELL_CUH_

#include <math.h>

#if defined(__CUDACC__)
#define AAI_HD __host__ __device__ __forceinline__
#else
#define AAI_HD inline
#endif

// image-wide constants of the footprint shape (all FP64, computed once on the host)
struct AaiShape {
    double cs, sn;     // cos, sin of the reduced angle
    double half;       // h
    double hc, hs;     // h*c, h*s
    double k_sc, k_hc; // s/c, h/c
    double k_cs, k_hs; // c/s, h/s
    double inv_c, inv_s;
    double m;          // (c+s)/2: half extent of a unit cell along u or v
    double thr;        // |c-s|/2: a line isolates exactly one cell corner iff thr < |dist| < m
    // per-edge quirk events (aai_edge_quirk_f64; same meaning as the AaiShapeF fields of the same names)
    double hb, he, ik, hq, smin, smax, hm, area_total;
    int steep, ncross;
};

// image-wide FP64 constants (host side; shared by the C ABI and the CPU tests)
inline AaiShape aai_make_shape(double c, double s, double L) {
    AaiShape g;
    const double h = L / 2;
    g.cs = c;
    g.sn = s;
    g.half = h;
    g.hc = h * c;
    g.hs = h * s;
    g.k_sc = s / c;
    g.k_hc = h / c;
    g.k_cs = c / s;  // +inf when the reduced angle is exactly 0: the separable path never reads it
    g.k_hs = h / s;
    g.inv_c = 1.0 / c;
    g.inv_s = 1.0 / s;
    g.m = (c + s) / 2;
    g.thr = fabs(c - s) / 2;
    const double mn = s < c ? s : c, mx = s < c ? c : s;
    g.hb = h * (c + s);
    g.he = h * fabs(c - s);
    g.ik = mx / mn;
    g.hq = (1.0 + mn / mx) / 2;
    g.smin = mn;
    g.smax = mx;
    g.hm = h - (c + s) / 2;
    g.area_total = L * L;
    g.steep = s <= c ? 1 : 0;
    const double nc = floor(L * mn) + 1;
    g.ncross = nc < 1e6 ? (int)nc : 1000000;
    return g;
}

// chord of the footprint on the horizontal grid line y = Cy + ty:  x in Cx + [xl, xr]  (empty if xl > xr)
AAI_HD void aai_chord_h(const AaiShape &g, double ty, double &xl, double &xr) {
    const double p = ty * g.k_sc, q = ty * g.k_cs;
    xl = fmax(p - g.k_hc, -q - g.k_hs);
    xr = fmin(p + g.k_hc, g.k_hs - q);
}
// chord of the footprint on the vertical grid line x = Cx + tx:  y in Cy + [yt, yb]
AAI_HD void aai_chord_v(const AaiShape &g, double tx, double &yt, double &yb) {
    const double p = tx * g.k_cs, q = tx * g.k_sc;
    yt = fmax(p - g.k_hs, -q - g.k_hc);
    yb = fmin(p + g.k_hs, g.k_hc - q);
}
// length of [lo, hi] ∩ [r - 1/2, r + 1/2]
AAI_HD double aai_overlap1(double lo, double hi, double r) {
    return fmax(fmin(hi, r + 0.5) - fmax(lo, r - 0.5), 0.0);
}

// Overlap area of the footprint with the unit cell whose centre is (rx, ry) relative to the footprint centre,
// given the lengths of the four cell sides inside the footprint.  Reference-compatible (includes the shape 2/4
// leg quirk of Source.cpp:1055-1062).
AAI_HD double aai_cell_area(const AaiShape &g, double rx, double ry, double lenT, double lenB, double lenL,
                            double lenR, bool quirk = true) {
    // footprint-local coordinates of the cell centre; nearest footprint vertex V in cell-local coordinates
    const double u0 = rx * g.cs - ry * g.sn;
    const double v0 = rx * g.sn + ry * g.cs;
    const double vx = (copysign(g.hc, u0) + copysign(g.hs, v0)) - rx;
    const double vy = (copysign(g.hc, v0) - copysign(g.hs, u0)) - ry;
    // Green's theorem about V: A = 1/2 sum_sides dist(V, side) * len(side ∩ footprint)
    double area = 0.25 * ((lenT + lenB) + (lenL + lenR)) + 0.5 * (vy * (lenT - lenB) + vx * (lenL - lenR));
    // Reference quirk.  a = signed distance of the cell centre inside the nearest left/right edge.
    const double a = g.half - fabs(u0);
    const double aa = fabs(a);
    if (quirk && aa > g.thr && aa < g.m) {  // that edge's line isolates exactly one cell corner
        const double sv = copysign(1.0, v0), su = copysign(1.0, u0);
        // the left/right edge is the ray from W = sv*V along -(s,c); the cell is [-1/2,1/2]^2 (slab test)
        const double wx = sv * vx, wy = sv * vy;
        const double u_in = fmax((wx - 0.5) * g.inv_s, (wy - 0.5) * g.inv_c);
        const double u_out = fmin((wx + 0.5) * g.inv_s, (wy + 0.5) * g.inv_c);
        // the top/bottom edge is the ray from Z = su*V along (-c, s)
        const double zx = su * vx, zy = su * vy;
        const double v_in = fmax((zx - 0.5) * g.inv_c, (-0.5 - zy) * g.inv_s);
        const double v_out = fmin((zx + 0.5) * g.inv_c, (0.5 - zy) * g.inv_s);
        const bool u_through = u_in > 0.0 && u_in < u_out;  // crosses two cell sides inside the edge segment
        const bool v_hits = v_in < v_out && v_out > 0.0;    // top/bottom edge segment meets the cell
        if (u_through && !v_hits) {
            if (a < 0.0) {  // one corner inside, at distance d from the edge: reference shape 2
                const double d = a + g.m;
                area = 0.5 * (1.0 - d * g.inv_c) * (1.0 - d * g.inv_s);
            } else {  // one corner outside (d < 0): reference shape 4
                const double d = a - g.m;
                area = 1.0 - 0.5 * (1.0 + d * g.inv_c) * (1.0 + d * g.inv_s);
            }
        }
    }
    return area;
}

// Exact overlap only (no quirk), Green form with the vertex rotation folded into the side coefficients (the form the
// FP32 kernel uses, in FP64): what the unrolled FP64 kernel evaluates per cell.
AAI_HD double aai_cell_exact_f64(const AaiShape &g, double rx, double ry, double lenT, double lenB, double lenL,
                                 double lenR) {
    const double u0 = rx * g.cs - ry * g.sn;
    const double v0 = rx * g.sn + ry * g.cs;
    const double ca = copysign(g.half, u0) - u0;  // V - cell centre along u, v
    const double cb = copysign(g.half, v0) - v0;
    const double aT = 0.25 + 0.5 * (cb * g.cs - ca * g.sn);
    const double aL = 0.25 + 0.5 * (ca * g.cs + cb * g.sn);
    return aT * (lenT - lenB) + (aL * (lenL - lenR) + 0.5 * (lenB + lenR));
}
// value of x clamped into the chord [lo, hi] (hi < lo, a grid line that misses the footprint, gives hi for every x):
// the length of [lo,hi] inside [a,b] is clamp(b) - clamp(a), bit-identical to aai_overlap1 and one min/max cheaper when
// consecutive cells share a boundary
AAI_HD double aai_clamp_chord(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }

// Stand-alone form for one (footprint centre, cell) pair: computes the four chords itself.
AAI_HD double aai_pair_area(const AaiShape &g, double cx, double cy, int i, int j, bool quirk = true) {
    const double rx = (double)i - cx, ry = (double)j - cy;
    double xlT, xrT, xlB, xrB, ytL, ybL, ytR, ybR;
    aai_chord_h(g, ry - 0.5, xlT, xrT);
    aai_chord_h(g, ry + 0.5, xlB, xrB);
    aai_chord_v(g, rx - 0.5, ytL, ybL);
    aai_chord_v(g, rx + 0.5, ytR, ybR);
    return aai_cell_area(g, rx, ry, aai_overlap1(xlT, xrT, rx), aai_overlap1(xlB, xrB, rx),
                         aai_overlap1(ytL, ybL, ry), aai_overlap1(ytR, ybR, ry), quirk);
}

// ------------------------------------------------------------------------------------------------------------
// FP32 variant ("FP32 kernel" of the north star): coordinates are taken relative to the footprint centre in FP64
// and rounded once; lengths, areas and sums are FP32; the shape decision of the quirk is made in FP32 with a
// guard band: when any decisive margin is within `tau` of zero the caller must redo the pixel in FP64
// (`uncertain` is set), so that no FP32 rounding can flip a discontinuous decision (SURVEY.md §0.3).
// ------------------------------------------------------------------------------------------------------------
struct AaiShapeF {
    float cs, sn, half;
    float k_sc, k_hc, k_cs, k_hs;
    float inv_c, inv_s;
    float m, thr;
    float tau;  // guard band of the FP32 decisions (distance / edge-parameter units)
    // constants of the per-row cross-check formulation (tests/cell_legacy_forms.h)
    float hk;    // (1 + c/s)/2
    float hm;    // h - m: |v0| <= hm  <=>  the whole cell lies inside the top/bottom slab
    float y_lf;  // h(s-c): y of the footprint's left vertex = top end of the left edge   (relative to the centre)
    float y_bt;  // h(s+c): y of the bottom vertex = bottom end of the left edge
    // per-edge quirk events (aai_edge_quirk_f32): "major" axis = the grid axis the left/right edges mostly run along
    // (y when sin <= cos, else x), "minor" axis = the other one
    float hb;    // h(c+s): half extent of the footprint's bounding box
    float he;    // h|c-s|
    float ik;    // max(s,c)/min(s,c): advance along the major axis per unit of the minor axis
    float hq;    // (1 + min/max)/2
    float smin, smax;  // min(s,c), max(s,c)
    float hc2, hs2;    // c/2, s/2 (side coefficients of the Green form)
    float area_total;  // L^2: total overlap of a footprint that lies inside the image (exact areas)
    // quadrant weights of the upscaling path (aai_quadrant_areas_f32): edge parameters normalised to [0, 1]
    float kq_s, kq_c;  // 1/(s L), 1/(c L)
    float qq_cs, qq_sc;  // c/(2 s), s/(2 c)
    float half_side;   // L/2
    // tips of the footprint outside its cell window (aai_tip_strips_f32)
    float tk_sc, tk_cs;  // s/(2c), c/(2s)
    int steep;   // 1: sin <= cos (major axis = y, the edges cross vertical grid lines rarely)
    int ncross;  // floor(L min(s,c)) + 1: most minor-axis grid lines one left/right edge can cross
};

// image-wide FP32 constants from the FP64 plan values (host side; shared by the C ABI and the CPU tests)
inline AaiShapeF aai_make_shape_f(double c, double s, double L) {
    AaiShapeF g;
    const double h = L / 2;
    g.cs = (float)c;
    g.sn = (float)s;
    g.half = (float)h;
    g.k_sc = (float)(s / c);
    g.k_hc = (float)(h / c);
    g.k_cs = (float)(c / s);
    g.k_hs = (float)(h / s);
    g.inv_c = (float)(1.0 / c);
    g.inv_s = (float)(1.0 / s);
    g.m = (float)((c + s) / 2);
    g.thr = (float)(fabs(c - s) / 2);
    // guard band of the FP32 decisions: ~8x the rounding error of the FP32 margins, which scales with 1/sin, 1/cos
    g.tau = (float)(4e-6 * fmax(1.0, fmax(1.0 / c, 1.0 / s)));
    g.hk = (float)((1.0 + c / s) / 2);
    g.hm = (float)(h - (c + s) / 2);
    g.y_lf = (float)(h * (s - c));
    g.y_bt = (float)(h * (s + c));
    const double mn = s < c ? s : c, mx = s < c ? c : s;
    g.hb = (float)(h * (c + s));
    g.he = (float)(h * fabs(c - s));
    g.ik = (float)(mx / mn);
    g.hq = (float)((1.0 + mn / mx) / 2);
    g.hc2 = (float)(c / 2);
    g.hs2 = (float)(s / 2);
    g.smin = (float)mn;
    g.smax = (float)mx;
    g.area_total = (float)(L * L);
    g.kq_s = (float)(1.0 / (s * L));
    g.kq_c = (float)(1.0 / (c * L));
    g.qq_cs = (float)(c / (2.0 * s));
    g.qq_sc = (float)(s / (2.0 * c));
    g.half_side = (float)(L / 2);
    g.tk_sc = (float)(s / (2.0 * c));
    g.tk_cs = (float)(c / (2.0 * s));
    g.steep = s <= c ? 1 : 0;
    g.ncross = (int)floor(L * mn) + 1;
    return g;
}

AAI_HD float aai_sat(float x) {
#if defined(__CUDA_ARCH__)
    return __saturatef(x);
#else
    return fminf(fmaxf(x, 0.0f), 1.0f);
#endif
}
// length of [lo, hi] ∩ [e, e+1] for hi >= lo, without min/max (maps to FADD.SAT)
AAI_HD float aai_overlap1_f32(float lo, float hi, float e) { return aai_sat(hi - e) - aai_sat(lo - e); }

AAI_HD void aai_chord_h_f32(const AaiShapeF &g, float ty, float &xl, float &xr) {
    xl = fmaxf(fmaf(ty, g.k_sc, -g.k_hc), fmaf(-ty, g.k_cs, -g.k_hs));
    xr = fminf(fmaf(ty, g.k_sc, g.k_hc), fmaf(-ty, g.k_cs, g.k_hs));
    xr = fmaxf(xr, xl);  // empty chord -> zero length
}
AAI_HD void aai_chord_v_f32(const AaiShapeF &g, float tx, float &yt, float &yb) {
    yt = fmaxf(fmaf(tx, g.k_cs, -g.k_hs), fmaf(-tx, g.k_sc, -g.k_hc));
    yb = fminf(fmaf(tx, g.k_cs, g.k_hs), fmaf(-tx, g.k_sc, g.k_hc));
    yb = fmaxf(yb, yt);
}

// ------------------------------------------------------------------------------------------------------------
// Packed FP32: two horizontally adjacent cells (or the two left/right edges of a quirk crossing) per instruction on
// Blackwell's packed FP32 pipe (FFMA2 / FMUL2 / FADD2, `fma.rn.f32x2` -- sm_100a).  The overlap kernel is
// instruction-issue bound and every multiply/add of the cell math is independent between cells, so two cells share
// one instruction.  (The host build of this header evaluates the two lanes with scalar fmaf.)
// ------------------------------------------------------------------------------------------------------------
struct AaiF2 {
    float x, y;
};
AAI_HD AaiF2 aai_f2(float x, float y) {
    AaiF2 r;
    r.x = x;
    r.y = y;
    return r;
}
AAI_HD AaiF2 aai_f2(float v) { return aai_f2(v, v); }
#if defined(__CUDA_ARCH__)
AAI_HD AaiF2 aai_fma2(AaiF2 a, AaiF2 b, AaiF2 c) {
    const float2 r = __ffma2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y), make_float2(c.x, c.y));
    return aai_f2(r.x, r.y);
}
AAI_HD AaiF2 aai_mul2(AaiF2 a, AaiF2 b) {
    const float2 r = __fmul2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y));
    return aai_f2(r.x, r.y);
}
AAI_HD AaiF2 aai_add2(AaiF2 a, AaiF2 b) {
    const float2 r = __fadd2_rn(make_float2(a.x, a.y), make_float2(b.x, b.y));
    return aai_f2(r.x, r.y);
}
#else
AAI_HD AaiF2 aai_fma2(AaiF2 a, AaiF2 b, AaiF2 c) { return aai_f2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
AAI_HD AaiF2 aai_mul2(AaiF2 a, AaiF2 b) { return aai_f2(a.x * b.x, a.y * b.y); }
AAI_HD AaiF2 aai_add2(AaiF2 a, AaiF2 b) { return aai_f2(a.x + b.x, a.y + b.y); }
#endif
AAI_HD AaiF2 aai_sub2(AaiF2 a, AaiF2 b) { return aai_fma2(b, aai_f2(-1.0f), a); }  // a - b as one FFMA2
// chords of the footprint on two vertical grid lines at once (same arithmetic as aai_chord_v_f32, lane by lane)
AAI_HD void aai_chord_v_f32x2(const AaiShapeF &g, AaiF2 tx, AaiF2 &yt, AaiF2 &yb) {
    const AaiF2 a = aai_fma2(tx, aai_f2(g.k_cs), aai_f2(-g.k_hs)), b = aai_fma2(tx, aai_f2(-g.k_sc), aai_f2(-g.k_hc));
    const AaiF2 c = aai_fma2(tx, aai_f2(g.k_cs), aai_f2(g.k_hs)), d = aai_fma2(tx, aai_f2(-g.k_sc), aai_f2(g.k_hc));
    yt = aai_f2(fmaxf(a.x, b.x), fmaxf(a.y, b.y));
    yb = aai_f2(fmaxf(fminf(c.x, d.x), yt.x), fmaxf(fminf(c.y, d.y), yt.y));
}


// Green form with the vertex rotation folded into the side coefficients:
//   A = lenT (1/4 + vy/2) + lenB (1/4 - vy/2) + lenL (1/4 + vx/2) + lenR (1/4 - vx/2),
//   vx = ca c + cb s,  vy = cb c - ca s,  (ca, cb) = V - cell centre along (u, v)   (hc2 = c/2, hs2 = s/2)
AAI_HD float aai_cell_exact_f32(const AaiShapeF &g, float u0, float v0, float lenT, float lenB, float lenL, float lenR) {
    const float ca = copysignf(g.half, u0) - u0;
    const float cb = copysignf(g.half, v0) - v0;
    const float aT = fmaf(cb, g.hc2, fmaf(ca, -g.hs2, 0.25f));
    const float aL = fmaf(ca, g.hc2, fmaf(cb, g.hs2, 0.25f));
    // lenT aT + lenB (1/2 - aT) + lenL aL + lenR (1/2 - aL), arranged as a shallow tree (the kernel is latency-bound)
    return fmaf(aT, lenT - lenB, fmaf(aL, lenL - lenR, 0.5f * (lenB + lenR)));
}
AAI_HD AaiF2 aai_cell_exact_f32x2(const AaiShapeF &g, AaiF2 u0, AaiF2 v0, AaiF2 lenT, AaiF2 lenB, AaiF2 lenL,
                                  AaiF2 lenR) {
    const AaiF2 ca = aai_sub2(aai_f2(copysignf(g.half, u0.x), copysignf(g.half, u0.y)), u0);
    const AaiF2 cb = aai_sub2(aai_f2(copysignf(g.half, v0.x), copysignf(g.half, v0.y)), v0);
    const AaiF2 aT = aai_fma2(cb, aai_f2(g.hc2), aai_fma2(ca, aai_f2(-g.hs2), aai_f2(0.25f)));
    const AaiF2 aL = aai_fma2(ca, aai_f2(g.hc2), aai_fma2(cb, aai_f2(g.hs2), aai_f2(0.25f)));
    const AaiF2 half_br = aai_fma2(lenB, aai_f2(0.5f), aai_mul2(lenR, aai_f2(0.5f)));
    return aai_fma2(aT, aai_sub2(lenT, lenB), aai_fma2(aL, aai_sub2(lenL, lenR), half_br));
}

// ------------------------------------------------------------------------------------------------------------
// Cell window + tips.  Anchor a window of NW x NW cells at the first cell column and row a footprint box touches; what
// of the footprint lies outside the window is its RIGHT tip F ∩ {x > window's right edge} and its BOTTOM tip
// F ∩ {y > window's bottom edge}.  When aai_tip_window_ok holds for the shape and NW = nmax - 1, for every interior
// footprint each tip is the triangle at the footprint's extreme vertex in x (resp. y), lies in the one cell column (row)
// after the window, inside the window's rows (columns), and meets at most 3 of them; the two tips are disjoint.  So the
// window's cells plus the strips of the two tips are the footprint's whole box, with the tip cells' exact areas.
// ------------------------------------------------------------------------------------------------------------
// Host, FP64, per plan: nmax = cells per axis the FP32 kernel is compiled for.  With D = L(c+s) the width of the footprint
// box, the box starts up to one cell (+ the margin m for FP32 rounding of the cell range) before the footprint, so a tip
// is at most w = D + 2 - nmax + m wide.  The right tip's lowest point, h(c-s) + w s/c, stays above the window's bottom
// edge (nmax - 1 - hb - 1 - m from the centre at worst) iff w (c+s) <= L c s; the bottom tip's rightmost point gives the
// same condition (this also keeps w below L min(c,s): the tip is bounded by the two edges at the vertex only).  Along the
// strip axis a tip is w (c/s + s/c) long: at most 3 strips while that is below 2.
inline bool aai_tip_window_ok(double c, double s, double L, int nmax) {
    const double m = 1e-3;
    const double D = L * (c + s);
    const double w = D + 2.0 - nmax + m;
    return c > 0.0 && s > 0.0 && D >= nmax - 2 + m && w < 1.0 - m && w * (c + s) <= L * c * s - m &&
           w / (c * s) <= 2.0 - m;
}

// Device (and host tests): the tips of one footprint.  e0 / t0 = left / top boundary of the window, relative to the
// centre.  Lane x: the right tip in window rows first[0] .. first[0] + 2, lane y: the bottom tip in window columns
// first[1] .. first[1] + 2; area[j] = the tip's area in its strip first + j (indices clamped into 0 .. NW-1: strips
// beyond the tip get 0).  Along the strip axis, at d from the vertex, a tip is w + k d wide on one side of the vertex and
// w - d/k on the other (k = s/c for the right tip, c/s for the bottom one), so its area up to d is
//     T(d) = a^2 / (2k) + (k/2) e (2w - e),   a = clamp(w + k d, 0, w),  e = clamp(d / k, 0, w),
// and the strip [d_j, d_j+1] holds T(d_j+1) - T(d_j).  T is 0 at the strip boundary before the tip's near end (the first
// strip is the one holding that end).  A footprint without a tip has w = 0, and every area is 0.  Branch-free; the two
// tips share packed FP32 instructions.
template <int NW>
AAI_HD void aai_tip_strips_f32(const AaiShapeF &g, float e0, float t0, int (&first)[2], AaiF2 (&area)[3]) {
    const AaiF2 o = aai_f2(t0, e0);           // strip boundary 0: top of window row 0, left of window column 0
    const AaiF2 v = aai_f2(-g.y_lf, g.y_lf);  // the vertex along the strip axis: y = h(c-s) (right), x = h(s-c) (bottom)
    const AaiF2 k = aai_f2(g.k_sc, g.k_cs), ki = aai_f2(g.k_cs, g.k_sc);
    const AaiF2 hk = aai_f2(g.tk_sc, g.tk_cs), hki = aai_f2(g.tk_cs, g.tk_sc);
    const AaiF2 wr = aai_sub2(aai_f2(g.hb - (float)NW), aai_f2(e0, t0));  // hb - the window's right / bottom edge
    const AaiF2 w = aai_f2(fmaxf(wr.x, 0.0f), fmaxf(wr.y, 0.0f)), w2 = aai_add2(w, w);
    const AaiF2 rel = aai_sub2(aai_fma2(w, aai_f2(-ki.x, -ki.y), v), o);  // the tip's near end, from boundary 0
    int f0 = (int)floorf(rel.x), f1 = (int)floorf(rel.y);
    f0 = f0 < 0 ? 0 : (f0 > NW - 1 ? NW - 1 : f0);
    f1 = f1 < 0 ? 0 : (f1 > NW - 1 ? NW - 1 : f1);
    first[0] = f0;
    first[1] = f1;
    const AaiF2 d0 = aai_add2(aai_sub2(o, v), aai_f2((float)f0, (float)f1));
    AaiF2 prev = aai_f2(0.0f);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const AaiF2 d = aai_add2(d0, aai_f2((float)(j + 1)));
        const AaiF2 a = aai_fma2(k, d, w), e = aai_mul2(d, ki);
        const AaiF2 ac = aai_f2(fminf(fmaxf(a.x, 0.0f), w.x), fminf(fmaxf(a.y, 0.0f), w.y));
        const AaiF2 ec = aai_f2(fminf(fmaxf(e.x, 0.0f), w.x), fminf(fmaxf(e.y, 0.0f), w.y));
        const AaiF2 t = aai_fma2(aai_mul2(ac, ac), hki, aai_mul2(hk, aai_mul2(ec, aai_sub2(w2, ec))));
        area[j] = aai_sub2(t, prev);
        prev = t;
    }
}

// ------------------------------------------------------------------------------------------------------------
// Upscaling (expansion S >= 3, footprint narrower than one source pixel + 1 cell): the <= 4 x 4 expanded cells a
// footprint touches are replicas of at most 2 x 2 source pixels, separated by ONE vertical source-pixel boundary
// x = Cx + tX and ONE horizontal one y = Cy + tY (coordinates relative to the footprint centre; hasX / hasY false
// when there is no such boundary inside the cell range: every cell then lies on its near side).  The exact cell areas of Source.cpp:1052-1401 add up, per source pixel, to
// the area of the footprint inside that pixel's quadrant, so the four weights are computed directly instead of cell
// by cell: Green's theorem about the corner P = (tX, tY) --
//     area(footprint ∩ quadrant) = 1/2 sum over the 4 footprint edges of  dist(P, edge line) * |edge ∩ quadrant|
// (the two boundary lines pass through P and contribute nothing; the signed distance makes it valid for P outside the
// footprint too).  Along an edge the quadrant changes where the edge crosses x = tX resp. y = tY: two clamped linear
// parameters per edge (one FFMA.SAT each, normalised to [0, 1]), so the four weights cost ~60 instructions instead of
// a row loop over 16 cells.  W[r][c]: r = 0 above the horizontal boundary (y < tY), c = 0 left of the vertical one.
// The four weights add up to L^2.  (The reference's shape-2/4 quirk is applied on top, per edge crossing, as in the
// general path.)
// ------------------------------------------------------------------------------------------------------------
AAI_HD void aai_quadrant_areas_f32(const AaiShapeF &g, float tX, float tY, bool hasX, bool hasY, float &W00,
                                   float &W01, float &W10, float &W11) {
    // A boundary that does not cross the footprint puts every cell on its near side (x < tX resp. y < tY always true);
    // P then sits on the footprint's centre line, so that the signed distances stay O(L) and nothing cancels.
    const float px = hasX ? tX : 0.0f, py = hasY ? tY : 0.0f;
    // footprint-local coordinates of P and its signed distances to the four edge lines (positive inside), times L/2
    const float uP = fmaf(px, g.cs, -py * g.sn), vP = fmaf(px, g.sn, py * g.cs);
    const float D1 = (g.half - uP) * g.half_side, D2 = (g.half + uP) * g.half_side;  // edges u = +h, u = -h
    const float D3 = (g.half - vP) * g.half_side, D4 = (g.half + vP) * g.half_side;  // edges v = +h, v = -h
    // u = +-h (direction (s, c): x and y both grow with the parameter): x < tX <=> t < a, y < tY <=> t < b
    {
        const float a1 = hasX ? aai_sat(fmaf(px, g.kq_s, 0.5f - g.qq_cs)) : 1.0f, b1 = hasY ? aai_sat(fmaf(py, g.kq_c, 0.5f + g.qq_sc)) : 1.0f;
        const float a2 = hasX ? aai_sat(fmaf(px, g.kq_s, 0.5f + g.qq_cs)) : 1.0f, b2 = hasY ? aai_sat(fmaf(py, g.kq_c, 0.5f - g.qq_sc)) : 1.0f;
        const float lo1 = fminf(a1, b1), hi1 = fmaxf(a1, b1), lo2 = fminf(a2, b2), hi2 = fmaxf(a2, b2);
        W00 = fmaf(D1, lo1, D2 * lo2);
        W11 = fmaf(D1, 1.0f - hi1, D2 * (1.0f - hi2));
        // the middle piece lies left of the vertical boundary (and below the horizontal one) iff a > b
        const float m1 = D1 * (hi1 - lo1), m2 = D2 * (hi2 - lo2);
        W10 = (a1 > b1 ? m1 : 0.0f) + (a2 > b2 ? m2 : 0.0f);
        W01 = (a1 > b1 ? 0.0f : m1) + (a2 > b2 ? 0.0f : m2);
    }
    // v = +-h (direction (c, -s): x grows, y falls with the parameter): x < tX <=> t < a, y < tY <=> t > b
    {
        const float a3 = hasX ? aai_sat(fmaf(px, g.kq_c, 0.5f - g.qq_sc)) : 1.0f, b3 = hasY ? aai_sat(fmaf(-py, g.kq_s, 0.5f + g.qq_cs)) : 0.0f;
        const float a4 = hasX ? aai_sat(fmaf(px, g.kq_c, 0.5f + g.qq_sc)) : 1.0f, b4 = hasY ? aai_sat(fmaf(-py, g.kq_s, 0.5f - g.qq_cs)) : 0.0f;
        const float lo3 = fminf(a3, b3), hi3 = fmaxf(a3, b3), lo4 = fminf(a4, b4), hi4 = fmaxf(a4, b4);
        W10 += fmaf(D3, lo3, D4 * lo4);
        W01 += fmaf(D3, 1.0f - hi3, D4 * (1.0f - hi4));
        const float m3 = D3 * (hi3 - lo3), m4 = D4 * (hi4 - lo4);
        W00 += (a3 > b3 ? m3 : 0.0f) + (a4 > b4 ? m4 : 0.0f);
        W11 += (a3 > b3 ? 0.0f : m3) + (a4 > b4 ? 0.0f : m4);
    }
}

// ------------------------------------------------------------------------------------------------------------
// Edge formulation of the reference's shape-2/4 quirk (what the kernels run).  Every cell first gets its exact overlap
// (Green form above, no decision).  For a corner cut with legs (lx, ly) by a left/right footprint edge,
//     reference area - exact area = +1/2 (1 - lx - ly)   if the cut corner is the only one inside (shape 2),
//                                   -1/2 (1 - lx - ly)   if it is the only one outside (shape 4),
// and it applies iff no other footprint edge meets the cell.  The affected cells are exactly those in which a
// left/right edge changes from "advancing along its major axis" to "stepping over a minor-axis grid line" -- one pair
// of cells per minor-axis grid line the edge SEGMENT crosses, at most floor(L min(s,c)) + 1 of them -- so they are
// enumerated per edge.  (tests/cell_legacy_forms.h keeps the earlier per-cell and per-row formulations as
// independent cross-checks.)
//
// Axes: the left/right edges have direction (s,c).  Major axis = y if s <= c ("steep"), else x; minor = the other.
// Along the edge both coordinates increase; kappa = min/max is the minor advance per unit of major advance.  At a
// crossing of the minor grid line Q, at major coordinate p* = (cell index Mi) + f:
//   "before" cell (minor index mi,   major index Mi): the edge entered through its lower major side and leaves through
//            the grid line: legs f and f*kappa                     -> 1/2 (1 - lx - ly) = 1/2 - f hq
//   "after"  cell (minor index mi+1, major index Mi): legs (1-f) and (1-f)*kappa     -> 1/2 - (1-f) hq
// (steep: before = top-right cut, after = bottom-left cut; shallow: the other way round).  In (major, minor)
// coordinates relative to the footprint centre the edges are, with D = h(c+s), E = h|c-s|:
//   ALPHA (left edge if steep, right edge if shallow): major in [-E, D], minor in [-D, -E]; the before cell has its
//         cut corner INSIDE the footprint (reference shape 2, +), the after cell OUTSIDE (shape 4, -);
//   BETA  (right edge if steep, left edge if shallow): major in [-D, E], minor in [E, D]; before = outside, after =
//         inside.
// Validity: inside case <=> both crossing points of the cell lie on the edge segment;
// outside case <=> the whole cell lies in the top/bottom slab, |v0| <= h - m, v0 = minor*min(s,c) + major*max(s,c).
//   g0m, g0M : coordinate of grid line 0 on the minor / major axis (left boundary of column 0 resp. top of row 0)
//   n        : which crossing of this edge (0 = first minor grid line after the edge's start)
// Outputs: (mi, Mi) = before cell (the after cell is (mi+1, Mi)); d_before / d_after = signed area corrections, 0
// when the cell is not a quirk cell.  `worst` accumulates the smallest decision margin.
// ------------------------------------------------------------------------------------------------------------
template <bool ALPHA>
AAI_HD void aai_edge_quirk_f32(const AaiShapeF &g, float g0m, float g0M, int n, int &mi, int &Mi, float &d_before,
                               float &d_after, float &worst) {
    const float qA = ALPHA ? -g.hb : g.he, qB = ALPHA ? -g.he : g.hb;
    const float pA = ALPHA ? -g.he : -g.hb;
    const float span = g.hb + g.he;  // pB - pA
    const float icf = ceilf(qA - g0m) + (float)n;
    const float Q = g0m + icf;
    const float dq = Q - qA;
    const float ex = fminf(dq, qB - Q);  // the grid line really crosses the segment
    const float along = dq * g.ik;       // major-axis distance from the edge's start to the crossing
    const float rel = (pA - g0M) + along;
    const float Mf = floorf(rel);
    const float f = rel - Mf, f1 = 1.0f - f;
    const float d_b = fmaf(-f, g.hq, 0.5f), d_a = fmaf(-f1, g.hq, 0.5f);
    const float pc = (g0M + Mf) + 0.5f;  // major coordinate of the two cells' centres
    float val_in, val_out;
    if (ALPHA) {
        val_in = fminf(along - f, span - along);
        val_out = g.hm - fabsf(fmaf(Q + 0.5f, g.smin, pc * g.smax));
    } else {
        val_in = fminf((span - along) - f1, along);
        val_out = g.hm - fabsf(fmaf(Q - 0.5f, g.smin, pc * g.smax));
    }
    val_in = fminf(val_in, ex);
    val_out = fminf(val_out, ex);
    // Decision margins.  A crossing within the guard band of a lattice corner (f ~ 0 or 1) may be assigned to the wrong
    // pair of cells, so it is flagged whatever the validity of the cells FP32 happened to pick.
    if (ex > -g.tau) worst = fminf(worst, fminf(f, f1));
    if (fmaxf(val_in, val_out) > -g.tau) worst = fminf(worst, fminf(fabsf(val_in), fabsf(val_out)));
    mi = (int)icf - 1;
    Mi = (int)Mf;
    if (ALPHA) {
        d_before = val_in > 0.0f ? d_b : 0.0f;
        d_after = val_out > 0.0f ? -d_a : 0.0f;
    } else {
        d_before = val_out > 0.0f ? -d_b : 0.0f;
        d_after = val_in > 0.0f ? d_a : 0.0f;
    }
}

// Both edges of one crossing index at once on the packed FP32 pipe: lane .x = ALPHA, lane .y = BETA.  Same arithmetic as
// aai_edge_quirk_f32, operation by operation (the CPU tests compare the two bit for bit); the kernel is issue-bound
// and the two edges' computations are independent, so they share instructions.
AAI_HD void aai_edge_quirk_pair_f32(const AaiShapeF &g, float g0m, float g0M, int n, int (&mi)[2], int (&Mi)[2],
                                    float (&d_before)[2], float (&d_after)[2], float &worst) {
    const AaiF2 qA = aai_f2(-g.hb, g.he), qB = aai_f2(-g.he, g.hb), pA = aai_f2(-g.he, -g.hb);
    const float span = g.hb + g.he;
    const AaiF2 t = aai_sub2(qA, aai_f2(g0m));
    const AaiF2 icf = aai_add2(aai_f2(ceilf(t.x), ceilf(t.y)), aai_f2((float)n));
    const AaiF2 Q = aai_add2(aai_f2(g0m), icf);
    const AaiF2 dq = aai_sub2(Q, qA);
    const AaiF2 qr = aai_sub2(qB, Q);
    const float ex_a = fminf(dq.x, qr.x), ex_b = fminf(dq.y, qr.y);
    const AaiF2 along = aai_mul2(dq, aai_f2(g.ik));
    const AaiF2 rel = aai_add2(aai_sub2(pA, aai_f2(g0M)), along);
    const AaiF2 Mf = aai_f2(floorf(rel.x), floorf(rel.y));
    const AaiF2 f = aai_sub2(rel, Mf), f1 = aai_sub2(aai_f2(1.0f), f);
    const AaiF2 d_b = aai_fma2(f, aai_f2(-g.hq), aai_f2(0.5f)), d_a = aai_fma2(f1, aai_f2(-g.hq), aai_f2(0.5f));
    const AaiF2 pc = aai_add2(aai_add2(aai_f2(g0M), Mf), aai_f2(0.5f));
    const AaiF2 rest = aai_sub2(aai_f2(span), along);         // span - along
    const AaiF2 af = aai_sub2(along, f), rf1 = aai_sub2(rest, f1);
    const AaiF2 vv = aai_fma2(aai_add2(Q, aai_f2(0.5f, -0.5f)), aai_f2(g.smin), aai_mul2(pc, aai_f2(g.smax)));
    const float vin_a = fminf(fminf(af.x, rest.x), ex_a), vout_a = fminf(g.hm - fabsf(vv.x), ex_a);
    const float vin_b = fminf(fminf(rf1.y, along.y), ex_b), vout_b = fminf(g.hm - fabsf(vv.y), ex_b);
    if (ex_a > -g.tau) worst = fminf(worst, fminf(f.x, f1.x));
    if (fmaxf(vin_a, vout_a) > -g.tau) worst = fminf(worst, fminf(fabsf(vin_a), fabsf(vout_a)));
    if (ex_b > -g.tau) worst = fminf(worst, fminf(f.y, f1.y));
    if (fmaxf(vin_b, vout_b) > -g.tau) worst = fminf(worst, fminf(fabsf(vin_b), fabsf(vout_b)));
    mi[0] = (int)icf.x - 1;
    mi[1] = (int)icf.y - 1;
    Mi[0] = (int)Mf.x;
    Mi[1] = (int)Mf.y;
    d_before[0] = vin_a > 0.0f ? d_b.x : 0.0f;   // ALPHA: before = corner inside (+), after = corner outside (-)
    d_after[0] = vout_a > 0.0f ? -d_a.x : 0.0f;
    d_before[1] = vout_b > 0.0f ? -d_b.y : 0.0f;  // BETA: the other way round
    d_after[1] = vin_b > 0.0f ? d_a.y : 0.0f;
}

// FP64 form of aai_edge_quirk_f32 (the unrolled FP64 kernel): decisions are made directly on FP64 margins, there is no
// guard band.
template <bool ALPHA>
AAI_HD void aai_edge_quirk_f64(const AaiShape &g, double g0m, double g0M, int n, int &mi, int &Mi, double &d_before,
                               double &d_after) {
    const double qA = ALPHA ? -g.hb : g.he, qB = ALPHA ? -g.he : g.hb;
    const double pA = ALPHA ? -g.he : -g.hb;
    const double span = g.hb + g.he;
    const double icf = ceil(qA - g0m) + (double)n;
    const double Q = g0m + icf;
    const double dq = Q - qA;
    const double ex = fmin(dq, qB - Q);
    const double along = dq * g.ik;
    const double rel = (pA - g0M) + along;
    const double Mf = floor(rel);
    const double f = rel - Mf, f1 = 1.0 - f;
    const double d_b = 0.5 - f * g.hq, d_a = 0.5 - f1 * g.hq;
    const double pc = (g0M + Mf) + 0.5;
    double val_in, val_out;
    if (ALPHA) {
        val_in = fmin(along - f, span - along);
        val_out = g.hm - fabs((Q + 0.5) * g.smin + pc * g.smax);
    } else {
        val_in = fmin((span - along) - f1, along);
        val_out = g.hm - fabs((Q - 0.5) * g.smin + pc * g.smax);
    }
    val_in = fmin(val_in, ex);
    val_out = fmin(val_out, ex);
    // (saturating conversions: a crossing that does not exist can lie far outside the int range at tiny angles)
    mi = icf > -1e9 && icf < 1e9 ? (int)icf - 1 : -1;
    Mi = Mf > -1e9 && Mf < 1e9 ? (int)Mf : -1;
    if (ALPHA) {
        d_before = val_in > 0.0 ? d_b : 0.0;
        d_after = val_out > 0.0 ? -d_a : 0.0;
    } else {
        d_before = val_out > 0.0 ? -d_b : 0.0;
        d_after = val_in > 0.0 ? d_a : 0.0;
    }
}


#endif  // AAI_CELL_CUH_
