// sf_prep.cu -- K1+K2 fused, marching form: bilinear warp + image derivatives + two-frame data term
// + div(psi grad w) + 2x2 block inverse in ONE pass over the frame pair (sm_100a).
//
// Replaces, per outer iteration of the two-frame path (variational.c:40-57):
//     image_warp                  variational_aux.c:18-52     (the warped image and its mask never exist in HBM)
//     get_derivatives             variational_aux.c:55-78     (nor do the 24 derivative planes)
//     compute_data_and_match      variational_aux.c:215-302
//     sub_laplacian x2            variational_aux.c:153-180
//     block inverse of sor_coupled's first sweep              solver.c:101-106
// HBM traffic: read wx,wy (8 B/px) + im1 (12) + im2 through L1/L2 gathers (12) + psi_h,psi_v (8); write the five
// system planes (20).  SURVEY 8(d) counts 52 B/px for this step.
// k_prep_fused (the default loop, niter_inner == 1) also does the smoothness pass that precedes it (k_flow_smooth):
// it reads dpsis (4 B/px) and, after the first outer iteration, du,dv (8) instead of psi_h,psi_v, and writes
// psi_h,psi_v (8) and the updated flow (8): 64 B/px in the first outer iteration, 80 after it.
//
// Work decomposition (no CTA barrier):
//   * one WARP owns a strip of 64 columns (lane l = columns 2l, 2l+1) and marches down a segment of rows;
//   * every per-row quantity is a packed (column 2l, column 2l+1) pair in one 64-bit register, so the vertical
//     stencils, the robust weights and the 2x2 system run on FFMA2 (sf_pack.cuh);
//   * vertical taps come from rolling 4-row windows (m, z, Ix, Iy, Iyz per channel = 60 packed values per lane) that
//     live in the warp's PRIVATE slice of shared memory ([array][channel][slot][lane]: conflict-free 8-byte accesses, no
//     synchronisation); horizontal taps come from the neighbouring lanes by warp shuffle.  The 5-tap-of-5-tap stencil
//     needs +-4 columns = 2 lanes, so lanes 2..29 (56 columns) produce output and consecutive strips overlap by 8;
//   * row r is loaded (and im2 warped) at step r; the output row of step r is o = r - 4.
// Why shared-memory windows: with the windows in registers the slot of a row had to be a compile-time index, i.e. the
// marching step was unrolled four times -- 255 registers (8 warps per SM) and a loop body of ~77 KB that thrashed the
// instruction cache (ncu: 11 % of the stall samples "no instruction").  A run-time slot index into shared memory gives
// a rolled loop, 168 registers, 12 resident warps per SM: 135.7 us -> 112.7 us per launch at 2560x1440.
// Border semantics follow image.c:400-526: rows / columns outside the image are clamped at load time, which
// reproduces the replicate border of the first derivative stage; the second stage (d/dx of Ix, d/dy of Iy)
// replicates the first-stage VALUE, which is patched explicitly in edge strips / segments.
#include <atomic>
#include <type_traits>

#include "sf_internal.cuh"
#include "sf_pack.cuh"
#include "sf_stencil.cuh"
#include "sf_march.cuh"

namespace sf {

constexpr int PR_WARPS = 2;                             // warps per CTA (independent; 2 x 15 KB of window storage)
#ifndef SF_PREP_MINB
#define SF_PREP_MINB 6 // resident CTAs per SM the register allocation aims at (6 x 2 warps, 6 x 30 KB of windows)
#endif
constexpr int PR_RING = 60 * 32;                        // packed values of one warp's windows
constexpr int PR_RING_PSI = 68 * 32;                    // ... plus 4 rows of the flow (u, v) when the kernel forms psi


// 1/sqrt of both halves of a pair whose values are >= 1e-6 (or NaN): MUFU.RSQ as rsqrtf issues it, without the
// rescaling of denormal inputs that rsqrtf wraps around it (it never triggers above FLT_MIN), so the result is
// bit-identical to rsqrtf's for these inputs
__device__ __forceinline__ p64 rsqrt2_normal(p64 s) {
    float a, b;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(a) : "f"(lo_of(s)));
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(b) : "f"(hi_of(s)));
    return pk(a, b);
}

struct PrepArgs {
    Geom g;
    const float *im1, *im2; // 3 planes each
    const float *wx, *wy;   // flow: warps im2 and is the argument of the Laplacian
    const float *du, *dv;   // INC: current increment (nullable: 0); UPDATE: the flow is (wx + du, wy + dv)
    const float *ph, *pv;   // smoothness diffusivities (read unless the kernel forms them: PSI)
    float *a11, *a12, *a22, *b1, *b2;
    float hd, hg;           // 0.5*delta/3, 0.5*gamma/3
    int strips, seg_rows, nwork;
    // PSI only: the diffusivities are formed from the flow and the weight map dpsis and stored to (ph_out, pv_out);
    // UPDATE also stores the updated flow to (wx_out, wy_out)
    const float *dpsis;
    float half_alpha;
    float *ph_out, *pv_out, *wx_out, *wy_out;
};

// One warp marches down its (strip, segment).  EDGE: the strip touches the left or right image border.
// INC: the data term is linearised around a non-zero increment (du,dv); the default two-frame path (niter_inner == 1)
// evaluates it at du = dv = 0, where the residuals are Iz / Ixz / Iyz themselves.
// PSI: the smoothness diffusivities psi_h / psi_v of the output row are computed here (what k_flow_smooth<UPDATE, 1>
// computes, with the same rounding) instead of being read; UPDATE (PSI only): the flow is w + du, formed on the fly.
// The flow rows r-3 .. r then live in the warp's ring: a row is loaded once, for the warp, and read back three steps
// later for the Laplacian and psi of the output row, whose Laplacian window (rows o-1, o, o+1) is exactly what psi_h(o)
// and psi_v(o) are made of.
template <bool COLOR, bool EDGE, bool INC, bool PSI = false, bool UPDATE = false>
__device__ __forceinline__ void prep_march(const PrepArgs &a, const int strip, const int seg, const int lane, p64 *ring_sm) {
    static_assert(!(PSI && INC) && (PSI || !UPDATE), "PSI is the niter_inner == 1 form (data term at du = 0)");
    const Geom g = a.g;
    const int W = g.W, H = g.H, H1 = H - 1, S = g.S;
    const int P = (int)g.plane();

    Lane L;
    const int X0 = strip * PR_OUT_W - 2 * PR_OUT_LO;
    L.x0 = X0 + 2 * lane;
    L.xc0 = clampi(L.x0, 0, W - 1);
    L.xc1 = clampi(L.x0 + 1, 0, W - 1);
    L.lane_l = clampi((0 - X0) >> 1, 0, 31);
    L.lane_r = clampi((W - 1 - X0) >> 1, 0, 31);
    L.comp_r = (W - 1 - X0) & 1;

    const int Y0 = seg * a.seg_rows;
    const int Yend = min(Y0 + a.seg_rows, H);
    const int Rbase = Y0 - 4;

    const bool out_lane = (lane >= PR_OUT_LO) && (lane <= PR_OUT_HI) && (L.x0 < S);
    const bool v0 = L.x0 < W, v1 = L.x0 + 1 < W; // valid (non-padding) columns of the pair
    const float fxc0 = (float)L.xc0, fxc1 = (float)L.xc1;

    const p64 zero2 = splat2(0.0f), half2 = splat2(0.5f), mone2 = splat2(-1.0f);
    const p64 dnorm2 = splat2(0.1f * 0.1f);
    const float eps_color = 0.001f * 0.001f, eps_grad = 0.001f * 0.001f;
    const float Wm1 = (float)(W - 1), Hm1 = (float)H1;

    // rolling windows in the warp's slice of shared memory; the slot of a row is a run-time index
    enum { RG_M = 0, RG_Z = 1, RG_IX = 2, RG_IYZ = 3, RG_IY = 4 };
    p64 *const sm = ring_sm + lane;
    auto rd = [&](int arr, int c, int s) -> p64 { return sm[((arr * 3 + c) * 4 + s) * 32]; };
    auto wr = [&](int arr, int c, int s, p64 v) { sm[((arr * 3 + c) * 4 + s) * 32] = v; };
#pragma unroll
    for (int k = 0; k < (PSI ? 68 : 60); k++) sm[k * 32] = zero2;
    // PSI: flow ring, slot s of u / v (the slot of row r is the same as in the derivative windows)
    enum { RG_FU = 60, RG_FV = 64 };
    auto frd = [&](int arr, int s) -> p64 { return sm[(arr + s) * 32]; };
    auto fwr = [&](int arr, int s, p64 v) { sm[(arr + s) * 32] = v; };

    // software pipeline: im1 and the flow of the NEXT row to be warped are loaded one step ahead
    p64 An[3], fx, fy, fdx = zero2, fdy = zero2;
    {
        const int ro = clampi(Rbase, 0, H1) * S;
#pragma unroll
        for (int c = 0; c < 3; c++) An[c] = load_pair<EDGE>(a.im1 + c * P, ro, L);
        fx = load_pair<EDGE>(a.wx, ro, L);
        fy = load_pair<EDGE>(a.wy, ro, L);
        if (UPDATE) {
            fdx = load_pair<EDGE>(a.du, ro, L);
            fdy = load_pair<EDGE>(a.dv, ro, L);
        }
    }
    p64 lu_m = zero2, lu_0 = zero2, lv_m = zero2, lv_0 = zero2; // Laplacian window: flow of rows o-1, o
    p64 vt = zero2;                                            // psi_v of row o-1
    // PSI: dpsis of row o; the neighbouring lanes' edge columns of the flow: left and right of row o, right of row o-1
    p64 dw0 = zero2;
    float u0l = 0.0f, u0r = 0.0f, v0l = 0.0f, v0r = 0.0f, umr = 0.0f, vmr = 0.0f;
    const p64 ha2 = splat2(a.half_alpha), q2 = splat2(0.25f), eps_s2 = splat2(0.001f * 0.001f);

    // PSI, start of step r: the (updated) flow of row r enters the ring; row o+1 = r-3 comes back out of it with its
    // edge columns from the neighbouring lanes, and dpsis of row o+1 is loaded
    auto psi_rows = [&](const int U, const int U1, const int on, p64 &lu_p, p64 &lv_p, p64 &dw_p, float &upl, float &upr,
                        float &vpl, float &vpr) {
        if (UPDATE) { // variational.c:60-61 for niter_inner == 1: w + du (k_flow_smooth<1, 1> forms the same sum)
            fx = add2(fx, fdx);
            fy = add2(fy, fdy);
        }
        fwr(RG_FU, U, fx);
        fwr(RG_FV, U, fy);
        lu_p = frd(RG_FU, U1);
        lv_p = frd(RG_FV, U1);
        dw_p = load_pair<EDGE>(a.dpsis, on, L);
        upl = __shfl_up_sync(0xffffffffu, hi_of(lu_p), 1);
        upr = __shfl_down_sync(0xffffffffu, lo_of(lu_p), 1);
        vpl = __shfl_up_sync(0xffffffffu, hi_of(lv_p), 1);
        vpr = __shfl_down_sync(0xffffffffu, lo_of(lv_p), 1);
    };
    // psi_v of row o (variational_aux.c:127-142 with the arithmetic of k_flow_smooth: the cross term is
    // 0.25 * ((w(x+1) - w(x-1)) + (w'(x+1) - w'(x-1))), its square is added by FFMA to dy^2, the two flow components are
    // summed, and (w + w') * half_alpha is multiplied by MUFU.RSQ of that plus 1e-6); 0 in the last row and beyond W-1
    auto psi_v = [&](const int o, const p64 wl_u, const p64 wr_u, const p64 wl_v, const p64 wr_v, const p64 lu_p,
                     const p64 lv_p, const p64 dw_p, float upl, float upr, float vpl, float vpr) -> p64 {
        const p64 tu = mul2(q2, add2(sub2(wr_u, wl_u), sub2(pk(hi_of(lu_p), upr), pk(upl, lo_of(lu_p)))));
        const p64 tv = mul2(q2, add2(sub2(wr_v, wl_v), sub2(pk(hi_of(lv_p), vpr), pk(vpl, lo_of(lv_p)))));
        const p64 uy = sub2(lu_p, lu_0), vy = sub2(lv_p, lv_0);
        const p64 s = add2(add2(fma2(uy, uy, mul2(tu, tu)), fma2(vy, vy, mul2(tv, tv))), eps_s2);
        const p64 r = mul2(mul2(add2(dw0, dw_p), ha2), rsqrt2_normal(s)); // s >= 1e-6
        const bool rowok = o < H1;
        return pk((rowok && L.x0 < W) ? lo_of(r) : 0.0f, (rowok && L.x0 + 1 < W) ? hi_of(r) : 0.0f);
    };

    // one marching step; U = (r - Rbase) & 3 is the ring slot of row r.  Everything is computed unconditionally
    // (rows are clamped); only the stores are predicated, so every shuffle sits in straight-line code.
    auto step = [&](const int U, const int r) {
        const int U1 = (U + 1) & 3, U2 = (U + 2) & 3, U3 = (U + 3) & 3;
        const int rr = clampi(r, 0, H1);
        const int o = r - 4, oc = clampi(o, 0, H1);
        const bool out_row = (o >= Y0) && (o < Yend); // warp-uniform
        const int oo = oc * S, on = clampi(o + 1, 0, H1) * S;
        p64 lu_p, lv_p, dw_p = zero2; // flow of row o+1; PSI: dpsis of row o+1
        float upl = 0.0f, upr = 0.0f, vpl = 0.0f, vpr = 0.0f;
        if (PSI) psi_rows(U, U1, on, lu_p, lv_p, dw_p, upl, upr, vpl, vpr);

        // ---- issue the gathers of row r (flow prefetched one step ago) and the loads of the next row
        const Taps t0 = warp_taps(g, fxc0 + lo_of(fx), (float)rr + lo_of(fy));
        const Taps t1 = warp_taps(g, fxc1 + hi_of(fx), (float)rr + hi_of(fy));
        p64 A[3], B[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            A[c] = An[c];
            B[c] = pk(warp_fetch(a.im2 + c * P, t0), warp_fetch(a.im2 + c * P, t1));
        }
        {
            const int rn = clampi(r + 1, 0, H1) * S;
#pragma unroll
            for (int c = 0; c < 3; c++) An[c] = load_pair<EDGE>(a.im1 + c * P, rn, L);
            fx = load_pair<EDGE>(a.wx, rn, L);
            fy = load_pair<EDGE>(a.wy, rn, L);
            if (UPDATE) {
                fdx = load_pair<EDGE>(a.du, rn, L);
                fdy = load_pair<EDGE>(a.dv, rn, L);
            }
        }
        p64 hr, vb; // psi_h, psi_v of row o
        if (!PSI) {
            lu_p = load_pair<EDGE>(a.wx, on, L);
            lv_p = load_pair<EDGE>(a.wy, on, L);
            hr = load_pair<EDGE>(a.ph, oo, L);
            vb = load_pair<EDGE>(a.pv, oo, L);
        }
        if (PSI) {
            // psi_h of row o (variational_aux.c:112-126, arithmetic of k_flow_smooth as in psi_v); 0 from column W-1 on
            const p64 wl_u = pk(u0l, lo_of(lu_0)), wr_u = pk(hi_of(lu_0), u0r); // columns x-1 / x+1 of row o
            const p64 wl_v = pk(v0l, lo_of(lv_0)), wr_v = pk(hi_of(lv_0), v0r);
            const float dwr = __shfl_down_sync(0xffffffffu, lo_of(dw0), 1);
            const p64 du_ = sub2(lu_p, lu_m), dv_ = sub2(lv_p, lv_m);
            const p64 tu = mul2(q2, add2(du_, pk(hi_of(du_), upr - umr)));
            const p64 tv = mul2(q2, add2(dv_, pk(hi_of(dv_), vpr - vmr)));
            const p64 ux = sub2(wr_u, lu_0), vx = sub2(wr_v, lv_0);
            const p64 s = add2(add2(fma2(ux, ux, mul2(tu, tu)), fma2(vx, vx, mul2(tv, tv))), eps_s2);
            const p64 h = mul2(mul2(add2(dw0, pk(hi_of(dw0), dwr)), ha2), rsqrt2_normal(s));
            hr = pk(L.x0 < W - 1 ? lo_of(h) : 0.0f, L.x0 + 1 < W - 1 ? hi_of(h) : 0.0f);
            vb = psi_v(o, wl_u, wr_u, wl_v, wr_v, lu_p, lv_p, dw_p, upl, upr, vpl, vpr);
        }
        p64 u = zero2, v = zero2;
        if (INC) {
            u = load_pair<EDGE>(a.du, oo, L);
            v = load_pair<EDGE>(a.dv, oo, L);
        }

        // ---- work that does not need row r: Ix of row r-2, the x-derivatives and Ixy of the output row
        p64 ix_new[3], ixx[3], ixz[3], ixy[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            ix_new[c] = hconv_pair(rd(RG_M, c, U2));
            if (EDGE) ix_new[c] = xedge_fix(ix_new[c], L, W);
            ixx[c] = hconv_pair(rd(RG_IX, c, U)); // (columns outside the image were patched in Ix itself)
            ixz[c] = hconv_pair(rd(RG_Z, c, U));
            ixy[c] = vconv_pair(rd(RG_IX, c, U2), rd(RG_IX, c, U3), rd(RG_IX, c, U1), ix_new[c]);
            wr(RG_IX, c, U2, ix_new[c]); // Ix of row r-6 is not needed any more: its slot takes row r-2
        }
        // psi_h of the left edge from the neighbouring lane (0 at column 0), psi_v of the row above (0 at row 0),
        // flow neighbours in row o, mask of the warp at row o
        const float hl_lane = __shfl_up_sync(0xffffffffu, hi_of(hr), 1);
        const p64 hl = pk(L.x0 > 0 ? hl_lane : 0.0f, lo_of(hr));
        const p64 vtt = (o > 0) ? vt : zero2;
        float ul, ur, vl, vr;
        if (PSI) { // carried from the step that brought row o out of the ring
            ul = u0l; ur = u0r; vl = v0l; vr = v0r;
        } else {
            ul = __shfl_up_sync(0xffffffffu, hi_of(lu_0), 1), ur = __shfl_down_sync(0xffffffffu, lo_of(lu_0), 1);
            vl = __shfl_up_sync(0xffffffffu, hi_of(lv_0), 1), vr = __shfl_down_sync(0xffffffffu, lo_of(lv_0), 1);
        }
        float mk0, mk1;
        {
            const float xx0 = fxc0 + lo_of(lu_0), yy0 = (float)o + lo_of(lv_0);
            const float xx1 = fxc1 + hi_of(lu_0), yy1 = (float)o + hi_of(lv_0);
            mk0 = (xx0 >= 0.0f && xx0 <= Wm1 && yy0 >= 0.0f && yy0 <= Hm1) ? 1.0f : 0.0f;
            mk1 = (xx1 >= 0.0f && xx1 <= Wm1 && yy1 >= 0.0f && yy1 <= Hm1) ? 1.0f : 0.0f;
        }

        // ---- row r: m = (B + A)/2, z = B - A; first-stage y-derivatives of row r-2; Iyy of the output row; data term
        p64 n = zero2, s11 = zero2, s12 = zero2, s22 = zero2, sb1 = zero2, sb2 = zero2;
        p64 cn = zero2, c11 = zero2, c12 = zero2, c22 = zero2, cb1 = zero2, cb2 = zero2;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const p64 m_new = mul2(add2(B[c], A[c]), half2);
            const p64 z_new = fma2(A[c], mone2, B[c]);
            p64 iy_new = vconv_pair(rd(RG_M, c, U), rd(RG_M, c, U1), rd(RG_M, c, U3), m_new);
            const p64 iyz_new = vconv_pair(rd(RG_Z, c, U), rd(RG_Z, c, U1), rd(RG_Z, c, U3), z_new);
            // second-stage replicate border in y: Iy of rows beyond the last row is Iy(H-1)
            const p64 iy_c = rd(RG_IY, c, U), iy_p1 = rd(RG_IY, c, U1), iy_b = rd(RG_IY, c, U3);
            if (r - 2 > H1) iy_new = iy_p1;
            p64 iy_m2 = rd(RG_IY, c, U2), iy_m1 = iy_b;
            if (o == 0) iy_m2 = iy_m1 = iy_c;           // rows -2, -1 take Iy(0)
            else if (o == 1) iy_m2 = iy_b;              // row -1 takes Iy(0)
            const p64 iyy = vconv_pair(iy_m2, iy_m1, iy_p1, iy_new);
            const p64 iyz = rd(RG_IYZ, c, U);
            // gradient constancy (variational_aux.c:268-296)
            const p64 ivx = rcp2(fma2(ixx[c], ixx[c], fma2(ixy[c], ixy[c], dnorm2)));
            const p64 ivy = rcp2(fma2(iyy, iyy, fma2(ixy[c], ixy[c], dnorm2)));
            const p64 rx = INC ? fma2(ixy[c], v, fma2(ixx[c], u, ixz[c])) : ixz[c];
            const p64 ry = INC ? fma2(iyy, v, fma2(ixy[c], u, iyz)) : iyz;
            n = fma2(mul2(rx, rx), ivx, n);
            n = fma2(mul2(ry, ry), ivy, n);
            const p64 px = mul2(ixx[c], ivx), sx = mul2(ixy[c], ivx), qy = mul2(ixy[c], ivy), ty = mul2(iyy, ivy);
            s11 = fma2(qy, ixy[c], fma2(px, ixx[c], s11));
            s12 = fma2(qy, iyy, fma2(px, ixy[c], s12));
            s22 = fma2(sx, ixy[c], fma2(ty, iyy, s22));
            sb1 = fma2(qy, iyz, fma2(px, ixz[c], sb1));
            sb2 = fma2(sx, ixz[c], fma2(ty, iyz, sb2));
            if (COLOR) { // colour constancy (variational_aux.c:241-266)
                const p64 ix = rd(RG_IX, c, U), iy = iy_c, iz = rd(RG_Z, c, U);
                const p64 inv = rcp2(fma2(iy, iy, fma2(ix, ix, dnorm2)));
                const p64 rc = INC ? fma2(iy, v, fma2(ix, u, iz)) : iz;
                cn = fma2(mul2(rc, rc), inv, cn);
                const p64 gx = mul2(ix, inv), gy = mul2(iy, inv);
                c11 = fma2(gx, ix, c11);
                c12 = fma2(gx, iy, c12);
                c22 = fma2(gy, iy, c22);
                cb1 = fma2(gx, iz, cb1);
                cb2 = fma2(gy, iz, cb2);
            }
            // rotate this channel's windows (every value of the slots being overwritten has been consumed above)
            wr(RG_M, c, U, m_new);
            wr(RG_Z, c, U, z_new);
            wr(RG_IY, c, U2, iy_new);
            wr(RG_IYZ, c, U2, iyz_new);
        }
        // ---- robust weights, system, Laplacian, block inverse
        const p64 tg = pk(mk0 * a.hg * rsqrtf(lo_of(n) + eps_grad), mk1 * a.hg * rsqrtf(hi_of(n) + eps_grad));
        p64 a11 = mul2(tg, s11), a12 = mul2(tg, s12), a22 = mul2(tg, s22);
        const p64 ntg = mul2(tg, mone2);
        p64 b1 = mul2(ntg, sb1), b2 = mul2(ntg, sb2);
        if (COLOR) {
            const p64 tc = pk(mk0 * a.hd * rsqrtf(lo_of(cn) + eps_color), mk1 * a.hd * rsqrtf(hi_of(cn) + eps_color));
            const p64 ntc = mul2(tc, mone2);
            a11 = fma2(tc, c11, a11);
            a12 = fma2(tc, c12, a12);
            a22 = fma2(tc, c22, a22);
            b1 = fma2(ntc, cb1, b1);
            b2 = fma2(ntc, cb2, b2);
        }
        {
            // b += div(psi grad w): left edge, right edge, upper edge, lower edge (variational_aux.c:158-179)
            const p64 nhl = mul2(hl, mone2), nvt = mul2(vtt, mone2);
            const p64 wl_u = pk(ul, lo_of(lu_0)), wr_u = pk(hi_of(lu_0), ur);
            const p64 wl_v = pk(vl, lo_of(lv_0)), wr_v = pk(hi_of(lv_0), vr);
            b1 = fma2(nhl, fma2(wl_u, mone2, lu_0), b1);
            b1 = fma2(hr, fma2(lu_0, mone2, wr_u), b1);
            b1 = fma2(nvt, fma2(lu_m, mone2, lu_0), b1);
            b1 = fma2(vb, fma2(lu_0, mone2, lu_p), b1);
            b2 = fma2(nhl, fma2(wl_v, mone2, lv_0), b2);
            b2 = fma2(hr, fma2(lv_0, mone2, wr_v), b2);
            b2 = fma2(nvt, fma2(lv_m, mone2, lv_0), b2);
            b2 = fma2(vb, fma2(lv_0, mone2, lv_p), b2);
        }
        // inverse of [[a11 + sum psi, a12], [a12, a22 + sum psi]] (solver.c:101-106)
        const p64 sp = add2(add2(add2(hl, hr), vtt), vb);
        const p64 D11 = add2(a22, sp), D22 = add2(a11, sp);
        const p64 det = fma2(mul2(a12, a12), mone2, mul2(D11, D22));
        const p64 rdet = rcp2(det);
        const p64 i11 = mul2(D11, rdet), i22 = mul2(D22, rdet), i12 = mul2(mul2(a12, mone2), rdet);
        if (out_row && out_lane) {
            const int off = o * S + L.x0;
            // padding columns: defined zeros (the reference leaves garbage there, SURVEY Q1)
            *reinterpret_cast<float2 *>(a.a11 + off) = make_float2(v0 ? lo_of(i11) : 0.0f, v1 ? hi_of(i11) : 0.0f);
            *reinterpret_cast<float2 *>(a.a12 + off) = make_float2(v0 ? lo_of(i12) : 0.0f, v1 ? hi_of(i12) : 0.0f);
            *reinterpret_cast<float2 *>(a.a22 + off) = make_float2(v0 ? lo_of(i22) : 0.0f, v1 ? hi_of(i22) : 0.0f);
            *reinterpret_cast<float2 *>(a.b1 + off) = make_float2(v0 ? lo_of(b1) : 0.0f, v1 ? hi_of(b1) : 0.0f);
            *reinterpret_cast<float2 *>(a.b2 + off) = make_float2(v0 ? lo_of(b2) : 0.0f, v1 ? hi_of(b2) : 0.0f);
            if (PSI) { // (already 0 in the padding columns)
                *reinterpret_cast<p64 *>(a.ph_out + off) = hr;
                *reinterpret_cast<p64 *>(a.pv_out + off) = vb;
            }
            if (UPDATE) {
                // the updated flow goes to the other buffer (neighbouring rows are read by other warps).  The ring holds
                // clamped columns; padding columns get the unclamped sum, as k_flow_smooth<1, 1> stores it
                p64 su = lu_0, sv = lv_0;
                if (EDGE && L.x0 + 1 >= W) {
                    float u0 = lo_of(su), v0f = lo_of(sv);
                    if (L.x0 >= W) {
                        u0 = a.wx[off] + a.du[off];
                        v0f = a.wy[off] + a.dv[off];
                    }
                    su = pk(u0, a.wx[off + 1] + a.du[off + 1]);
                    sv = pk(v0f, a.wy[off + 1] + a.dv[off + 1]);
                }
                *reinterpret_cast<p64 *>(a.wx_out + off) = su;
                *reinterpret_cast<p64 *>(a.wy_out + off) = sv;
            }
        }

        // ---- rotate the row windows of the Laplacian
        vt = vb;
        lu_m = lu_0; lu_0 = lu_p;
        lv_m = lv_0; lv_0 = lv_p;
        if (PSI) {
            umr = u0r; u0l = upl; u0r = upr;
            vmr = v0r; v0l = vpl; v0r = vpr;
            dw0 = dw_p;
        }
    };

    // The first 8 steps of a segment only fill the windows (their output rows lie above the segment): the lean step
    // loads / warps row r and rotates the windows exactly like step(), but skips the second-stage derivatives, the data
    // term, the Laplacian and the block inverse -- about 60 % of a step's instructions.
    // LAST (a std::bool_constant): the last warm-up step, the only one whose psi_v is used (PSI); a compile-time switch,
    // since a run-time test in the rolled loop costs registers
    auto lean_step = [&](const int U, const int r, auto LAST) {
        const int U1 = (U + 1) & 3, U2 = (U + 2) & 3, U3 = (U + 3) & 3;
        const int rr = clampi(r, 0, H1);
        const int o = r - 4;
        const int oo = clampi(o, 0, H1) * S, on = clampi(o + 1, 0, H1) * S;
        p64 lu_p, lv_p, dw_p = zero2;
        float upl = 0.0f, upr = 0.0f, vpl = 0.0f, vpr = 0.0f;
        if (PSI) psi_rows(U, U1, on, lu_p, lv_p, dw_p, upl, upr, vpl, vpr);
        const Taps t0 = warp_taps(g, fxc0 + lo_of(fx), (float)rr + lo_of(fy));
        const Taps t1 = warp_taps(g, fxc1 + hi_of(fx), (float)rr + hi_of(fy));
        p64 A[3], B[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            A[c] = An[c];
            B[c] = pk(warp_fetch(a.im2 + c * P, t0), warp_fetch(a.im2 + c * P, t1));
        }
        {
            const int rn = clampi(r + 1, 0, H1) * S;
#pragma unroll
            for (int c = 0; c < 3; c++) An[c] = load_pair<EDGE>(a.im1 + c * P, rn, L);
            fx = load_pair<EDGE>(a.wx, rn, L);
            fy = load_pair<EDGE>(a.wy, rn, L);
            if (UPDATE) {
                fdx = load_pair<EDGE>(a.du, rn, L);
                fdy = load_pair<EDGE>(a.dv, rn, L);
            }
        }
        p64 vb = zero2;
        if (PSI) {
            // only psi_v of the last warm-up row is used (as psi_v of the row above the first output row)
            if (decltype(LAST)::value)
                vb = psi_v(o, pk(u0l, lo_of(lu_0)), pk(hi_of(lu_0), u0r), pk(v0l, lo_of(lv_0)), pk(hi_of(lv_0), v0r), lu_p,
                           lv_p, dw_p, upl, upr, vpl, vpr);
        } else {
            lu_p = load_pair<EDGE>(a.wx, on, L);
            lv_p = load_pair<EDGE>(a.wy, on, L);
            vb = load_pair<EDGE>(a.pv, oo, L);
        }
#pragma unroll
        for (int c = 0; c < 3; c++) {
            p64 ix_new = hconv_pair(rd(RG_M, c, U2));
            if (EDGE) ix_new = xedge_fix(ix_new, L, W);
            const p64 m_new = mul2(add2(B[c], A[c]), half2);
            const p64 z_new = fma2(A[c], mone2, B[c]);
            p64 iy_new = vconv_pair(rd(RG_M, c, U), rd(RG_M, c, U1), rd(RG_M, c, U3), m_new);
            const p64 iyz_new = vconv_pair(rd(RG_Z, c, U), rd(RG_Z, c, U1), rd(RG_Z, c, U3), z_new);
            if (r - 2 > H1) iy_new = rd(RG_IY, c, U1);
            wr(RG_IX, c, U2, ix_new);
            wr(RG_M, c, U, m_new);
            wr(RG_Z, c, U, z_new);
            wr(RG_IY, c, U2, iy_new);
            wr(RG_IYZ, c, U2, iyz_new);
        }
        vt = vb;
        lu_m = lu_0; lu_0 = lu_p;
        lv_m = lv_0; lv_0 = lv_p;
        if (PSI) {
            umr = u0r; u0l = upl; u0r = upr;
            vmr = v0r; v0l = vpl; v0r = vpr;
            dw0 = dw_p;
        }
    };

    const int Rend = Yend + 4; // last loaded row is Yend + 3
#ifndef SF_PREP_LEAN
#define SF_PREP_LEAN 1
#endif
#if SF_PREP_LEAN
    // output row o = r - 4 reaches the segment at r = Y0 + 4: steps Rbase .. Y0 + 3 are warm-up
#pragma unroll 1
    for (int r = Rbase; r < Y0 + 3; r++) lean_step((r - Rbase) & 3, r, std::false_type());
    lean_step((Y0 + 3 - Rbase) & 3, Y0 + 3, std::true_type());
#pragma unroll 1
    for (int r = Y0 + 4; r < Rend; r++) step((r - Rbase) & 3, r);
#else
#pragma unroll 1
    for (int r = Rbase; r < Rend; r++) step((r - Rbase) & 3, r);
#endif
}

template <bool COLOR, bool INC>
__global__ void __launch_bounds__(PR_WARPS * 32, SF_PREP_MINB) k_prep_two_frame(PrepArgs a) {
    pdl_enter();
    __shared__ p64 ring[PR_WARPS * PR_RING];
    const int lane = threadIdx.x & 31;
    const int work = blockIdx.x * PR_WARPS + (threadIdx.x >> 5);
    if (work >= a.nwork) return; // whole warp
    const int strip = work % a.strips, seg = work / a.strips;
    const int X0 = strip * PR_OUT_W - 2 * PR_OUT_LO;
    p64 *ring_sm = ring + (threadIdx.x >> 5) * PR_RING;
    if ((X0 < 0) || (X0 + 63 > a.g.W - 1)) prep_march<COLOR, true, INC>(a, strip, seg, lane, ring_sm);
    else prep_march<COLOR, false, INC>(a, strip, seg, lane, ring_sm);
}

// One outer iteration of the default two-frame loop (niter_inner == 1) in one pass: k_flow_smooth<UPDATE, 1> (flow
// update w += du, psi_h / psi_v) followed by k_prep_two_frame<COLOR, 0>, with the same results bit for bit
template <bool COLOR, bool UPDATE>
__global__ void __launch_bounds__(PR_WARPS * 32, SF_PREP_MINB) k_prep_fused(PrepArgs a) {
    pdl_enter();
    __shared__ p64 ring[PR_WARPS * PR_RING_PSI];
    const int lane = threadIdx.x & 31;
    const int work = blockIdx.x * PR_WARPS + (threadIdx.x >> 5);
    if (work >= a.nwork) return; // whole warp
    const int strip = work % a.strips, seg = work / a.strips;
    const int X0 = strip * PR_OUT_W - 2 * PR_OUT_LO;
    p64 *ring_sm = ring + (threadIdx.x >> 5) * PR_RING_PSI;
    if ((X0 < 0) || (X0 + 63 > a.g.W - 1)) prep_march<COLOR, true, false, true, UPDATE>(a, strip, seg, lane, ring_sm);
    else prep_march<COLOR, false, false, true, UPDATE>(a, strip, seg, lane, ring_sm);
}

// rows per segment: the largest number of (strip, segment) work items that is still ONE wave of resident warps
// (a second, mostly empty wave would double the kernel time), but at least 16 rows (8 warm-up rows per segment)
static int prep_seg_rows(Geom g, int num_sms, int resident_warps_per_sm) {
    const int strips = (g.S + PR_OUT_W - 1) / PR_OUT_W;
    int segs = (num_sms * resident_warps_per_sm) / strips;
    if (segs < 1) segs = 1;
    int rows = (g.H + segs - 1) / segs;
    if (rows < 16) rows = 16;
    return (rows + 3) & ~3;
}

template <void (*KERNEL)(PrepArgs)>
static void launch_march(cudaStream_t st, Geom g, int num_sms, PrepArgs &a) {
    // resident warps per SM (the same on every device of the box: all are sm_100a; relaxed atomics because one host
    // thread per device may get here at the same time)
    static std::atomic<int> resident{0};
    int res = resident.load(std::memory_order_relaxed);
    if (!res) {
        int blocks_per_sm = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, KERNEL, PR_WARPS * 32, 0);
        res = (blocks_per_sm > 0 ? blocks_per_sm : 1) * PR_WARPS;
        resident.store(res, std::memory_order_relaxed);
    }
    a.seg_rows = prep_seg_rows(g, num_sms, res);
    const int segs = (g.H + a.seg_rows - 1) / a.seg_rows;
    a.nwork = a.strips * segs;
    const int blocks = (a.nwork + PR_WARPS - 1) / PR_WARPS;
    launch_pdl(KERNEL, dim3(blocks), dim3(PR_WARPS * 32), 0, st, a);
}
template <bool COLOR, bool INC>
static void launch_prep_variant(cudaStream_t st, Geom g, int num_sms, PrepArgs &a) {
    launch_march<k_prep_two_frame<COLOR, INC>>(st, g, num_sms, a);
}

void launch_prep_fused(cudaStream_t st, Geom g, int num_sms, const float *im1, const float *im2, const float *wx, const float *wy,
                       const float *du, const float *dv, const float *dpsis, float half_alpha, float half_delta_over3,
                       float half_gamma_over3, float *wx_out, float *wy_out, float *ph, float *pv, float *a11, float *a12,
                       float *a22, float *b1, float *b2) {
    PrepArgs a;
    a.g = g;
    a.im1 = im1; a.im2 = im2; a.wx = wx; a.wy = wy; a.du = du; a.dv = dv; a.ph = nullptr; a.pv = nullptr;
    a.a11 = a11; a.a12 = a12; a.a22 = a22; a.b1 = b1; a.b2 = b2;
    a.hd = half_delta_over3; a.hg = half_gamma_over3;
    a.strips = (g.S + PR_OUT_W - 1) / PR_OUT_W;
    a.dpsis = dpsis; a.half_alpha = half_alpha;
    a.ph_out = ph; a.pv_out = pv; a.wx_out = wx_out; a.wy_out = wy_out;
    const bool update = du != nullptr;
    if (half_delta_over3 != 0.0f) {
        if (update) launch_march<k_prep_fused<true, true>>(st, g, num_sms, a);
        else launch_march<k_prep_fused<true, false>>(st, g, num_sms, a);
    } else {
        if (update) launch_march<k_prep_fused<false, true>>(st, g, num_sms, a);
        else launch_march<k_prep_fused<false, false>>(st, g, num_sms, a);
    }
}

void launch_prep_two_frame(cudaStream_t st, Geom g, int num_sms, const float *im1, const float *im2, const float *wx, const float *wy, const float *du, const float *dv, const float *ph, const float *pv,
                           float half_delta_over3, float half_gamma_over3, float *a11, float *a12, float *a22, float *b1,
                           float *b2) {
    PrepArgs a;
    a.g = g;
    a.im1 = im1; a.im2 = im2; a.wx = wx; a.wy = wy; a.du = du; a.dv = dv; a.ph = ph; a.pv = pv;
    a.a11 = a11; a.a12 = a12; a.a22 = a22; a.b1 = b1; a.b2 = b2;
    a.hd = half_delta_over3; a.hg = half_gamma_over3;
    a.strips = (g.S + PR_OUT_W - 1) / PR_OUT_W;
    const bool inc = du != nullptr;
    if (half_delta_over3 != 0.0f) {
        if (inc) launch_prep_variant<true, true>(st, g, num_sms, a);
        else launch_prep_variant<true, false>(st, g, num_sms, a);
    } else {
        if (inc) launch_prep_variant<false, true>(st, g, num_sms, a);
        else launch_prep_variant<false, false>(st, g, num_sms, a);
    }
}

} // namespace sf
