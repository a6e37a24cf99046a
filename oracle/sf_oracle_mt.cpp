/*
 * sf_oracle_mt.cpp -- CPU restatement of the multi-frame, occlusion-aware refinement (Variational_MT).
 * TEST INFRASTRUCTURE ONLY; never linked into or loaded by the product library.
 *
 * Restates, in the reference's evaluation order (scalar loops standing in for its v4sf code, fp32, no FMA):
 *   normalize                              epic_flow_extended/variational_mt.cpp:17-85
 *   Variational_MT::get_derivatives        :87-166
 *   Variational_MT::compute_one_level      :169-493
 *   Variational_MT::variational            :526-784
 *   Variational_AUX_MT::compute_smoothness variational_aux_mt.cpp:18-127 (modes 0, 1)
 *   ...::add_data_and_match                :166-403
 *   ...::add_data_and_match_ref            :408-634 (incl. the copy-paste slips of the un-normalised branch)
 *   ...::compute_dpsis_weight              :673-719
 *   ...::optimizeOcc                       :758-887
 *   penalty_functions/{*}.h                both the scalar (double inside) and the v4sf (float) overloads
 * Third-party arithmetic that is NOT in the reference tree is restated from its published behaviour and is
 * "parity unpinned" by reference tests (there are none): cv::GaussianBlur / cv::resize (pinned to python cv2 4.13,
 * tests/test_oracle_pin.py) and gco-v3.0's expansion (exact binary min-cut, sfo_gridcut.hpp).
 * Pinning: bit-compared against oracle/_ref (the reference's unmodified driver) and tests/golden/mt_*.npz.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "sf_oracle.h"
#include "sfo_gridcut.hpp"

#define SF_MT_MAX_REF 8
extern "C" {
/* layout of sf_mt_params_t (include/slowflow_gpu.h) */
typedef struct sfo_mt_params_s {
    int S, layers; float p_scale; float alpha, gamma, delta; int dataterm, smoothing, one_direction;
    float rho[SF_MT_MAX_REF], omega[SF_MT_MAX_REF];
    int robust_color; float robust_color_eps, robust_color_truncation;
    int robust_grad; float robust_grad_eps, robust_grad_truncation;
    int robust_reg; float robust_reg_eps, robust_reg_truncation;
    int niter_alter, niter_outer, niter_inner, niter_solver, niter_graphc;
    float thres_outer, thres_inner, sor_omega;
    int occlusion_reasoning; float occlusion_penalty, occlusion_alpha;
    int graphcut_int_terms, hbit;
    float img_norm_avg[3], img_norm_std[3];
} sfo_mt_params_t;
}

namespace {

typedef sfo_image_t Img;
typedef sfo_color_image_t CImg;

/* ---------------------------------------------------------------- penalties (penalty_functions/ *.h) */
struct Pen {
    int type; /* 0 quadratic, 1 modified L1, 2 Lorentzian, 3 truncated modified L1, 4 Geman-McClure */
    double eps_d; float eps_f; float trunc;
    Pen(int t, float e, float tr) : type(t), trunc(tr) { const float e2 = e * e; eps_f = e2; eps_d = e2; }
    /* v4sf overloads, per lane */
    float deriv_v(float x) const {
        switch (type) {
        case 0: return 1.0f;
        case 2: return 1.0f / (2.0f * eps_f + x);
        case 4: { float t = eps_f + x; t = t * t; return (eps_f + 2.0f * x) / t; }
        case 3: { float o = 1.0f / (2.0f * sqrtf(x + eps_f)); if (sqrtf(x) > trunc) o = 0.0f; return o; }
        default: return 1.0f / (2.0f * sqrtf(x + eps_f));
        }
    }
    float apply_v(float x) const {
        switch (type) {
        case 0: return x;
        case 2: return (float)log(1 + 0.5 * x / eps_d);
        case 4: return x / ((x + 1.0f) * (x + 1.0f));
        case 3: { float o = sqrtf(x + eps_f); if (sqrtf(x) > trunc) o = sqrtf(trunc + eps_f); return o; }
        default: return sqrtf(x + eps_f);
        }
    }
    /* scalar overloads (double where epsilon_sq is a double member) */
    float deriv_s(float x) const {
        switch (type) {
        case 0: return 1.0f;
        case 2: return (float)(1 / (2 * eps_d + x));
        case 4: { float t = (float)(eps_d + x); t = t * t; return (float)((eps_d + 2 * x) / t); }
        case 3: { if (sqrtf(x) > trunc) return 0.0f; return 1 / (2 * sqrtf(x + eps_f)); }
        default: return (float)(1 / (2 * sqrt(x + eps_d)));
        }
    }
};

const float dnorm = 0.1f * 0.1f;

void deriv5(float t[5]) { const float h1 = -8.0f / 12.0f, h2 = 1.0f / 12.0f; t[0] = h2; t[1] = h1; t[2] = -0.0f; t[3] = -h1; t[4] = -h2; }
void deriv3(float t[3]) { t[0] = -0.5f; t[1] = -0.0f; t[2] = 0.5f; }

void color_conv(CImg *dst, const CImg *src, int horiz, const float *c5) {
    float *dp[3] = {dst->c1, dst->c2, dst->c3}, *sp[3] = {src->c1, src->c2, src->c3};
    for (int ch = 0; ch < 3; ch++) {
        Img d = {src->width, src->height, src->stride, dp[ch]}, s = {src->width, src->height, src->stride, sp[ch]};
        if (horiz) sfo_convolve_horiz(&d, &s, 2, c5); else sfo_convolve_vert(&d, &s, 2, c5);
    }
}

/* mean / temporal difference + 7 convolutions (variational_mt.cpp:112-136 and :138-161) */
void pair_derivs(const CImg *im1, const CImg *im2, CImg *Ix, CImg *Iy, CImg *Iz, CImg *Ixx, CImg *Ixy, CImg *Iyy, CImg *Ixz, CImg *Iyz) {
    float c5[5];
    deriv5(c5);
    CImg *mean = sfo_color_image_new(im1->width, im1->height);
    const size_t n = 3 * (size_t)im1->height * im1->stride;
    for (size_t k = 0; k < n; k++) {
        mean->c1[k] = 0.5f * (im2->c1[k] + im1->c1[k]);
        Iz->c1[k] = im1->c1[k] - im2->c1[k];
    }
    color_conv(Ix, mean, 1, c5);
    color_conv(Iy, mean, 0, c5);
    color_conv(Ixx, Ix, 1, c5);
    color_conv(Ixy, Ix, 0, c5);
    color_conv(Iyy, Iy, 0, c5);
    color_conv(Ixz, Iz, 1, c5);
    color_conv(Iyz, Iz, 0, c5);
    sfo_color_image_delete(mean);
}

struct DerivSet { CImg *Ix, *Iy, *Iz, *Ixx, *Ixy, *Iyy, *Ixz, *Iyz; };
DerivSet new_set(int w, int h) {
    DerivSet d = {sfo_color_image_new(w, h), sfo_color_image_new(w, h), sfo_color_image_new(w, h), sfo_color_image_new(w, h),
                  sfo_color_image_new(w, h), sfo_color_image_new(w, h), sfo_color_image_new(w, h), sfo_color_image_new(w, h)};
    return d;
}
void free_set(DerivSet &d) {
    sfo_color_image_delete(d.Ix); sfo_color_image_delete(d.Iy); sfo_color_image_delete(d.Iz); sfo_color_image_delete(d.Ixx);
    sfo_color_image_delete(d.Ixy); sfo_color_image_delete(d.Iyy); sfo_color_image_delete(d.Ixz); sfo_color_image_delete(d.Iyz);
}

/* warp with the factor == 0 shortcut of variational_aux_mt.cpp:723-728 (mask is NULL whenever factor is 0) */
void warp_mt(CImg *dst, Img *mask, const CImg *src, const Img *wx, const Img *wy, int factor) {
    if (factor == 0) {
        memcpy(dst->c1, src->c1, sizeof(float) * 3 * (size_t)src->stride * src->height);
        return;
    }
    sfo_image_warp(dst, mask, src, wx, wy, factor);
}

/* Variational_MT::get_derivatives (variational_mt.cpp:87-166) */
void get_derivatives(CImg *const *im, const Img *wx, const Img *wy, CImg *ws, CImg *wsp1, Img **mask, DerivSet *succ, DerivSet *toref,
                     int ref, bool one_direction) {
    for (int s = one_direction ? ref : 0; s < 2 * ref; s++) {
        if (s < ref) {
            warp_mt(ws, mask[s], im[s], wx, wy, s - ref);
            warp_mt(wsp1, NULL, im[s + 1], wx, wy, s - ref + 1);
        } else {
            warp_mt(ws, NULL, im[s], wx, wy, s - ref);
            warp_mt(wsp1, mask[s], im[s + 1], wx, wy, s - ref + 1);
        }
        pair_derivs(ws, wsp1, succ[s].Ix, succ[s].Iy, succ[s].Iz, succ[s].Ixx, succ[s].Ixy, succ[s].Iyy, succ[s].Ixz, succ[s].Iyz);
        const CImg *a = (s < ref) ? ws : im[ref], *b = (s < ref) ? im[ref] : wsp1;
        pair_derivs(a, b, toref[s].Ix, toref[s].Iy, toref[s].Iz, toref[s].Ixx, toref[s].Ixy, toref[s].Iyy, toref[s].Ixz, toref[s].Iyz);
    }
}

/* Variational_AUX_MT::compute_smoothness, modes 0 and 1 (variational_aux_mt.cpp:18-92) */
void smoothness_mt(int method, Img *dh, Img *dv, const Img *uu, const Img *vv, const Img *w, float alpha, const Pen &reg) {
    const int W = uu->width, H = uu->height, S = uu->stride;
    float c3[3];
    deriv3(c3);
    Img *ux2 = sfo_image_new(W, H), *uy2 = sfo_image_new(W, H), *vx2 = sfo_image_new(W, H), *vy2 = sfo_image_new(W, H);
    sfo_convolve_horiz(ux2, uu, 1, c3);
    sfo_convolve_horiz(vx2, vv, 1, c3);
    sfo_convolve_vert(uy2, uu, 1, c3);
    sfo_convolve_vert(vy2, vv, 1, c3);
    for (int j = 0; j < H; j++) {
        for (int i = 0; i < W - 1; i++) {
            const size_t o = (size_t)j * S + i;
            float tmp = 0, tmp2 = 0;
            const float tw = w->data[o] + w->data[o + 1];
            if (method == 1) {
                tmp = 0.5f * (uy2->data[o] + uy2->data[o + 1]);
                tmp2 = 0.5f * (vy2->data[o] + vy2->data[o + 1]);
            }
            const float ux1 = uu->data[o + 1] - uu->data[o], vx1 = vv->data[o + 1] - vv->data[o];
            tmp = ux1 * ux1 + tmp * tmp;
            tmp2 = vx1 * vx1 + tmp2 * tmp2;
            tmp = tmp + tmp2;
            dh->data[o] = tw * alpha * reg.deriv_s(tmp);
        }
        for (int i = W - 1; i < S; i++) dh->data[(size_t)j * S + i] = 0.0f;
    }
    for (int j = 0; j < H - 1; j++)
        for (int i = 0; i < W; i++) {
            const size_t o = (size_t)j * S + i;
            float tmp = 0, tmp2 = 0;
            const float tw = w->data[o] + w->data[o + S];
            if (method == 1) {
                tmp = 0.5f * (ux2->data[o] + ux2->data[o + S]);
                tmp2 = 0.5f * (vx2->data[o] + vx2->data[o + S]);
            }
            const float uy1 = uu->data[o + S] - uu->data[o], vy1 = vv->data[o + S] - vv->data[o];
            tmp = uy1 * uy1 + tmp * tmp;
            tmp2 = vy1 * vy1 + tmp2 * tmp2;
            tmp = tmp + tmp2;
            dv->data[o] = tw * alpha * reg.deriv_s(tmp);
        }
    for (int i = 0; i < S; i++) dv->data[(size_t)(H - 1) * S + i] = 0.0f;
    sfo_image_delete(ux2); sfo_image_delete(uy2); sfo_image_delete(vx2); sfo_image_delete(vy2);
}

struct Sys { Img *a11, *a12, *a22, *b1, *b2; };

/* add_data_and_match (variational_aux_mt.cpp:166-403) */
void add_succ(Sys &A, const Img *mask, const Img *du, const Img *dv, const DerivSet &D, const CImg *cw, float delta_over3,
              float gamma_over3, float s, bool dt_norm, const Pen &pc, const Pen &pg) {
    const size_t n = (size_t)du->height * du->stride, P = n;
    const float f = s, f1 = s + 1;
    for (size_t k = 0; k < n; k++) {
        const float u = du->data[k], v = dv->data[k], m = mask->data[k];
        float a11 = A.a11->data[k], a12 = A.a12->data[k], a22 = A.a22->data[k], b1 = A.b1->data[k], b2 = A.b2->data[k];
        const float w[3] = {cw->c1[k], cw->c2[k], cw->c3[k]};
        if (delta_over3) {
            float r[3], gx[3], gy[3];
            for (int c = 0; c < 3; c++) {
                const float ix = D.Ix->c1[k + c * P], iy = D.Iy->c1[k + c * P], iz = D.Iz->c1[k + c * P];
                r[c] = w[c] * (iz + ix * f * u + iy * f * v - ix * f1 * u - iy * f1 * v);
                gx[c] = f * ix - f1 * ix;
                gy[c] = f * iy - f1 * iy;
            }
            if (!dt_norm) {
                const float t = m * delta_over3 * pc.deriv_v(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
                for (int c = 0; c < 3; c++) {
                    const float iz = D.Iz->c1[k + c * P], g = t * w[c];
                    a11 += g * gx[c] * gx[c]; a12 += g * gx[c] * gy[c]; a22 += g * gy[c] * gy[c];
                    b1 -= g * iz * gx[c]; b2 -= g * iz * gy[c];
                }
            } else {
                float nn[3], g[3];
                for (int c = 0; c < 3; c++) nn[c] = gx[c] * gx[c] + gy[c] * gy[c] + dnorm;
                const float t = m * delta_over3 * pc.deriv_v(r[0] * r[0] / nn[0] + r[1] * r[1] / nn[1] + r[2] * r[2] / nn[2]);
                g[2] = t / nn[2]; g[1] = t / nn[1]; g[0] = t / nn[0];
                for (int c = 0; c < 3; c++) {
                    const float iz = D.Iz->c1[k + c * P], gg = g[c] * w[c];
                    a11 += gg * gx[c] * gx[c]; a12 += gg * gx[c] * gy[c]; a22 += gg * gy[c] * gy[c];
                    b1 -= gg * iz * gx[c]; b2 -= gg * iz * gy[c];
                }
            }
        }
        float rx[3], ry[3], gxx[3], gyy[3], gxy[3];
        for (int c = 0; c < 3; c++) {
            const float ixx = D.Ixx->c1[k + c * P], ixy = D.Ixy->c1[k + c * P], iyy = D.Iyy->c1[k + c * P];
            const float ixz = D.Ixz->c1[k + c * P], iyz = D.Iyz->c1[k + c * P];
            rx[c] = w[c] * (ixz + ixx * f * u + ixy * f * v - ixx * f1 * u - ixy * f1 * v);
            ry[c] = w[c] * (iyz + ixy * f * u + iyy * f * v - ixy * f1 * u - iyy * f1 * v);
            gxx[c] = f * ixx - f1 * ixx;
            gyy[c] = f * iyy - f1 * iyy;
            gxy[c] = f * ixy - f1 * ixy;
        }
        if (!dt_norm) {
            const float t = m * gamma_over3 * pg.deriv_v(rx[0] * rx[0] + ry[0] * ry[0] + rx[1] * rx[1] + ry[1] * ry[1] + rx[2] * rx[2] + ry[2] * ry[2]);
            for (int c = 0; c < 3; c++) {
                const float ixz = D.Ixz->c1[k + c * P], iyz = D.Iyz->c1[k + c * P], g = t * w[c];
                a11 += g * gxx[c] * gxx[c] + g * gxy[c] * gxy[c];
                a12 += g * gxx[c] * gxy[c] + g * gxy[c] * gyy[c];
                a22 += g * gyy[c] * gyy[c] + g * gxy[c] * gxy[c];
                b1 -= g * ixz * gxx[c] + g * iyz * gxy[c];
                b2 -= g * iyz * gyy[c] + g * ixz * gxy[c];
            }
        } else {
            float nx[3], ny[3], g1[3], g2[3];
            for (int c = 0; c < 3; c++) {
                nx[c] = gxx[c] * gxx[c] + gxy[c] * gxy[c] + dnorm;
                ny[c] = gyy[c] * gyy[c] + gxy[c] * gxy[c] + dnorm;
            }
            const float t = m * gamma_over3 * pg.deriv_v(rx[0] * rx[0] / nx[0] + ry[0] * ry[0] / ny[0] + rx[1] * rx[1] / nx[1] +
                                                         ry[1] * ry[1] / ny[1] + rx[2] * rx[2] / nx[2] + ry[2] * ry[2] / ny[2]);
            g2[2] = t / ny[2]; g1[2] = t / nx[2]; g2[1] = t / ny[1]; g1[1] = t / nx[1]; g2[0] = t / ny[0]; g1[0] = t / nx[0];
            for (int c = 0; c < 3; c++) {
                const float ixz = D.Ixz->c1[k + c * P], iyz = D.Iyz->c1[k + c * P];
                const float h1 = g1[c] * w[c], h2 = g2[c] * w[c];
                a11 += h1 * gxx[c] * gxx[c] + h2 * gxy[c] * gxy[c];
                a12 += h1 * gxx[c] * gxy[c] + h2 * gxy[c] * gyy[c];
                a22 += h2 * gyy[c] * gyy[c] + h1 * gxy[c] * gxy[c];
                b1 -= h1 * ixz * gxx[c] + h2 * iyz * gxy[c];
                b2 -= h2 * iyz * gyy[c] + h1 * ixz * gxy[c];
            }
        }
        A.a11->data[k] = a11; A.a12->data[k] = a12; A.a22->data[k] = a22; A.b1->data[k] = b1; A.b2->data[k] = b2;
    }
}

/* add_data_and_match_ref (variational_aux_mt.cpp:408-634) */
void add_ref(Sys &A, const Img *mask, const Img *du, const Img *dv, const DerivSet &D, const CImg *cw, float delta_over3,
             float gamma_over3, float s, bool dt_norm, const Pen &pc, const Pen &pg) {
    const size_t n = (size_t)du->height * du->stride, P = n;
    float f = s;
    const float fsq = f * f;
    if (s >= 0) f = -f;
    for (size_t k = 0; k < n; k++) {
        const float u = du->data[k], v = dv->data[k], m = mask->data[k];
        float a11 = A.a11->data[k], a12 = A.a12->data[k], a22 = A.a22->data[k], b1 = A.b1->data[k], b2 = A.b2->data[k];
        const float w[3] = {cw->c1[k], cw->c2[k], cw->c3[k]};
        if (delta_over3) {
            float r[3];
            for (int c = 0; c < 3; c++) {
                const float ix = D.Ix->c1[k + c * P], iy = D.Iy->c1[k + c * P], iz = D.Iz->c1[k + c * P];
                r[c] = w[c] * (iz + ix * f * u + iy * f * v);
            }
            if (!dt_norm) {
                float t = m * delta_over3 * pc.deriv_v(r[0] * r[0] / fsq + r[1] * r[1] / fsq + r[2] * r[2] / fsq);
                t /= fsq;
                for (int c = 0; c < 3; c++) {
                    const float ix = D.Ix->c1[k + c * P], iy = D.Iy->c1[k + c * P], iz = D.Iz->c1[k + c * P];
                    float g = (c == 0) ? t * w[0] * f : t * f * w[c];
                    b1 -= g * iz * ix; b2 -= g * iz * iy;
                    g = (c == 2) ? t * f : g * f; /* :469 as written */
                    a11 += g * ix * ix; a12 += g * ix * iy; a22 += g * iy * iy;
                }
            } else {
                float nn[3], g[3];
                for (int c = 0; c < 3; c++) {
                    const float ix = D.Ix->c1[k + c * P], iy = D.Iy->c1[k + c * P];
                    nn[c] = fsq * ix * ix + fsq * iy * iy + dnorm;
                }
                const float t = m * delta_over3 * pc.deriv_v(r[0] * r[0] / nn[0] + r[1] * r[1] / nn[1] + r[2] * r[2] / nn[2]);
                g[2] = t / nn[2]; g[1] = t / nn[1]; g[0] = t / nn[0];
                for (int c = 0; c < 3; c++) {
                    const float ix = D.Ix->c1[k + c * P], iy = D.Iy->c1[k + c * P], iz = D.Iz->c1[k + c * P];
                    float gg = g[c] * w[c] * f;
                    b1 -= gg * iz * ix; b2 -= gg * iz * iy;
                    gg = gg * f;
                    a11 += gg * ix * ix; a12 += gg * ix * iy; a22 += gg * iy * iy;
                }
            }
        }
        float rx[3], ry[3];
        for (int c = 0; c < 3; c++) {
            const float ixx = D.Ixx->c1[k + c * P], ixy = D.Ixy->c1[k + c * P], iyy = D.Iyy->c1[k + c * P];
            rx[c] = w[c] * (D.Ixz->c1[k + c * P] + ixx * f * u + ixy * f * v);
            ry[c] = w[c] * (D.Iyz->c1[k + c * P] + ixy * f * u + iyy * f * v);
        }
        if (!dt_norm) {
            float t = m * gamma_over3 * pg.deriv_v(rx[0] * rx[0] / fsq + ry[0] * ry[0] / fsq + rx[1] * rx[1] / fsq + ry[1] * ry[1] / fsq +
                                                   rx[2] * rx[2] / fsq + ry[2] * ry[2] / fsq);
            t /= fsq;
            for (int c = 0; c < 3; c++) {
                const float ixx = D.Ixx->c1[k + c * P], ixy = D.Ixy->c1[k + c * P], iyy = D.Iyy->c1[k + c * P];
                const float ixz = D.Ixz->c1[k + c * P], iyz = D.Iyz->c1[k + c * P];
                float g = t * w[c] * f;
                b1 -= g * ixx * ixz + g * ixy * iyz;
                b2 -= g * iyy * iyz + g * ixy * ixz;
                g = g * f;
                if (c == 0) { /* :528-530 as written: extra factorsq on channel 1 */
                    a11 += g * fsq * ixx * ixx + g * fsq * ixy * ixy;
                    a12 += g * fsq * ixx * ixy + g * fsq * ixy * iyy;
                    a22 += g * fsq * iyy * iyy + g * fsq * ixy * ixy;
                } else {
                    a11 += g * ixx * ixx + g * ixy * ixy;
                    a12 += g * ixx * ixy + g * ixy * iyy;
                    a22 += g * iyy * iyy + g * ixy * ixy;
                }
            }
        } else {
            float nx[3], ny[3], g1[3], g2[3];
            for (int c = 0; c < 3; c++) {
                const float ixx = D.Ixx->c1[k + c * P], ixy = D.Ixy->c1[k + c * P], iyy = D.Iyy->c1[k + c * P];
                nx[c] = fsq * ixx * ixx + fsq * ixy * ixy + dnorm;
                ny[c] = fsq * iyy * iyy + fsq * ixy * ixy + dnorm;
            }
            const float t = m * gamma_over3 * pg.deriv_v(rx[0] * rx[0] / nx[0] + ry[0] * ry[0] / ny[0] + rx[1] * rx[1] / nx[1] +
                                                         ry[1] * ry[1] / ny[1] + rx[2] * rx[2] / nx[2] + ry[2] * ry[2] / ny[2]);
            g2[2] = t / ny[2]; g1[2] = t / nx[2]; g2[1] = t / ny[1]; g1[1] = t / nx[1]; g2[0] = t / ny[0]; g1[0] = t / nx[0];
            for (int c = 0; c < 3; c++) {
                const float ixx = D.Ixx->c1[k + c * P], ixy = D.Ixy->c1[k + c * P], iyy = D.Iyy->c1[k + c * P];
                const float ixz = D.Ixz->c1[k + c * P], iyz = D.Iyz->c1[k + c * P];
                float h1 = g1[c] * w[c] * f, h2 = g2[c] * w[c] * f;
                b1 -= h1 * ixx * ixz + h2 * ixy * iyz;
                b2 -= h2 * iyy * iyz + h1 * ixy * ixz;
                h1 = h1 * f; h2 = h2 * f;
                a11 += h1 * ixx * ixx + h2 * ixy * ixy;
                a12 += h1 * ixx * ixy + h2 * ixy * iyy;
                a22 += h2 * iyy * iyy + h1 * ixy * ixy;
            }
        }
        A.a11->data[k] = a11; A.a12->data[k] = a12; A.a22->data[k] = a22; A.b1->data[k] = b1; A.b2->data[k] = b2;
    }
}

/* compute_dpsis_weight, 7-out-argument overload (variational_aux_mt.cpp:673-719); only `lum` is used downstream */
void dpsis_mt(const CImg *im, Img *lum, float coef, const float avg[3], const float sd[3], bool hbit) {
    const int W = im->width, H = im->height;
    float c5[5];
    deriv5(c5);
    Img *lx = sfo_image_new(W, H), *ly = sfo_image_new(W, H);
    const size_t n = (size_t)im->height * im->stride;
    const float div = hbit ? 65535.0f : 255.0f;
    for (size_t k = 0; k < n; k++)
        lum->data[k] = (0.299f * (im->c1[k] * sd[0] + avg[0]) + 0.587f * (im->c2[k] * sd[1] + avg[1]) + 0.114f * (im->c3[k] * sd[2] + avg[2])) / div;
    sfo_convolve_horiz(lx, lum, 2, c5);
    sfo_convolve_vert(ly, lum, 2, c5);
    for (size_t k = 0; k < n; k++)
        lum->data[k] = 0.5f * expf(-coef * sqrtf(lx->data[k] * lx->data[k] + ly->data[k] * ly->data[k]));
    sfo_image_delete(lx);
    sfo_image_delete(ly);
}

/* the colour, gradient and regularisation penalties of a parameter set (select_robust_function,
 * variational_aux_mt.cpp:889-926); robust_grad < 0 reuses the colour penalty */
struct Pens {
    Pen pc, pg, preg;
    explicit Pens(const sfo_mt_params_t *p)
        : pc(p->robust_color, p->robust_color_eps, p->robust_color_truncation),
          pg(p->robust_grad >= 0 ? Pen(p->robust_grad, p->robust_grad_eps, p->robust_grad_truncation) : pc),
          preg(p->robust_reg, p->robust_reg_eps, p->robust_reg_truncation) {}
};

/* data costs of the two occlusion labels (variational_aux_mt.cpp:786-848) from the raw masks and the derivatives of
 * get_derivatives: d0 / d1 at the pixels of the occ plane's geometry */
void occ_costs(Img *d0, Img *d1, Img *const *mask, const DerivSet *succ, const DerivSet *toref, int ref, const float *rho, const float *omega,
               float delta_over3, float gamma_over3, float penalty, const Pen &pc, const Pen &pg) {
    const int W = d0->width, H = d0->height, S = d0->stride;
    const size_t P = (size_t)S * H;
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            const size_t k = (size_t)y * S + x;
            float e[2] = {0, 0}, nrm[2] = {0, 0};
            for (int s = 0; s < 2 * ref; s++) {
                const int idx = std::max(ref - s - 1, s - ref);
                const float m = mask[s]->data[k];
                auto sq3 = [&](const CImg *I) { return I->c1[k] * I->c1[k] + I->c1[k + P] * I->c1[k + P] + I->c1[k + 2 * P] * I->c1[k + 2 * P]; };
                auto sq6 = [&](const CImg *X, const CImg *Y) {
                    return X->c1[k] * X->c1[k] + X->c1[k + P] * X->c1[k + P] + X->c1[k + 2 * P] * X->c1[k + 2 * P] + Y->c1[k] * Y->c1[k] +
                           Y->c1[k + P] * Y->c1[k + P] + Y->c1[k + 2 * P] * Y->c1[k + 2 * P];
                };
                float term = rho[idx] * delta_over3 * m * pc.apply_v(sq3(succ[s].Iz));
                term += rho[idx] * gamma_over3 * m * pg.apply_v(sq6(succ[s].Ixz, succ[s].Iyz));
                term += omega[idx] * delta_over3 * m * pc.apply_v(sq3(toref[s].Iz));
                term += omega[idx] * gamma_over3 * m * pg.apply_v(sq6(toref[s].Ixz, toref[s].Iyz));
                const int l = (s >= ref) ? 0 : 1;
                e[l] += term;
                nrm[l] += m * (rho[idx] + rho[idx] + omega[idx] + omega[idx]);
            }
            float d[2];
            for (int l = 0; l < 2; l++) {
                if (nrm[l] == 0) nrm[l] = 1;
                d[l] = 0.01f * e[l] / nrm[l] + penalty * l;
            }
            d0->data[k] = d[0];
            d1->data[k] = d[1];
        }
}

/* optimizeOcc (variational_aux_mt.cpp:758-887) with the exact binary min-cut standing in for gco's expansion */
void optimize_occ(Img *occ, Img **mask, DerivSet *succ, DerivSet *toref, int ref, const float *rho, const float *omega, float delta_over3,
                  float gamma_over3, float penalty, float alpha, const Pen &pc, const Pen &pg, bool int_terms) {
    const int W = occ->width, H = occ->height, S = occ->stride;
    Img *d0 = sfo_image_new(W, H), *d1 = sfo_image_new(W, H);
    occ_costs(d0, d1, mask, succ, toref, ref, rho, omega, delta_over3, gamma_over3, penalty, pc, pg);
    sfo::GridCut gc(W, H);
    auto q = [&](double e) -> int64_t { return (int64_t)llround((int_terms ? (double)(int)e : e) * 16777216.0); };
    const int64_t pair = q((double)alpha);
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            const size_t k = (size_t)y * S + x;
            const int p = y * W + x;
            gc.set_terminal(p, q((double)d1->data[k]), q((double)d0->data[k]));
            if (x + 1 < W) gc.set_edge_right(p, pair);
            if (y + 1 < H) gc.set_edge_down(p, pair);
        }
    sfo_image_delete(d0);
    sfo_image_delete(d1);
    gc.maxflow();
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) occ->data[(size_t)y * S + x] = (float)(2 * gc.label(y * W + x) - 1);
}

/* the occlusion / window factor of variational_mt.cpp:293-320, applied in place to the raw masks of get_derivatives */
void occ_factor(Img *const *mask, const Img *occ, const sfo_mt_params_t *p) {
    const int ref = p->S - 1;
    const bool one_direction = p->one_direction != 0;
    const size_t n = (size_t)occ->stride * occ->height;
    float data_norm = 0;
    for (int s = 0; s < ref; s++) data_norm += p->rho[s] + p->omega[s];
    for (size_t k = 0; k < n; k++) {
        const float oc = occ->data[k];
        const float fac = (1 + ((oc == 0) ? 1.0f : 0.0f)) * data_norm;
        const float backward = ((oc >= 0) ? 1.0f : 0.0f) / fac, forward = ((oc <= 0) ? 1.0f : 0.0f) / fac;
        for (int s = one_direction ? ref : 0; s < 2 * ref; s++)
            mask[s]->data[k] = (s < ref) ? (1.0f * backward * mask[s]->data[k]) : (1.0f * forward * mask[s]->data[k]);
    }
}

/* one linearisation up to the SOR (variational_mt.cpp:333-365): smoothness weights of (uu, vv), every data term of
 * :343-361 at the increment (du, dv) on the factored masks, b -= div(psi grad uu), b -= div(psi grad vv).  The blocks are
 * left as sor_coupled takes them (not inverted). */
void assemble_system(Sys &A, Img *sh, Img *sv, Img *const *mask, const Img *du, const Img *dv, const DerivSet *succ, const DerivSet *toref,
                     const Img *uu, const Img *vv, const Img *dpsis, const CImg *cw, const sfo_mt_params_t *p, const Pens &pen) {
    const int ref = p->S - 1;
    const size_t n = (size_t)uu->stride * uu->height;
    const bool one_direction = p->one_direction != 0, dt_norm = p->dataterm != 0;
    const float gamma_over3 = p->gamma / 3.0f, delta_over3 = p->delta / 3.0f;
    smoothness_mt(p->smoothing, sh, sv, uu, vv, dpsis, p->alpha, pen.preg);
    memset(A.a11->data, 0, n * sizeof(float)); memset(A.a12->data, 0, n * sizeof(float)); memset(A.a22->data, 0, n * sizeof(float));
    memset(A.b1->data, 0, n * sizeof(float)); memset(A.b2->data, 0, n * sizeof(float));
    for (int s = 0; s < ref; s++) { /* :343-361 */
        if (!one_direction) {
            if (p->rho[ref - 1 - s] > 0)
                add_succ(A, mask[s], du, dv, succ[s], cw, p->rho[ref - 1 - s] * delta_over3, p->rho[ref - 1 - s] * gamma_over3, (float)(s - ref), dt_norm, pen.pc, pen.pg);
            if (p->omega[ref - 1 - s] > 0)
                add_ref(A, mask[s], du, dv, toref[s], cw, p->omega[ref - 1 - s] * delta_over3, p->omega[ref - 1 - s] * gamma_over3, (float)(s - ref), dt_norm, pen.pc, pen.pg);
        }
        if (p->rho[s] > 0)
            add_succ(A, mask[ref + s], du, dv, succ[ref + s], cw, p->rho[s] * delta_over3, p->rho[s] * gamma_over3, (float)s, dt_norm, pen.pc, pen.pg);
        if (p->omega[s] > 0)
            add_ref(A, mask[ref + s], du, dv, toref[ref + s], cw, p->omega[s] * delta_over3, p->omega[s] * gamma_over3, (float)(s + 1), dt_norm, pen.pc, pen.pg);
    }
    sfo_sub_laplacian(A.b1, uu, sh, sv);
    sfo_sub_laplacian(A.b2, vv, sh, sv);
}

/* the per-frame planes of one level's get_derivatives */
struct LevelPlanes {
    std::vector<Img *> mask;
    std::vector<DerivSet> succ, toref;
    CImg *ws, *wsp1;
    LevelPlanes(int W, int H, int ref) : mask(2 * ref), succ(2 * ref), toref(2 * ref) {
        for (int s = 0; s < 2 * ref; s++) { mask[s] = sfo_image_new(W, H); succ[s] = new_set(W, H); toref[s] = new_set(W, H); }
        ws = sfo_color_image_new(W, H);
        wsp1 = sfo_color_image_new(W, H);
    }
    ~LevelPlanes() {
        sfo_color_image_delete(ws); sfo_color_image_delete(wsp1);
        for (size_t s = 0; s < mask.size(); s++) { sfo_image_delete(mask[s]); free_set(succ[s]); free_set(toref[s]); }
    }
    void derivatives(CImg *const *im, const Img *wx, const Img *wy, int ref, bool one_direction) {
        get_derivatives(im, wx, wy, ws, wsp1, mask.data(), succ.data(), toref.data(), ref, one_direction);
    }
};

struct LevelOut { float cx, cy; int outer_its, gco_calls; };

/* Variational_MT::compute_one_level (variational_mt.cpp:169-493) */
LevelOut compute_one_level(Img *wx, Img *wy, CImg *const *im, const sfo_mt_params_t *p, const CImg *cw, Img *occ_out, int sor_mode,
                           const Pens &pen) {
    const int W = wx->width, H = wx->height, S = wx->stride, ref = p->S - 1;
    const size_t n = (size_t)S * H;
    const bool one_direction = p->one_direction != 0;
    const float gamma_over3 = p->gamma / 3.0f, delta_over3 = p->delta / 3.0f;
    Img *du = sfo_image_new(W, H), *dv = sfo_image_new(W, H), *odu = sfo_image_new(W, H), *odv = sfo_image_new(W, H),
        *sh = sfo_image_new(W, H), *sv = sfo_image_new(W, H), *uu = sfo_image_new(W, H), *vv = sfo_image_new(W, H);
    Sys A = {sfo_image_new(W, H), sfo_image_new(W, H), sfo_image_new(W, H), sfo_image_new(W, H), sfo_image_new(W, H)};
    LevelPlanes lp(W, H, ref);
    Img *occ = sfo_image_new(W, H);
    if (one_direction || p->occlusion_reasoning) std::fill_n(occ->data, n, -1.0f);
    Img *dpsis = sfo_image_new(W, H);
    dpsis_mt(im[ref], dpsis, 5.0f, p->img_norm_avg, p->img_norm_std, p->hbit != 0);
    memcpy(uu->data, wx->data, n * sizeof(float));
    memcpy(vv->data, wy->data, n * sizeof(float));
    LevelOut out = {0, 0, 0, 0};

    for (int alter = 0; alter < p->niter_alter; alter++) {
        lp.derivatives(im, wx, wy, ref, one_direction);
        if (alter > 0 && p->occlusion_reasoning && !one_direction) {
            optimize_occ(occ, lp.mask.data(), lp.succ.data(), lp.toref.data(), ref, p->rho, p->omega, delta_over3, gamma_over3,
                         p->occlusion_penalty, p->occlusion_alpha, pen.pc, pen.pg, p->graphcut_int_terms != 0);
            out.gco_calls++;
        }
        for (int outer = 0; outer < p->niter_outer; outer++) {
            if (outer > 0) lp.derivatives(im, wx, wy, ref, one_direction);
            out.outer_its++;
            occ_factor(lp.mask.data(), occ, p);
            memset(du->data, 0, n * sizeof(float));
            memset(dv->data, 0, n * sizeof(float));
            for (int inner = 0; inner < p->niter_inner; inner++) {
                memcpy(odu->data, du->data, n * sizeof(float));
                memcpy(odv->data, dv->data, n * sizeof(float));
                assemble_system(A, sh, sv, lp.mask.data(), du, dv, lp.succ.data(), lp.toref.data(), uu, vv, dpsis, cw, p, pen);
                sfo_sor_coupled(du, dv, A.a11, A.a12, A.a22, A.b1, A.b2, sh, sv, p->niter_solver, p->sor_omega, sor_mode);
                float ch_du = 0, ch_dv = 0; /* :376-402: float accumulators, |.| of each group of 4 summed left to right in float */
                for (int j = 0; j < H; j++)
                    for (int i = W; i < S; i++) { du->data[(size_t)j * S + i] = 0; dv->data[(size_t)j * S + i] = 0; }
                for (size_t k = 0; k < n; k += 4) {
                    float a = fabsf(odu->data[k] - du->data[k]), b = fabsf(odv->data[k] - dv->data[k]);
                    for (int t = 1; t < 4; t++) {
                        a = a + fabsf(odu->data[k + t] - du->data[k + t]);
                        b = b + fabsf(odv->data[k + t] - dv->data[k + t]);
                    }
                    ch_du += a;
                    ch_dv += b;
                    for (int t = 0; t < 4; t++) {
                        uu->data[k + t] = wx->data[k + t] + du->data[k + t];
                        vv->data[k + t] = wy->data[k + t] + dv->data[k + t];
                    }
                }
                ch_du /= (H * W);
                ch_dv /= (H * W);
                if (std::max(ch_du, ch_dv) < p->thres_inner) break;
            }
            float cx = 0, cy = 0; /* :412-429 */
            for (size_t k = 0; k < n; k += 4) {
                float a = fabsf(uu->data[k] - wx->data[k]), b = fabsf(vv->data[k] - wy->data[k]);
                for (int t = 1; t < 4; t++) {
                    a = a + fabsf(uu->data[k + t] - wx->data[k + t]);
                    b = b + fabsf(vv->data[k + t] - wy->data[k + t]);
                }
                cx += a;
                cy += b;
            }
            cx /= (H * W);
            cy /= (H * W);
            memcpy(wx->data, uu->data, n * sizeof(float));
            memcpy(wy->data, vv->data, n * sizeof(float));
            out.cx = cx;
            out.cy = cy;
            if (std::max(cx, cy) < p->thres_outer) break;
        }
    }
    if (occ_out && occ_out->width == W && occ_out->height == H) memcpy(occ_out->data, occ->data, n * sizeof(float));
    sfo_image_delete(du); sfo_image_delete(dv); sfo_image_delete(odu); sfo_image_delete(odv); sfo_image_delete(sh); sfo_image_delete(sv);
    sfo_image_delete(uu); sfo_image_delete(vv); sfo_image_delete(A.a11); sfo_image_delete(A.a12); sfo_image_delete(A.a22);
    sfo_image_delete(A.b1); sfo_image_delete(A.b2); sfo_image_delete(dpsis); sfo_image_delete(occ);
    return out;
}

/* ---------------------------------------------------------------- cv::GaussianBlur / cv::resize restated (SURVEY A.8) */
inline int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

void gaussian_blur(const float *src, float *dst, int R, int C, int pitch, double sigma) { /* one plane, replicate border */
    const int n = ((int)lrint(sigma * 8 + 1)) | 1, r = n / 2;
    std::vector<double> t(n);
    std::vector<float> k(n);
    double sum = 0;
    for (int i = 0; i < n; i++) { const double x = i - (n - 1) * 0.5; t[i] = exp(-0.5 / (sigma * sigma) * x * x); sum += t[i]; }
    for (int i = 0; i < n; i++) k[i] = (float)(t[i] / sum);
    std::vector<float> tmp((size_t)R * C);
    for (int i = 0; i < R; i++)
        for (int j = 0; j < C; j++) {
            float acc = k[r] * src[(size_t)i * pitch + j];
            for (int q = 1; q <= r; q++) acc += k[r + q] * (src[(size_t)i * pitch + clampi(j - q, 0, C - 1)] + src[(size_t)i * pitch + clampi(j + q, 0, C - 1)]);
            tmp[(size_t)i * C + j] = acc;
        }
    for (int i = 0; i < R; i++)
        for (int j = 0; j < C; j++) {
            float acc = k[r] * tmp[(size_t)i * C + j];
            for (int q = 1; q <= r; q++) acc += k[r + q] * (tmp[(size_t)clampi(i - q, 0, R - 1) * C + j] + tmp[(size_t)clampi(i + q, 0, R - 1) * C + j]);
            dst[(size_t)i * pitch + j] = acc;
        }
}

void resize_linear(const float *src, int sr, int sc, int spitch, float *dst, int dr, int dc, int dpitch) {
    const double scale_x = (double)sc / dc, scale_y = (double)sr / dr;
    for (int y = 0; y < dr; y++) {
        float fy = (float)((y + 0.5) * scale_y - 0.5);
        int sy = (int)floorf(fy);
        fy -= sy;
        if (sy < 0) { sy = 0; fy = 0; }
        if (sy >= sr - 1) { sy = sr - 1; fy = 0; }
        const int y1 = std::min(sy + 1, sr - 1);
        const float b1 = fy, b0 = 1.f - fy;
        for (int x = 0; x < dc; x++) {
            float fx = (float)((x + 0.5) * scale_x - 0.5);
            int sx = (int)floorf(fx);
            fx -= sx;
            if (sx < 0) { sx = 0; fx = 0; }
            if (sx >= sc - 1) { sx = sc - 1; fx = 0; }
            const int x1 = std::min(sx + 1, sc - 1);
            const float a1 = fx, a0 = 1.f - fx;
            const float r0 = src[(size_t)sy * spitch + sx] * a0 + src[(size_t)sy * spitch + x1] * a1;
            const float r1 = src[(size_t)y1 * spitch + sx] * a0 + src[(size_t)y1 * spitch + x1] * a1;
            dst[(size_t)y * dpitch + x] = r0 * b0 + r1 * b1;
        }
    }
}

Img *resize_flow(const Img *src, int w, int h, float mul) { /* resize + image_mul_scalar (variational_mt.cpp:667-680, 703-717) */
    Img *d = sfo_image_new(w, h);
    resize_linear(src->data, src->height, src->width, src->stride, d->data, h, w, d->stride);
    const size_t n = (size_t)d->stride * h;
    for (size_t k = 0; k < n; k++) d->data[k] *= mul;
    return d;
}

} // namespace

extern "C" {

/* frame pre-scale of slow_flow.cpp:538-542: GaussianBlur(sigma = 1/sqrt(2*scale), BORDER_REPLICATE) + resize(Size(0,0), scale,
 * scale, INTER_LINEAR) on a CV_32F image.  cv::resize by factor: dsize = cvRound(src*f) and the coordinate map uses 1/f
 * (not the ratio of the rounded sizes) -- pinned to python cv2 in tests/test_oracle_pin_mt.py. */
int sfo_prescale_size(int width, int height, float scale, int *ow, int *oh) {
    *ow = (int)lrint((double)width * (double)scale);
    *oh = (int)lrint((double)height * (double)scale);
    return (*ow > 0 && *oh > 0) ? 0 : 1;
}
int sfo_prescale(sfo_color_image_t *dst, const sfo_color_image_t *src, float scale) {
    const double sigma = 1.0 / sqrt((double)(2.0f * scale));
    const double inv = 1.0 / (double)scale;
    const size_t Ps = (size_t)src->stride * src->height, Pd = (size_t)dst->stride * dst->height;
    std::vector<float> blur(Ps);
    for (int c = 0; c < 3; c++) {
        gaussian_blur(src->c1 + c * Ps, blur.data(), src->height, src->width, src->stride, sigma);
        float *d = dst->c1 + c * Pd;
        for (int y = 0; y < dst->height; y++) {
            float fy = (float)((y + 0.5) * inv - 0.5);
            int sy = (int)floorf(fy);
            fy -= sy;
            if (sy < 0) { sy = 0; fy = 0; }
            if (sy >= src->height - 1) { sy = src->height - 1; fy = 0; }
            const int y1 = std::min(sy + 1, src->height - 1);
            for (int x = 0; x < dst->width; x++) {
                float fx = (float)((x + 0.5) * inv - 0.5);
                int sx = (int)floorf(fx);
                fx -= sx;
                if (sx < 0) { sx = 0; fx = 0; }
                if (sx >= src->width - 1) { sx = src->width - 1; fx = 0; }
                const int x1 = std::min(sx + 1, src->width - 1);
                const float a1 = fx, a0 = 1.f - fx, b1 = fy, b0 = 1.f - fy;
                const float r0 = blur[(size_t)sy * src->stride + sx] * a0 + blur[(size_t)sy * src->stride + x1] * a1;
                const float r1 = blur[(size_t)y1 * src->stride + sx] * a0 + blur[(size_t)y1 * src->stride + x1] * a1;
                d[(size_t)y * dst->stride + x] = r0 * b0 + r1 * b1;
            }
        }
    }
    return 0;
}

/* rawWeighting (utils/utils.cpp:1336-1374): channel weights of a Bayer mosaic, red site at (red_x, red_y) */
int sfo_raw_weighting(sfo_color_image_t *weights, int red_x, int red_y, float weight) {
    weight = (float)fmin(fmax(weight, 0.0), 3.0);
    float *R = weights->c1, *G = weights->c2, *B = weights->c3;
    for (int x = 0; x < weights->width; x++)
        for (int y = 0; y < weights->height; y++) {
            const size_t o = (size_t)y * weights->stride + x;
            const float other = (float)(0.5 * (3 - weight));
            if ((y + (1 - red_y)) % 2 == 0) { /* blue row */
                if ((red_y == 1 && (x + (1 - red_x)) % 2 == 0) || (red_y == 0 && (x + red_x) % 2 == 0)) { R[o] = other; G[o] = weight; B[o] = other; }
                else { R[o] = other; G[o] = other; B[o] = weight; }
            } else { /* red row */
                if ((red_y == 0 && (x + (1 - red_x)) % 2 == 0) || (red_y == 1 && (x + red_x) % 2 == 0)) { R[o] = other; G[o] = weight; B[o] = other; }
                else { R[o] = weight; G[o] = other; B[o] = other; }
            }
        }
    return 0;
}

/* labelling step of optimizeOcc alone (variational_aux_mt.cpp:851-881) on dense w*h cost arrays: the checker of the
 * product's sfgpu_grid_mincut */
int sfo_mincut(int w, int h, const float *d0, const float *d1, float alpha, int int_terms, int *labels) {
    auto q = [&](double e) -> int64_t { return (int64_t)llround((int_terms ? (double)(int)e : e) * 16777216.0); };
    sfo::GridCut gc(w, h);
    const int64_t pair = q((double)alpha);
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            const int p = y * w + x;
            gc.set_terminal(p, q((double)d1[p]), q((double)d0[p]));
            if (x + 1 < w) gc.set_edge_right(p, pair);
            if (y + 1 < h) gc.set_edge_down(p, pair);
        }
    gc.maxflow();
    for (int p = 0; p < w * h; p++) labels[p] = gc.label(p);
    return 0;
}

/* ---- operator entries: the functions compute_one_level and optimize_occ are made of, on one level's planes */

/* Variational_AUX_MT::compute_smoothness, modes 0 and 1; robust_reg < 0 is not a reference penalty */
int sfo_mt_smoothness(sfo_image_t *dh, sfo_image_t *dv, const sfo_image_t *uu, const sfo_image_t *vv, const sfo_image_t *w, float alpha,
                      int mode, int robust_reg, float eps, float trunc) {
    if (mode < 0 || mode > 1 || robust_reg < 0) return 1;
    smoothness_mt(mode, dh, dv, uu, vv, w, alpha, Pen(robust_reg, eps, trunc));
    return 0;
}

/* compute_dpsis_weight of the de-normalised luminance (variational_aux_mt.cpp:673-719) */
int sfo_mt_dpsis_weight(sfo_image_t *dst, const sfo_color_image_t *im, float coef, const float avg3[3], const float std3[3], int hbit) {
    dpsis_mt(im, dst, coef, avg3, std3, hbit != 0);
    return 0;
}

/* One linearisation of compute_one_level up to the SOR: get_derivatives of the level frames im[0 .. 2(S-1)] at (wx, wy),
 * the occlusion / window factor of occ on the masks, smoothness on uu = wx + du, every data term at the increment
 * (du, dv) (NULL: zero, the first inner iteration) and the Laplacian of uu, vv subtracted from b.  The blocks are left
 * as sfo_sor_coupled takes them; channel_w NULL means all-ones weights. */
int sfo_mt_system(sfo_image_t *a11, sfo_image_t *a12, sfo_image_t *a22, sfo_image_t *b1, sfo_image_t *b2, sfo_image_t *psi_h,
                  sfo_image_t *psi_v, sfo_color_image_t *const *im, const sfo_image_t *wx, const sfo_image_t *wy, const sfo_image_t *du,
                  const sfo_image_t *dv, const sfo_image_t *occ, const sfo_color_image_t *channel_w, const sfo_mt_params_t *p) {
    const int W = wx->width, H = wx->height, ref = p->S - 1;
    if (ref < 1 || ref > SF_MT_MAX_REF || p->smoothing < 0 || p->smoothing > 1 || (du == NULL) != (dv == NULL)) return 1;
    const size_t n = (size_t)wx->stride * H;
    const Pens pen(p);
    CImg *ones = NULL;
    if (!channel_w) {
        ones = sfo_color_image_new(W, H);
        std::fill_n(ones->c1, 3 * n, 1.0f);
        channel_w = ones;
    }
    Img *zu = sfo_image_new(W, H), *zv = sfo_image_new(W, H), *uu = sfo_image_new(W, H), *vv = sfo_image_new(W, H);
    Img *dpsis = sfo_image_new(W, H);
    memset(zu->data, 0, n * sizeof(float));
    memset(zv->data, 0, n * sizeof(float));
    if (!du) { du = zu; dv = zv; }
    for (size_t k = 0; k < n; k++) { uu->data[k] = wx->data[k] + du->data[k]; vv->data[k] = wy->data[k] + dv->data[k]; }
    dpsis_mt(im[ref], dpsis, 5.0f, p->img_norm_avg, p->img_norm_std, p->hbit != 0);
    {
        LevelPlanes lp(W, H, ref);
        lp.derivatives(im, wx, wy, ref, p->one_direction != 0);
        occ_factor(lp.mask.data(), occ, p);
        Sys A = {a11, a12, a22, b1, b2};
        assemble_system(A, psi_h, psi_v, lp.mask.data(), du, dv, lp.succ.data(), lp.toref.data(), uu, vv, dpsis, channel_w, p, pen);
    }
    sfo_image_delete(zu); sfo_image_delete(zv); sfo_image_delete(uu); sfo_image_delete(vv); sfo_image_delete(dpsis);
    if (ones) sfo_color_image_delete(ones);
    return 0;
}

/* The cost half of optimizeOcc: get_derivatives of the level frames at (wx, wy) in both directions, then the data costs
 * d0 / d1 of the two labels at every pixel (the stride padding is not written) */
int sfo_mt_occ_costs(sfo_image_t *d0, sfo_image_t *d1, sfo_color_image_t *const *im, const sfo_image_t *wx, const sfo_image_t *wy,
                     const sfo_mt_params_t *p) {
    const int ref = p->S - 1;
    if (ref < 1 || ref > SF_MT_MAX_REF) return 1;
    const Pens pen(p);
    LevelPlanes lp(wx->width, wx->height, ref);
    lp.derivatives(im, wx, wy, ref, false);
    occ_costs(d0, d1, lp.mask.data(), lp.succ.data(), lp.toref.data(), ref, p->rho, p->omega, p->delta / 3.0f, p->gamma / 3.0f,
              p->occlusion_penalty, pen.pc, pen.pg);
    return 0;
}

/* normalize (variational_mt.cpp:17-85) */
int sfo_normalize(sfo_color_image_t *const *seq, int F, sfo_mt_params_t *p) {
    double avg[3] = {0, 0, 0}, sd[3] = {0, 0, 0};
    for (int f = 0; f < F; f++) {
        double a[3] = {0, 0, 0}, s[3] = {0, 0, 0};
        const CImg *im = seq[f];
        for (int i = 0; i < im->height; i++)
            for (int j = 0; j < im->width; j++) {
                const size_t o = (size_t)i * im->stride + j;
                a[0] += im->c1[o]; a[1] += im->c2[o]; a[2] += im->c3[o];
                s[0] += im->c1[o] * im->c1[o]; s[1] += im->c2[o] * im->c2[o]; s[2] += im->c3[o] * im->c3[o];
            }
        for (int c = 0; c < 3; c++) { avg[c] += a[c] / (im->height * im->width); sd[c] += s[c] / (im->height * im->width); }
    }
    for (int c = 0; c < 3; c++) {
        avg[c] /= F;
        sd[c] = sqrt((sd[c] / F) - avg[c] * avg[c]) / 255.0f;
    }
    for (int f = 0; f < F; f++) {
        CImg *im = seq[f];
        for (int i = 0; i < im->height; i++)
            for (int j = 0; j < im->width; j++) {
                const size_t o = (size_t)i * im->stride + j;
                if (sd[0] > 0) im->c1[o] = (float)((im->c1[o] - avg[0]) / sd[0]);
                if (sd[1] > 0) im->c2[o] = (float)((im->c2[o] - avg[1]) / sd[1]);
                if (sd[2] > 0) im->c3[o] = (float)((im->c3[o] - avg[2]) / sd[2]);
            }
    }
    for (int c = 0; c < 3; c++) { /* published through a stringstream: 6 significant digits (:72-84) */
        char buf[64];
        snprintf(buf, sizeof(buf), "%.6g", avg[c]);
        p->img_norm_avg[c] = (float)atof(buf);
        snprintf(buf, sizeof(buf), "%.6g", sd[c]);
        p->img_norm_std[c] = (float)atof(buf);
    }
    return 0;
}

/* Variational_MT::variational (variational_mt.cpp:526-784).  stats: {outer iterations, graph-cut calls} */
int sfo_variational_mt(sfo_image_t *wx, sfo_image_t *wy, sfo_color_image_t *const *im, const sfo_mt_params_t *p,
                       const sfo_color_image_t *channel_w, sfo_image_t *occlusions_out, float avg_change[2], int sor_mode, int *stats) {
    const int ref = p->S - 1, F = 2 * ref + 1;
    int L = p->layers;
    const Pens pen(p);
    CImg *ones = NULL;
    const CImg *cw = channel_w;
    if (!cw) {
        ones = sfo_color_image_new(wx->width, wx->height);
        std::fill_n(ones->c1, 3 * (size_t)wx->height * wx->stride, 1.0f);
        cw = ones;
    }
    const float sigma = 1 / sqrt(2 * p->p_scale);
    const int order = (int)floor(3 * sigma) + 1; /* gaussian_filter order (image.c:320) */
    std::vector<std::vector<CImg *> > pyr(L);
    for (int l = 0; l < L; l++) {
        pyr[l].resize(F);
        for (int s = 0; s < F; s++) {
            if (l == 0) {
                pyr[l][s] = sfo_color_image_new(im[s]->width, im[s]->height);
                memcpy(pyr[l][s]->c1, im[s]->c1, sizeof(float) * 3 * (size_t)im[s]->stride * im[s]->height);
            } else {
                const CImg *src = pyr[l - 1][s];
                const float nw = floor(src->width * p->p_scale), nh = floor(src->height * p->p_scale);
                CImg *blur = sfo_color_image_new(src->width, src->height);
                CImg *dst = sfo_color_image_new((int)nw, (int)nh);
                const size_t Ps = (size_t)src->stride * src->height, Pd = (size_t)dst->stride * dst->height;
                for (int c = 0; c < 3; c++) {
                    gaussian_blur(src->c1 + c * Ps, blur->c1 + c * Ps, src->height, src->width, src->stride, sigma);
                    resize_linear(blur->c1 + c * Ps, src->height, src->width, src->stride, dst->c1 + c * Pd, dst->height, dst->width, dst->stride);
                }
                sfo_color_image_delete(blur);
                pyr[l][s] = dst;
            }
        }
        if (floor(pyr[l][0]->width * p->p_scale) <= order + 1 || floor(pyr[l][0]->height * p->p_scale) <= order + 1) {
            for (int s = 0; s < F; s++) sfo_color_image_delete(pyr[l][s]);
            L = l;
            break;
        }
    }
    Img *wxl = wx, *wyl = wy;
    if (L > 1) {
        const float fx = (1.0f * pyr[L - 1][0]->width) / pyr[0][0]->width, fy = (1.0f * pyr[L - 1][0]->height) / pyr[0][0]->height;
        wxl = resize_flow(wx, pyr[L - 1][0]->width, pyr[L - 1][0]->height, fx);
        wyl = resize_flow(wy, pyr[L - 1][0]->width, pyr[L - 1][0]->height, fy);
    }
    LevelOut last = {0, 0, 0, 0};
    int outer_total = 0, gco_total = 0;
    for (int l = L - 1; l >= 0; l--) {
        if (l < L - 1) {
            const float fx = (1.0f * pyr[l][0]->width) / pyr[l + 1][0]->width, fy = (1.0f * pyr[l][0]->height) / pyr[l + 1][0]->height;
            Img *tx = resize_flow(wxl, pyr[l][0]->width, pyr[l][0]->height, fx);
            Img *ty = resize_flow(wyl, pyr[l][0]->width, pyr[l][0]->height, fy);
            sfo_image_delete(wxl);
            sfo_image_delete(wyl);
            if (l > 0) { wxl = tx; wyl = ty; }
            else {
                memcpy(wx->data, tx->data, sizeof(float) * (size_t)wx->stride * wx->height);
                memcpy(wy->data, ty->data, sizeof(float) * (size_t)wy->stride * wy->height);
                sfo_image_delete(tx); sfo_image_delete(ty);
                wxl = wx; wyl = wy;
            }
        }
        last = compute_one_level(wxl, wyl, pyr[l].data(), p, cw, l == 0 ? occlusions_out : NULL, sor_mode, pen);
        outer_total += last.outer_its;
        gco_total += last.gco_calls;
    }
    for (int l = 0; l < L; l++)
        for (int s = 0; s < F; s++) sfo_color_image_delete(pyr[l][s]);
    if (ones) sfo_color_image_delete(ones);
    if (avg_change) { avg_change[0] = last.cx; avg_change[1] = last.cy; }
    if (stats) { stats[0] = outer_total; stats[1] = gco_total; }
    return 0;
}

} // extern "C"
