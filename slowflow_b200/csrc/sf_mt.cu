// sf_mt.cu -- the multi-frame, occlusion-aware refinement: device-side restatement of
//   Variational_MT::variational        epic_flow_extended/variational_mt.cpp:526-784 (pyramid, coarse-to-fine)
//   Variational_MT::compute_one_level  :169-493 (alternation / outer / inner loops, early exits)
//   Variational_MT::get_derivatives    :87-166  (here: only the warps; derivatives are fused into K2, sf_data.cu)
//   Variational_AUX_MT::optimizeOcc    variational_aux_mt.cpp:758-887 (data costs on device, min-cut on host)
//   normalize                          variational_mt.cpp:17-85
//   cv::GaussianBlur / cv::resize      as used at variational_mt.cpp:607-611, 672-673, 711-712 (SURVEY A.8)
//
// Frame f of the window (f = 0 .. 2*ref, reference frame at f = ref) is warped once per outer iteration with the
// integer time factor f - ref (variational_aux_mt.cpp:735); the reference warps most frames twice to identical
// results.  mask_f is the in-bounds mask of that warp; the reference's mask[s] is mask_s for s < ref and
// mask_{s+1} for s >= ref (variational_mt.cpp:98-110).  The occlusion / window factors of :293-320 are applied
// on the fly inside the data-term kernel, so the raw masks survive for optimizeOcc (SURVEY A.9).
#include "sf_context.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <vector>

#include "sf_gridcut.hpp"
#include "sf_penalty.cuh"
#include "sf_stencil.cuh"

using namespace sf;

namespace sf {

// ------------------------------------------------------------------------------------------ small kernels
// uu = wx + du, vv = wy + dv; block partial sums of |old_du - du|, |old_dv - dv| over valid pixels
// (variational_mt.cpp:371-399) and, when finalize, of |uu - wx|, |vv - wy| followed by wx = uu, wy = vv
// (:412-429).  Partials go to part[block*4 + k]; the host adds them in double (deterministic).
__global__ void __launch_bounds__(256) k_mt_update(Geom g, float *__restrict__ wx, float *__restrict__ wy,
                                                   const float *__restrict__ du, const float *__restrict__ dv,
                                                   const float *__restrict__ odu, const float *__restrict__ odv,
                                                   float *__restrict__ uu, float *__restrict__ vv, int finalize,
                                                   float *__restrict__ part) {
    if (g.cancelled()) return;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    const int i = blockIdx.x * 32 + threadIdx.x;
    for (int j = blockIdx.y * 8 + threadIdx.y; j < g.H; j += gridDim.y * 8) {
        if (i < g.W) {
            const size_t o = (size_t)j * g.S + i;
            const float a = du[o], b = dv[o];
            s0 += fabsf((odu ? odu[o] : 0.0f) - a);
            s1 += fabsf((odv ? odv[o] : 0.0f) - b);
            const float x = wx[o], y = wy[o];
            const float nu = x + a, nv = y + b;
            if (finalize) {
                s2 += fabsf(nu - x);
                s3 += fabsf(nv - y);
                wx[o] = nu;
                wy[o] = nv;
            }
            if (uu) { uu[o] = nu; vv[o] = nv; }
        }
    }
    __shared__ float red[4][256];
    const int t = threadIdx.y * 32 + threadIdx.x;
    red[0][t] = s0; red[1][t] = s1; red[2][t] = s2; red[3][t] = s3;
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) {
        if (t < k) {
            red[0][t] += red[0][t + k]; red[1][t] += red[1][t + k]; red[2][t] += red[2][t + k]; red[3][t] += red[3][t + k];
        }
        __syncthreads();
    }
    if (t < 4) part[(size_t)(blockIdx.y * gridDim.x + blockIdx.x) * 4 + t] = red[t][0];
}

// Device-side end of an outer iteration (niter_inner == 1): adds the block partials of k_mt_update in a fixed order
// (double, deterministic), publishes the mean absolute change of the iteration (variational_mt.cpp:412-429) and raises
// the skip flag when it is below thres_outer (:436-437) -- the launches of the remaining outer iterations of this
// alternation, already queued behind this kernel, then fall through.
struct MtLoopState {
    int stop;              // Geom::skip points here
    int outer_done;        // outer iterations executed since the level started
    float avg_change[2];   // of the last executed outer iteration
};
__global__ void __launch_bounds__(256) k_mt_close_iteration(Geom g, const float *__restrict__ part, int nblocks, double inv_n,
                                                            float thres_outer, MtLoopState *state) {
    if (g.cancelled()) return;
    __shared__ double red[2][256];
    double a = 0.0, b = 0.0;
    for (int k = threadIdx.x; k < nblocks; k += 256) { // fixed assignment of blocks to threads, fixed tree below
        a += (double)part[(size_t)k * 4 + 2];
        b += (double)part[(size_t)k * 4 + 3];
    }
    red[0][threadIdx.x] = a;
    red[1][threadIdx.x] = b;
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) {
        if ((int)threadIdx.x < k) {
            red[0][threadIdx.x] += red[0][threadIdx.x + k];
            red[1][threadIdx.x] += red[1][threadIdx.x + k];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float cx = (float)(red[0][0] * inv_n), cy = (float)(red[1][0] * inv_n);
        state->avg_change[0] = cx;
        state->avg_change[1] = cy;
        state->outer_done += 1;
        if (fmaxf(cx, cy) < thres_outer) state->stop = 1;
    }
}

// per-pixel data costs of the binary occlusion labelling (variational_aux_mt.cpp:786-848).
// W[f]: warped frame f (W[ref] = reference frame), mk[f]: raw mask of frame f.
struct OccArgs {
    const float *W[2 * SF_MT_MAX_REF + 1];
    const float *mk[2 * SF_MT_MAX_REF + 1];
    float rho[SF_MT_MAX_REF], omega[SF_MT_MAX_REF];
    int ref;
    float delta_over3, gamma_over3, penalty;
    Penalty pc, pg;
};
// The two data costs are quantised exactly like the labelling step does on the host (x 2^24, round half away from zero;
// gco's stock int EnergyTermType truncates the cost first) and only their difference leaves the GPU:
// tr[y*W + x] = q(d1) - q(d0) = cap(source -> p) - cap(p -> sink) of SinkForestCut (sf_gridcut.hpp).
__device__ __forceinline__ long long occ_quantise(float e, int int_terms) {
    return llround((int_terms ? (double)(int)e : (double)e) * 16777216.0);
}
__global__ void __launch_bounds__(256) k_occ_costs(Geom g, OccArgs a, float *__restrict__ d0, float *__restrict__ d1,
                                                   long long *__restrict__ tr, int int_terms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= g.W || j >= g.H) return;
    const size_t P = g.plane();
    const size_t o = (size_t)j * g.S + i;
    const int W1 = g.W - 1, H1 = g.H - 1;
    float e[2] = {0.f, 0.f}, nrm[2] = {0.f, 0.f};
    for (int s = 0; s < 2 * a.ref; s++) {
        const int idx = max(a.ref - s - 1, s - a.ref);
        const float m = a.mk[s < a.ref ? s : s + 1][o];
        float term = 0.f;
        for (int kind = 0; kind < 2; kind++) { // 0: successive pair (s, s+1); 1: frame vs reference
            const float *A, *B;
            if (kind == 0) { A = a.W[s]; B = a.W[s + 1]; }
            else if (s < a.ref) { A = a.W[s]; B = a.W[a.ref]; }
            else { A = a.W[a.ref]; B = a.W[s + 1]; }
            float sz = 0.f, sx = 0.f, sy = 0.f;
            for (int c = 0; c < 3; c++) {
                const float *pa = A + c * P, *pb = B + c * P;
                auto Z = [&](int x, int y) { const size_t q = (size_t)clampi(y, 0, H1) * g.S + clampi(x, 0, W1); return pa[q] - pb[q]; };
                const float z0 = Z(i, j);
                const float zx = hconv5(Z(i - 2, j), Z(i - 1, j), z0, Z(i + 1, j), Z(i + 2, j));
                const float zy = vconv5(Z(i, j - 2), Z(i, j - 1), z0, Z(i, j + 1), Z(i, j + 2), j, g.H);
                sz += z0 * z0;
                sx += zx * zx;
                sy += zy * zy;
            }
            const float w = (kind == 0) ? a.rho[idx] : a.omega[idx];
            const float part = w * a.delta_over3 * m * penalty_apply_v(a.pc, sz) + w * a.gamma_over3 * m * penalty_apply_v(a.pg, sx + sy);
            term += part;
        }
        const int l = (s >= a.ref) ? 0 : 1;
        e[l] += term;
        nrm[l] += m * (a.rho[idx] + a.rho[idx] + a.omega[idx] + a.omega[idx]);
    }
    if (nrm[0] == 0.f) nrm[0] = 1.f;
    if (nrm[1] == 0.f) nrm[1] = 1.f;
    const float c0 = 0.01f * e[0] / nrm[0] + a.penalty * 0.0f;
    const float c1 = 0.01f * e[1] / nrm[1] + a.penalty * 1.0f;
    if (d0) { d0[o] = c0; d1[o] = c1; }
    if (tr) tr[(size_t)j * g.W + i] = occ_quantise(c1, int_terms) - occ_quantise(c0, int_terms);
}

// labels of the min-cut (forest membership bytes, dense W*H) -> occlusion plane: +1 in the forest, -1 outside, 0 in
// the stride padding (variational_aux_mt.cpp:879)
__global__ void __launch_bounds__(256) k_occ_labels(Geom g, const unsigned char *__restrict__ member, unsigned char none,
                                                    float *__restrict__ occ) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= g.S || j >= g.H) return;
    occ[(size_t)j * g.S + i] = (i < g.W) ? (member[(size_t)j * g.W + i] != none ? 1.0f : -1.0f) : 0.0f;
}

// separable Gaussian (replicate border), symmetric-sum evaluation like cv::GaussianBlur's float path.  Both passes handle
// 4 consecutive pixels per thread with float4 loads / stores (rows are 16-byte aligned: stride = ceil4(width)).
struct BlurTaps { int r; float k[17]; }; // k[0] centre, k[i] at distance i
constexpr int BLUR_SEG = 128 * 4; // columns per block of the horizontal pass (128 threads x 4)
// horizontal pass: the block stages its row segment + r columns on either side (clamped to the row) in shared memory
__global__ void __launch_bounds__(128) k_blur_h4(Geom g, const float *__restrict__ src, float *__restrict__ dst, BlurTaps t, int planes) {
    __shared__ float row[BLUR_SEG + 2 * 16 + 8];
    const int y = blockIdx.y, x0 = blockIdx.x * BLUR_SEG;
    const size_t P = g.plane();
    const int lo = x0 - 16; // multiple of 4
    for (int c = 0; c < planes; c++) {
        const float *s = src + c * P + (size_t)y * g.S;
        for (int q = threadIdx.x; q < (BLUR_SEG + 32) / 4; q += 128) {
            const int x = lo + 4 * q;
            float4 v;
            if (x >= 0 && x + 3 < g.W) v = *reinterpret_cast<const float4 *>(s + x);
            else v = make_float4(s[clampi(x, 0, g.W - 1)], s[clampi(x + 1, 0, g.W - 1)], s[clampi(x + 2, 0, g.W - 1)], s[clampi(x + 3, 0, g.W - 1)]);
            *reinterpret_cast<float4 *>(row + 4 * q) = v;
        }
        __syncthreads();
        const int x = x0 + 4 * threadIdx.x;
        if (x < g.S) {
            const float *p = row + 16 + 4 * threadIdx.x;
            float a0 = t.k[0] * p[0], a1 = t.k[0] * p[1], a2 = t.k[0] * p[2], a3 = t.k[0] * p[3];
            for (int k = 1; k <= t.r; k++) {
                const float w = t.k[k];
                a0 += w * (p[-k] + p[k]);
                a1 += w * (p[1 - k] + p[1 + k]);
                a2 += w * (p[2 - k] + p[2 + k]);
                a3 += w * (p[3 - k] + p[3 + k]);
            }
            // the stride padding takes the value of the clamped column: it is never read as image data
            *reinterpret_cast<float4 *>(dst + c * P + (size_t)y * g.S + x) = make_float4(a0, a1, a2, a3);
        }
        __syncthreads();
    }
}
// vertical pass: float4 per row tap, rows clamped
__global__ void __launch_bounds__(256) k_blur_v4(Geom g, const float *__restrict__ src, float *__restrict__ dst, BlurTaps t, int planes) {
    const int x = (blockIdx.x * 32 + threadIdx.x) * 4, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= g.S || y >= g.H) return;
    const size_t P = g.plane();
    for (int c = 0; c < planes; c++) {
        const float *s = src + c * P + x;
        float4 acc = *reinterpret_cast<const float4 *>(s + (size_t)y * g.S);
        acc.x *= t.k[0]; acc.y *= t.k[0]; acc.z *= t.k[0]; acc.w *= t.k[0];
        for (int k = 1; k <= t.r; k++) {
            const float4 a = *reinterpret_cast<const float4 *>(s + (size_t)clampi(y - k, 0, g.H - 1) * g.S);
            const float4 b = *reinterpret_cast<const float4 *>(s + (size_t)clampi(y + k, 0, g.H - 1) * g.S);
            const float w = t.k[k];
            acc.x += w * (a.x + b.x); acc.y += w * (a.y + b.y); acc.z += w * (a.z + b.z); acc.w += w * (a.w + b.w);
        }
        *reinterpret_cast<float4 *>(dst + c * P + (size_t)y * g.S + x) = acc;
    }
}
static void launch_blur(cudaStream_t st, Geom g, const float *src, float *tmp, float *dst, const BlurTaps &t, int planes) {
    k_blur_h4<<<dim3((g.S + BLUR_SEG - 1) / BLUR_SEG, g.H), 128, 0, st>>>(g, src, tmp, t, planes);
    k_blur_v4<<<dim3((g.S / 4 + 31) / 32, (g.H + 7) / 8), dim3(32, 8), 0, st>>>(g, tmp, dst, t, planes);
}
// bilinear resize with pixel-centre mapping (cv::resize INTER_LINEAR), optional scale of the values; 4 destination pixels
// per thread, float4 stores (the stride padding is zeroed)
__global__ void __launch_bounds__(256) k_resize(Geom gs, const float *__restrict__ src, Geom gd, float *__restrict__ dst,
                                                double scale_x, double scale_y, float mul, int planes) {
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x4 >= gd.S || y >= gd.H) return;
    const size_t Ps = gs.plane(), Pd = gd.plane();
    float fy = (float)((y + 0.5) * scale_y - 0.5);
    int sy = (int)floorf(fy);
    fy -= sy;
    if (sy < 0) { sy = 0; fy = 0.f; }
    if (sy >= gs.H - 1) { sy = gs.H - 1; fy = 0.f; }
    const int y1 = min(sy + 1, gs.H - 1);
    const float b1 = fy, b0 = 1.f - fy;
    int sx[4], x1[4];
    float a0[4], a1[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        float fx = (float)((x4 + k + 0.5) * scale_x - 0.5);
        int q = (int)floorf(fx);
        fx -= q;
        if (q < 0) { q = 0; fx = 0.f; }
        if (q >= gs.W - 1) { q = gs.W - 1; fx = 0.f; }
        sx[k] = q;
        x1[k] = min(q + 1, gs.W - 1);
        a1[k] = fx;
        a0[k] = 1.f - fx;
    }
    for (int c = 0; c < planes; c++) {
        const float *s0 = src + c * Ps + (size_t)sy * gs.S, *s1 = src + c * Ps + (size_t)y1 * gs.S;
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (x4 + k < gd.W) {
                const float r0 = s0[sx[k]] * a0[k] + s0[x1[k]] * a1[k];
                const float r1 = s1[sx[k]] * a0[k] + s1[x1[k]] * a1[k];
                float v = r0 * b0 + r1 * b1;
                if (mul != 1.0f) v *= mul; // image_mul_scalar (image.c:49-57)
                o[k] = v;
            } else {
                o[k] = 0.0f;
            }
        }
        *reinterpret_cast<float4 *>(dst + c * Pd + (size_t)y * gd.S + x4) = make_float4(o[0], o[1], o[2], o[3]);
    }
}
static dim3 resize_grid(Geom gd) { return dim3((gd.S / 4 + 31) / 32, (gd.H + 7) / 8); }

// rawWeighting (utils/utils.cpp:1336-1374): per-pixel channel weights of a Bayer mosaic whose red site is at
// (red_x, red_y) mod 2 -- the measured channel gets `weight`, the two interpolated ones 0.5*(3 - weight)
__global__ void __launch_bounds__(256) k_raw_weights(Geom g, float *__restrict__ w3, int red_x, int red_y, float weight) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= g.W || y >= g.H) return;
    const size_t P = g.plane(), o = (size_t)y * g.S + x;
    const float other = 0.5f * (3.0f - weight);
    int measured; // 0 R, 1 G, 2 B
    if ((y + (1 - red_y)) % 2 == 0) { // blue row
        const bool green = (red_y == 1 && (x + (1 - red_x)) % 2 == 0) || (red_y == 0 && (x + red_x) % 2 == 0);
        measured = green ? 1 : 2;
    } else { // red row
        const bool green = (red_y == 0 && (x + (1 - red_x)) % 2 == 0) || (red_y == 1 && (x + red_x) % 2 == 0);
        measured = green ? 1 : 0;
    }
    w3[o] = measured == 0 ? weight : other;
    w3[o + P] = measured == 1 ? weight : other;
    w3[o + 2 * P] = measured == 2 ? weight : other;
}

// normalize(): per-channel sums in double (variational_mt.cpp:27-46), then (I - avg) / std (:61-69).  Every block writes
// its six partial sums to sums[block*6 + k]; the host adds them in block order (deterministic: no atomics on the path).
__global__ void __launch_bounds__(256) k_norm_sums(Geom g, const float *__restrict__ im, double *__restrict__ sums /*gridDim.x * 6*/) {
    double s[6] = {0, 0, 0, 0, 0, 0};
    const size_t P = g.plane();
    for (int j = blockIdx.x; j < g.H; j += gridDim.x)
        for (int i = threadIdx.x; i < g.W; i += blockDim.x)
            for (int c = 0; c < 3; c++) {
                const double v = im[c * P + (size_t)j * g.S + i];
                s[c] += v;
                s[3 + c] += v * v;
            }
    __shared__ double red[6][256];
    for (int k = 0; k < 6; k++) red[k][threadIdx.x] = s[k];
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) {
        if ((int)threadIdx.x < k)
            for (int q = 0; q < 6; q++) red[q][threadIdx.x] += red[q][threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x < 6) sums[(size_t)blockIdx.x * 6 + threadIdx.x] = red[threadIdx.x][0];
}
__global__ void __launch_bounds__(256) k_norm_apply(Geom g, float *__restrict__ im, double a0, double a1, double a2, double s0,
                                                    double s1, double s2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= g.W || j >= g.H) return;
    const size_t P = g.plane(), o = (size_t)j * g.S + i;
    if (s0 > 0) im[o] = (float)(((double)im[o] - a0) / s0);
    if (s1 > 0) im[o + P] = (float)(((double)im[o + P] - a1) / s1);
    if (s2 > 0) im[o + 2 * P] = (float)(((double)im[o + 2 * P] - a2) / s2);
}

static dim3 grid2d(int w, int h) { return dim3((w + 31) / 32, (h + 7) / 8); }

// ------------------------------------------------------------------------------------------ level state
struct MtLevel {
    Geom g;
    std::vector<float *> frames; // F colour images (3 planes each)
};

// Per-context multi-frame workspace; kept between calls (buffers only grow).
struct MtWork {
    float *pool = nullptr;
    size_t pool_floats = 0;
    float *part_dev = nullptr;
    float *part_host = nullptr; // pinned
    size_t part_cap = 0;
    long long *tr_host = nullptr; // pinned: terminal capacities of the occlusion min-cut
    unsigned char *lab_dev = nullptr;
    size_t cut_nodes = 0;
    MtLoopState *loop_dev = nullptr;  // device-side outer-loop state (skip flag, counters)
    MtLoopState *loop_host = nullptr; // pinned read-back
    SinkForestCut cut;
    ~MtWork() { release(); }
    void release() {
        if (pool) cudaFree(pool);
        if (part_dev) cudaFree(part_dev);
        if (part_host) cudaFreeHost(part_host);
        if (tr_host) cudaFreeHost(tr_host);
        if (lab_dev) cudaFree(lab_dev);
        if (loop_dev) cudaFree(loop_dev);
        if (loop_host) cudaFreeHost(loop_host);
        loop_dev = loop_host = nullptr;
        pool = part_dev = part_host = nullptr;
        tr_host = nullptr;
        lab_dev = nullptr;
        pool_floats = part_cap = cut_nodes = 0;
    }
    int reserve(size_t floats, size_t partials, size_t nodes) {
        if (!loop_dev) {
            SF_CUDA(cudaMalloc(&loop_dev, sizeof(MtLoopState)));
            SF_CUDA(cudaMallocHost(&loop_host, sizeof(MtLoopState)));
        }
        if (floats > pool_floats) {
            if (pool) cudaFree(pool);
            pool = nullptr; pool_floats = 0;
            SF_CUDA(cudaMalloc(&pool, floats * sizeof(float)));
            pool_floats = floats;
        }
        if (partials > part_cap) {
            if (part_dev) cudaFree(part_dev);
            if (part_host) cudaFreeHost(part_host);
            part_dev = part_host = nullptr; part_cap = 0;
            SF_CUDA(cudaMalloc(&part_dev, partials * sizeof(float)));
            SF_CUDA(cudaMallocHost(&part_host, partials * sizeof(float)));
            part_cap = partials;
        }
        if (nodes > cut_nodes) {
            if (tr_host) cudaFreeHost(tr_host);
            if (lab_dev) cudaFree(lab_dev);
            tr_host = nullptr; lab_dev = nullptr; cut_nodes = 0;
            SF_CUDA(cudaMallocHost(&tr_host, nodes * sizeof(long long)));
            SF_CUDA(cudaMalloc(&lab_dev, nodes));
            cut_nodes = nodes;
        }
        return SFGPU_OK;
    }
};
void mt_work_free(MtWork *w) { delete w; }

static BlurTaps make_taps(double sigma) {
    // cv::getGaussianKernel: n = cvRound(8 sigma + 1) | 1 for CV_32F, exp(-x^2 / 2 sigma^2) normalised
    BlurTaps t;
    int n = ((int)lrint(sigma * 8 + 1)) | 1;
    if (n > 33) n = 33;
    t.r = n / 2;
    std::vector<double> v(n);
    double sum = 0;
    for (int i = 0; i < n; i++) {
        const double x = i - (n - 1) * 0.5;
        v[i] = exp(-0.5 / (sigma * sigma) * x * x);
        sum += v[i];
    }
    for (int k = 0; k <= t.r; k++) t.k[k] = (float)(v[t.r + k] / sum);
    for (int k = t.r + 1; k < 17; k++) t.k[k] = 0.f;
    return t;
}

// ------------------------------------------------------------------------------------------ one level
struct LevelCtx {
    sfgpu_ctx *c;
    const sf_mt_params_t *p;
    Geom g;
    int ref;
    bool one_direction;
    float alpha, gamma_over3, delta_over3;
    Penalty pc, pg, preg;
    std::vector<float *> frames;  // level frames
    std::vector<float *> warped;  // per frame (warped[ref] == frames[ref])
    std::vector<float *> masks;   // per frame (masks[ref] unused)
    std::vector<float *> derivs;  // per frame: 15 derivative planes (fused_terms)
    bool fused_terms = false;     // data pass = per-frame derivatives + one pointwise all-terms kernel (sf_data.cu)
    float *wx, *wy, *uu, *vv, *odu, *odv, *dpsis, *occ, *d0, *d1;
    bool cut_pending = false;     // a device min-cut was queued: its status must be read when the stream is next synchronised
    const float *chw;             // channel weights (level-0 planes; Q14: not rescaled per level)
    size_t chw_pstride;
    MtWork *work;
};

static int read_partials(LevelCtx &L, dim3 grid, double out[4]) {
    const size_t n = (size_t)grid.x * grid.y * 4;
    SF_CUDA(cudaMemcpyAsync(L.work->part_host, L.work->part_dev, n * sizeof(float), cudaMemcpyDeviceToHost, L.c->stream));
    SF_CUDA(cudaStreamSynchronize(L.c->stream));
    out[0] = out[1] = out[2] = out[3] = 0.0;
    for (size_t b = 0; b < n; b += 4)
        for (int k = 0; k < 4; k++) out[k] += L.work->part_host[b + k];
    return SFGPU_OK;
}

static void warp_all(LevelCtx &L) { // Variational_MT::get_derivatives, warping part (variational_mt.cpp:96-110)
    const int F = 2 * L.ref + 1;
    if (L.fused_terms && L.c->mt_warp_variant == 0) {
        // warp + the frames' own derivative images in one marching pass over ALL warped frames (sf_wderivs.cu); every
        // term that uses a frame combines its derivative planes linearly
        const float *src[MT_MAX_FRAMES];
        float *warped[MT_MAX_FRAMES], *masks[MT_MAX_FRAMES], *derivs[MT_MAX_FRAMES];
        int factor[MT_MAX_FRAMES], n = 0;
        for (int f = (L.one_direction ? L.ref + 1 : 0); f < F; f++) {
            if (f == L.ref) continue;
            src[n] = L.frames[f]; factor[n] = f - L.ref; warped[n] = L.warped[f]; masks[n] = L.masks[f]; derivs[n] = L.derivs[f];
            n++;
        }
        cudaEvent_t ev;
        L.c->prof_begin(1, ev);
        launch_warp_derivs_batch(L.c->stream, L.g, L.c->num_sms, L.wx, L.wy, n, src, factor, warped, masks, derivs);
        L.c->prof_end(1, ev);
        L.c->prof_acc.kernel_launches += (n + 7) / 8;
        return;
    }
    for (int f = (L.one_direction ? L.ref + 1 : 0); f < F; f++) {
        if (f == L.ref) continue;
        launch_warp(L.c->stream, L.g, L.frames[f], L.wx, L.wy, f - L.ref, L.warped[f], L.masks[f]);
        L.c->prof_acc.kernel_launches++;
        if (L.fused_terms) { // A/B reference (SLOWFLOW_GPU_MT_WARP_VARIANT=1): separate warp kernel + tile-based derivative kernel
            cudaEvent_t ev;
            L.c->prof_begin(1, ev);
            launch_frame_derivs(L.c->stream, L.g, L.warped[f], L.derivs[f]);
            L.c->prof_end(1, ev);
            L.c->prof_acc.kernel_launches++;
        }
    }
}

static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static SinkForestCut::cap_t occ_quantise_host(double e, bool int_terms) {
    return (SinkForestCut::cap_t)llround((int_terms ? (double)(int)e : e) * 16777216.0);
}

static OccArgs occ_args(const LevelCtx &L) { // the inputs of k_occ_costs: warped frames, raw masks, weights, penalties
    OccArgs a;
    memset(&a, 0, sizeof(a));
    const int F = 2 * L.ref + 1;
    for (int f = 0; f < F; f++) { a.W[f] = L.warped[f]; a.mk[f] = L.masks[f]; }
    for (int s = 0; s < L.ref; s++) { a.rho[s] = L.p->rho[s]; a.omega[s] = L.p->omega[s]; }
    a.ref = L.ref;
    a.delta_over3 = L.delta_over3;
    a.gamma_over3 = L.gamma_over3;
    a.penalty = L.p->occlusion_penalty;
    a.pc = L.pc;
    a.pg = L.pg;
    return a;
}

static int optimize_occ(LevelCtx &L) { // variational_aux_mt.cpp:758-887
    const Geom g = L.g;
    const double t_begin = now_ms();
    const OccArgs a = occ_args(L);
    // d0,d1 are two consecutive planes: reused as the dense W*H array of 64-bit terminal capacities
    const bool int_terms = L.p->graphcut_int_terms != 0;
    long long *tr_dev = reinterpret_cast<long long *>(L.d0);
    MtWork &wk = *L.work;
    const size_t N = (size_t)g.W * g.H;
    cudaEvent_t ev;
    L.c->prof_begin(2, ev);
    k_occ_costs<<<grid2d(g.W, g.H), dim3(32, 8), 0, L.c->stream>>>(g, a, nullptr, nullptr, tr_dev, int_terms ? 1 : 0);
    L.c->prof_acc.kernel_launches++;
    const SinkForestCut::cap_t pair_cap = occ_quantise_host((double)L.p->occlusion_alpha, int_terms);
    if (!L.c->host_mincut) {
        // binary Potts labelling = one min-cut (gco stand-in semantics), on the device: the terminal capacities never
        // leave HBM and nothing synchronises; the solver's status is checked when the level ends
        const int rcc = device_grid_mincut(L.c, L.c->cut, g.W, g.H, tr_dev, (long long)pair_cap, L.occ, g.S);
        if (rcc != SFGPU_OK) return rcc;
        L.c->prof_acc.kernel_launches++;
        L.c->prof_end(2, ev);
        L.cut_pending = true;
    } else {
        SF_CUDA(cudaMemcpyAsync(wk.tr_host, tr_dev, N * sizeof(long long), cudaMemcpyDeviceToHost, L.c->stream));
        SF_CUDA(cudaStreamSynchronize(L.c->stream));
        const double t_flow = now_ms();
        wk.cut.solve(g.W, g.H, reinterpret_cast<SinkForestCut::cap_t *>(wk.tr_host), pair_cap);
        if (getenv("SLOWFLOW_GPU_TRACE"))
            fprintf(stderr, "optimize_occ %dx%d: costs+d2h %.2f ms, min-cut %.2f ms\n", g.W, g.H, t_flow - t_begin, now_ms() - t_flow);
        SF_CUDA(cudaMemcpyAsync(wk.lab_dev, wk.cut.in_forest(), N, cudaMemcpyHostToDevice, L.c->stream));
        k_occ_labels<<<grid2d(g.S, g.H), dim3(32, 8), 0, L.c->stream>>>(g, wk.lab_dev, (unsigned char)SinkForestCut::P_NONE, L.occ);
        L.c->prof_acc.kernel_launches++;
        L.c->prof_end(2, ev);
        SF_CUDA(cudaStreamSynchronize(L.c->stream)); // the forest bytes are read by the copy above
    }
    L.c->mt_stats.graphcut_calls++;
    L.c->mt_stats.graphcut_ms += now_ms() - t_begin;
    return SFGPU_OK;
}

// The data terms of one level in both data-pass forms: the per-term chain (SLOWFLOW_GPU_MT_DATA_VARIANT=1) and the
// all-terms pass.  The frames' derivative planes come from warp_all, the reference frame's from mt_system_setup.
struct MtSystemTerms {
    std::vector<DataTermDesc> terms; // ordered term list of :343-361
    MtTermsArgs ta;
    float data_norm = 0.f;
};

static void mt_system_setup(LevelCtx &L, MtSystemTerms &sys) {
    const sf_mt_params_t *p = L.p;
    const int ref = L.ref;
    for (int s = 0; s < ref; s++) sys.data_norm += p->rho[s] + p->omega[s];
    std::vector<DataTermDesc> &terms = sys.terms;
    MtTermsArgs &ta = sys.ta;
    auto pair_imgs = [&](int q, int kind, const float *&Aimg, const float *&Bimg) {
        if (kind == DK_MT_SUCC) { Aimg = L.warped[q]; Bimg = L.warped[q + 1]; }
        else if (q < ref) { Aimg = L.warped[q]; Bimg = L.frames[ref]; }
        else { Aimg = L.frames[ref]; Bimg = L.warped[q + 1]; }
    };
    memset(&ta, 0, sizeof(ta));
    auto add_term = [&](int q, int kind, float w, float time, int dir) {
        if (ta.nterms < MT_MAX_TERMS) {
            MtTerm &m = ta.term[ta.nterms++];
            m.fa = (kind == DK_MT_SUCC || q < ref) ? q : ref;
            m.fb = (kind == DK_MT_SUCC) ? q + 1 : (q < ref ? ref : q + 1);
            m.mask_frame = q < ref ? q : q + 1;
            m.kind = kind;
            m.dir = dir;
            m.wd = w * L.delta_over3;
            m.wg = w * L.gamma_over3;
            m.s = time;
        }
        DataTermDesc t;
        pair_imgs(q, kind, t.A, t.B);
        t.zsign = -1; // Iz = im1 - im2 (variational_mt.cpp:127,152)
        t.mask = L.masks[q < ref ? q : q + 1];
        t.kind = kind;
        t.wd = w * L.delta_over3;
        t.wg = w * L.gamma_over3;
        t.s = time;
        t.dir = dir;
        terms.push_back(t);
    };
    for (int s = 0; s < ref; s++) {
        if (!L.one_direction) {
            if (p->rho[ref - 1 - s] > 0) add_term(s, DK_MT_SUCC, p->rho[ref - 1 - s], (float)(s - ref), 0);
            if (p->omega[ref - 1 - s] > 0) add_term(s, DK_MT_REF, p->omega[ref - 1 - s], (float)(s - ref), 0);
        }
        if (p->rho[s] > 0) add_term(ref + s, DK_MT_SUCC, p->rho[s], (float)s, 1);
        if (p->omega[s] > 0) add_term(ref + s, DK_MT_REF, p->omega[s], (float)(s + 1), 1);
    }

    if (L.fused_terms) {
        for (int f = 0; f < 2 * ref + 1; f++) { ta.I[f] = L.warped[f]; ta.D[f] = L.derivs[f]; ta.mask[f] = L.masks[f]; }
        launch_frame_derivs(L.c->stream, L.g, L.frames[ref], L.derivs[ref]); // the reference frame is never warped: once per level
        L.c->prof_acc.kernel_launches++;
    }
}

// One linearisation up to the SOR (:333-365) into the arena planes SP_A11 .. SP_PV of A: smoothness weights of (uu, vv),
// every data term at the increment (du, dv) (nullptr: zero), b -= div(psi grad uu / vv) and the 2x2 block inverse.
static void launch_mt_system(LevelCtx &L, const MtSystemTerms &sys, const Geom &g, const float *uu, const float *vv, const float *du,
                             const float *dv, float *A) {
    sfgpu_ctx *c = L.c;
    cudaStream_t st = c->stream;
    const size_t P = g.plane();
    launch_smoothness(st, g, uu, vv, L.dpsis, L.alpha, L.preg, L.p->smoothing, A + SP_PH * P, A + SP_PV * P); // :333
    c->prof_acc.kernel_launches++;
    DataCommon cm{};
    cm.du = du;
    cm.dv = dv;
    cm.chw = L.chw;
    cm.chw_pstride = L.chw_pstride;
    cm.occ = L.occ;
    cm.data_norm = sys.data_norm;
    cm.dt_norm = L.p->dataterm;
    cm.pc = L.pc;
    cm.pg = L.pg;
    cm.ph = A + SP_PH * P; cm.pv = A + SP_PV * P;
    cm.lap_u = uu; cm.lap_v = vv; // MT passes uu, vv to sub_laplacian (:364-365, SURVEY Q11)
    cm.a11 = A + SP_A11 * P; cm.a12 = A + SP_A12 * P; cm.a22 = A + SP_A22 * P;
    cm.b1 = A + SP_B1 * P; cm.b2 = A + SP_B2 * P;
    cudaEvent_t ev;
    c->prof_begin(1, ev);
    if (sys.terms.empty()) { // no active data term: the system is the smoothness term alone
        launch_fill(st, cm.a11, 5 * P, 0.0f);
        launch_sub_laplacian(st, g, cm.b1, uu, cm.ph, cm.pv);
        launch_sub_laplacian(st, g, cm.b2, vv, cm.ph, cm.pv);
        launch_invert_blocks(st, g, cm.a11, cm.a12, cm.a22, cm.ph, cm.pv);
        c->prof_acc.kernel_launches += 4;
    } else if (L.fused_terms) { // all data terms of one linearisation (:343-361)
        launch_mt_terms(st, g, sys.ta, cm, c->mt_terms_scalar);
        c->prof_acc.kernel_launches++;
        c->prof_acc.data_launches++;
        c->prof_acc.data_pixels += (long long)g.W * g.H;
    } else {
        for (size_t k = 0; k < sys.terms.size(); k++) {
            cm.accumulate = (k > 0);
            cm.fuse_system = (k + 1 == sys.terms.size());
            launch_data_term(st, g, sys.terms[k], cm);
            c->prof_acc.kernel_launches++;
            c->prof_acc.data_launches++;
            c->prof_acc.data_pixels += (long long)g.W * g.H;
        }
    }
    c->prof_end(1, ev);
}

static int compute_one_level(LevelCtx &L, float avg_change[2]) { // variational_mt.cpp:169-493
    sfgpu_ctx *c = L.c;
    const sf_mt_params_t *p = L.p;
    const Geom g = L.g;
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    float *A = c->sor.arena;
    const int ref = L.ref;

    // occlusion labels: 0, or -1 everywhere ("occluded in the past") when reasoning / one direction (:213-220)
    launch_fill(st, L.occ, P, (L.one_direction || p->occlusion_reasoning) ? -1.0f : 0.0f);
    launch_dpsis_weight(st, g, L.frames[ref], L.dpsis, 5.0f, p->img_norm_avg, p->img_norm_std, p->hbit ? 65535.0f : 255.0f);
    c->prof_acc.kernel_launches += 2;
    MtSystemTerms sys;
    mt_system_setup(L, sys);
    const dim3 ugrid((g.W + 31) / 32, std::min((g.H + 7) / 8, 64));
    avg_change[0] = avg_change[1] = 0.f;
    const double inv_n = 1.0 / ((double)g.H * g.W);

    if (p->niter_inner == 1) {
        // ---- default shape (one inner iteration): no host round trip inside the level.  Every kernel of the outer loop
        // carries the skip flag; the host reads the loop state back once, after the last alternation (and whenever the
        // occlusion step synchronises anyway).
        MtLoopState *state = L.work->loop_dev;
        SF_CUDA(cudaMemsetAsync(state, 0, sizeof(MtLoopState), st));
        const int *flag = &state->stop;
        const int nblocks = (int)(ugrid.x * ugrid.y);
        for (int alter = 0; alter < p->niter_alter; alter++) {
            SF_CUDA(cudaMemsetAsync(&state->stop, 0, sizeof(int), st)); // a break leaves the outer loop, not the alternation loop
            L.g.skip = nullptr;
            c->sor.g.skip = nullptr;
            warp_all(L); // :266
            if (alter > 0 && p->occlusion_reasoning && !L.one_direction) { // :269-272
                int rc = optimize_occ(L);
                if (rc != SFGPU_OK) return rc;
            }
            L.g.skip = flag;
            c->sor.g.skip = flag;
            const Geom gs = L.g;
            for (int outer = 0; outer < p->niter_outer; outer++) {
                if (outer > 0) warp_all(L); // :289-290
                int cur = 0;
                launch_mt_system(L, sys, gs, L.wx, L.wy, nullptr, nullptr, A); // uu == wx at the start of an outer iteration
                int rc = run_sor(c, p->niter_solver, p->sor_omega, &cur, true); // :368
                if (rc != SFGPU_OK) { c->sor.g.skip = nullptr; return rc; }
                const float *ndu = A + (size_t)(cur ? SP_DUB : SP_DUA) * P, *ndv = A + (size_t)(cur ? SP_DVB : SP_DVA) * P;
                k_mt_update<<<ugrid, dim3(32, 8), 0, st>>>(gs, L.wx, L.wy, ndu, ndv, nullptr, nullptr, nullptr, nullptr, 1, L.work->part_dev);
                k_mt_close_iteration<<<1, 256, 0, st>>>(gs, L.work->part_dev, nblocks, inv_n, p->thres_outer, state);
                c->prof_acc.kernel_launches += 2;
            }
        }
        L.g.skip = nullptr;
        c->sor.g.skip = nullptr;
        SF_CUDA(cudaMemcpyAsync(L.work->loop_host, state, sizeof(MtLoopState), cudaMemcpyDeviceToHost, st));
        SF_CUDA(cudaStreamSynchronize(st));
        if (L.cut_pending && (device_cut_status(c->cut)[0] != 0 || device_cut_status(c->cut)[3] != 0)) {
            set_error("occlusion min-cut did not converge on the device (set SLOWFLOW_GPU_HOST_MINCUT=1 to use the host solver)");
            return SFGPU_ERR_CUDA;
        }
        const int done = L.work->loop_host->outer_done;
        c->mt_stats.outer_iterations += done;
        c->mt_stats.pixel_outer_iterations += (long long)done * g.W * g.H;
        c->mt_stats.sor_calls += done;
        if (done > 0) { // (niter_outer == 0 leaves the previous level's value, like the reference's member variable)
            avg_change[0] = L.work->loop_host->avg_change[0];
            avg_change[1] = L.work->loop_host->avg_change[1];
        }
        // (prof_acc's launch / pixel counters were accumulated per QUEUED iteration; the event times are of what really ran)
        SF_CUDA(cudaGetLastError());
        return SFGPU_OK;
    }
    for (int alter = 0; alter < p->niter_alter; alter++) {
        warp_all(L); // :266
        if (alter > 0 && p->occlusion_reasoning && !L.one_direction) { // :269-272
            int rc = optimize_occ(L);
            if (rc != SFGPU_OK) return rc;
        }
        for (int outer = 0; outer < p->niter_outer; outer++) {
            if (outer > 0) warp_all(L); // :289-290
            c->mt_stats.outer_iterations++;
            c->mt_stats.pixel_outer_iterations += (long long)g.W * g.H;
            int cur = 0;
            bool broke_inner = false;
            int inner_done = 0;
            for (int inner = 0; inner < p->niter_inner; inner++) {
                const bool first = (inner == 0);
                const float *uu = first ? L.wx : L.uu, *vv = first ? L.wy : L.vv; // uu == wx at the start of an outer iteration
                float *du_cur = A + (size_t)(cur ? SP_DUB : SP_DUA) * P, *dv_cur = A + (size_t)(cur ? SP_DVB : SP_DVA) * P;
                if (!first) { // :329-330 old_du = du
                    SF_CUDA(cudaMemcpyAsync(L.odu, du_cur, P * sizeof(float), cudaMemcpyDeviceToDevice, st));
                    SF_CUDA(cudaMemcpyAsync(L.odv, dv_cur, P * sizeof(float), cudaMemcpyDeviceToDevice, st));
                }
                launch_mt_system(L, sys, g, uu, vv, first ? nullptr : du_cur, first ? nullptr : dv_cur, A);
                int rc = run_sor(c, p->niter_solver, p->sor_omega, &cur, first); // :368
                if (rc != SFGPU_OK) return rc;
                c->mt_stats.sor_calls++;
                inner_done = inner + 1;
                const float *ndu = A + (size_t)(cur ? SP_DUB : SP_DUA) * P, *ndv = A + (size_t)(cur ? SP_DVB : SP_DVA) * P;
                const bool last_possible = (inner == p->niter_inner - 1);
                // :371-399; when this is certainly the last inner iteration the outer update (:412-429) is fused in
                k_mt_update<<<ugrid, dim3(32, 8), 0, st>>>(g, L.wx, L.wy, ndu, ndv, first ? nullptr : L.odu, first ? nullptr : L.odv,
                                                           last_possible ? nullptr : L.uu, last_possible ? nullptr : L.vv,
                                                           last_possible ? 1 : 0, L.work->part_dev);
                c->prof_acc.kernel_launches++;
                double sums[4];
                rc = read_partials(L, ugrid, sums);
                if (rc != SFGPU_OK) return rc;
                const float ch_du = (float)(sums[0] * inv_n), ch_dv = (float)(sums[1] * inv_n);
                if (last_possible) {
                    avg_change[0] = (float)(sums[2] * inv_n);
                    avg_change[1] = (float)(sums[3] * inv_n);
                } else if (std::max(ch_du, ch_dv) < p->thres_inner) { // :407-408
                    broke_inner = true;
                    break;
                }
            }
            if (p->niter_inner <= 0) avg_change[0] = avg_change[1] = 0.f;
            else if (broke_inner || inner_done < p->niter_inner) {
                // left the inner loop early: uu, vv hold wx + du; do the outer update now (:412-429)
                const float *ndu = A + (size_t)(cur ? SP_DUB : SP_DUA) * P, *ndv = A + (size_t)(cur ? SP_DVB : SP_DVA) * P;
                k_mt_update<<<ugrid, dim3(32, 8), 0, st>>>(g, L.wx, L.wy, ndu, ndv, nullptr, nullptr, nullptr, nullptr, 1,
                                                           L.work->part_dev);
                c->prof_acc.kernel_launches++;
                double sums[4];
                int rc = read_partials(L, ugrid, sums);
                if (rc != SFGPU_OK) return rc;
                avg_change[0] = (float)(sums[2] * inv_n);
                avg_change[1] = (float)(sums[3] * inv_n);
            }
            if (std::max(avg_change[0], avg_change[1]) < p->thres_outer) break; // :436-437
        }
    }
    if (L.cut_pending) {
        SF_CUDA(cudaStreamSynchronize(st));
        if (device_cut_status(c->cut)[0] != 0 || device_cut_status(c->cut)[3] != 0) {
            set_error("occlusion min-cut did not converge on the device (set SLOWFLOW_GPU_HOST_MINCUT=1 to use the host solver)");
            return SFGPU_ERR_CUDA;
        }
    }
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

} // namespace sf

// ------------------------------------------------------------------------------------------ ABI
extern "C" {

void sf_mt_params_default(sf_mt_params_t *p) { // slow_flow.cpp:64-128 (setDefault)
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->S = 2; p->layers = 1; p->p_scale = 0.9f;
    p->alpha = 4.0f; p->gamma = 6.0f; p->delta = 1.0f;
    p->dataterm = 1; p->smoothing = 1; p->one_direction = 0;
    for (int a = 0; a < SF_MT_MAX_REF; a++) { p->rho[a] = 1.0f; p->omega[a] = 1.0f; }
    p->rho[0] = 1.0f; p->rho[1] = 1.0f; p->omega[0] = 0.0f; p->omega[1] = 2.0f;
    p->robust_color = 1; p->robust_color_eps = 0.001f; p->robust_color_truncation = 0.5f;
    p->robust_grad = -1; p->robust_grad_eps = 0.001f; p->robust_grad_truncation = 0.5f;
    p->robust_reg = 1; p->robust_reg_eps = 0.001f; p->robust_reg_truncation = 0.5f;
    p->niter_alter = 10; p->niter_outer = 10; p->niter_inner = 1; p->niter_solver = 30; p->niter_graphc = 10;
    p->thres_outer = 1e-5f; p->thres_inner = 1e-5f; p->sor_omega = 1.9f;
    p->occlusion_reasoning = 1; p->occlusion_penalty = 0.1f; p->occlusion_alpha = 0.1f;
    p->graphcut_int_terms = 0; p->hbit = 1;
    for (int k = 0; k < 3; k++) { p->img_norm_avg[k] = 0.0f; p->img_norm_std[k] = 1.0f; }
}

int sfgpu_grid_mincut(int w, int h, const float *d0, const float *d1, float alpha, int int_terms, int *labels) {
    if (w <= 0 || h <= 0 || !d0 || !d1 || !labels) {
        set_error("sfgpu_grid_mincut: bad argument");
        return SFGPU_ERR_ARG;
    }
    const size_t n = (size_t)w * h;
    std::vector<SinkForestCut::cap_t> tr(n);
    for (size_t p = 0; p < n; p++) tr[p] = occ_quantise_host((double)d1[p], int_terms != 0) - occ_quantise_host((double)d0[p], int_terms != 0);
    SinkForestCut cut;
    cut.solve(w, h, tr.data(), occ_quantise_host((double)alpha, int_terms != 0));
    for (size_t p = 0; p < n; p++) labels[p] = cut.label((int)p);
    return SFGPU_OK;
}

int sfgpu_grid_mincut_dev(sfgpu_ctx *c, int w, int h, const float *d0, const float *d1, float alpha, int int_terms, int *labels,
                          int stats[2]) {
    if (!c || w <= 0 || h <= 0 || !d0 || !d1 || !labels) {
        set_error("sfgpu_grid_mincut_dev: bad argument");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(c->device));
    const size_t n = (size_t)w * h;
    std::vector<long long> tr(n);
    for (size_t p = 0; p < n; p++) tr[p] = occ_quantise_host((double)d1[p], int_terms != 0) - occ_quantise_host((double)d0[p], int_terms != 0);
    long long *tr_dev = nullptr;
    SF_CUDA(cudaMalloc(&tr_dev, n * sizeof(long long)));
    std::vector<unsigned char> lab(n);
    int rc = SFGPU_OK;
    if (!cuda_ok(cudaMemcpyAsync(tr_dev, tr.data(), n * sizeof(long long), cudaMemcpyHostToDevice, c->stream), "h2d")) rc = SFGPU_ERR_CUDA;
    if (rc == SFGPU_OK) rc = device_grid_mincut(c, c->cut, w, h, tr_dev, (long long)occ_quantise_host((double)alpha, int_terms != 0), nullptr, 0);
    if (rc == SFGPU_OK && !cuda_ok(cudaMemcpyAsync(lab.data(), device_cut_labels(c->cut), n, cudaMemcpyDeviceToHost, c->stream), "d2h")) rc = SFGPU_ERR_CUDA;
    if (rc == SFGPU_OK && !cuda_ok(cudaStreamSynchronize(c->stream), "min-cut")) rc = SFGPU_ERR_CUDA;
    cudaFree(tr_dev);
    if (rc != SFGPU_OK) return rc;
    const int *st = device_cut_status(c->cut);
    if (stats) { stats[0] = st[1]; stats[1] = st[2]; }
    if (st[0] != 0) {
        set_error("sfgpu_grid_mincut_dev: the solver hit its pass bound");
        return SFGPU_ERR_CUDA;
    }
    for (size_t p = 0; p < n; p++) labels[p] = lab[p];
    c->prof_acc.kernel_launches++;
    return SFGPU_OK;
}

int sfgpu_get_mt_stats(sfgpu_ctx *c, sfgpu_mt_stats_t *out) {
    if (!c || !out) return SFGPU_ERR_ARG;
    *out = c->mt_stats;
    return SFGPU_OK;
}

int sfgpu_normalize(sfgpu_ctx *c, color_image_t *const *seq, int F, sf_mt_params_t *params) {
    if (!c || !seq || F < 1 || !params) {
        set_error("sfgpu_normalize: bad argument");
        return SFGPU_ERR_ARG;
    }
    Geom g;
    if (!arg_geom("sfgpu_normalize: ", "seq[0]", seq[0], g)) return SFGPU_ERR_ARG;
    for (int f = 1; f < F; f++)
        if (!arg_is("sfgpu_normalize: ", "seq[" + std::to_string(f) + "]", seq[f], g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t P = g.plane();
    // Short sequences (a window) stay resident between the two passes; long ones (a whole high-speed sequence, as the
    // sharded driver normalises it) are streamed through ONE frame-sized buffer twice, so device memory stays bounded.
    size_t resident_limit = (size_t)2 << 30;
    if (const char *e = getenv("SLOWFLOW_GPU_NORMALIZE_RESIDENT_BYTES")) resident_limit = (size_t)strtoull(e, nullptr, 10); // tests
    const bool resident = (size_t)F * 3 * P * sizeof(float) <= resident_limit;
    const size_t fstride = resident ? 3 * P : 0;
    const int nblk = std::min(g.H, 592);
    struct Bufs { // freed on every path
        float *dev = nullptr;
        double *dsum = nullptr;
        ~Bufs() { if (dev) cudaFree(dev); if (dsum) cudaFree(dsum); }
    } b;
    SF_CUDA(cudaMalloc(&b.dev, (resident ? (size_t)F : 1) * 3 * P * sizeof(float)));
    SF_CUDA(cudaMalloc(&b.dsum, (size_t)F * nblk * 6 * sizeof(double)));
    float *dev = b.dev;
    double *dsum = b.dsum;
    for (int f = 0; f < F; f++) {
        SF_CUDA(cudaMemcpyAsync(dev + (size_t)f * fstride, seq[f]->c1, 3 * P * sizeof(float), cudaMemcpyHostToDevice, st));
        k_norm_sums<<<nblk, 256, 0, st>>>(g, dev + (size_t)f * fstride, dsum + (size_t)f * nblk * 6);
    }
    SF_CUDA(cudaGetLastError());
    std::vector<double> hs((size_t)F * nblk * 6);
    SF_CUDA(cudaMemcpyAsync(hs.data(), dsum, hs.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    double avg[3] = {0, 0, 0}, sd[3] = {0, 0, 0};
    const double n = (double)g.H * g.W;
    for (int f = 0; f < F; f++) {
        double fs[6] = {0, 0, 0, 0, 0, 0};
        for (int blk = 0; blk < nblk; blk++)
            for (int k = 0; k < 6; k++) fs[k] += hs[((size_t)f * nblk + blk) * 6 + k];
        for (int k = 0; k < 3; k++) { avg[k] += fs[k] / n; sd[k] += fs[3 + k] / n; }
    }
    for (int k = 0; k < 3; k++) {
        avg[k] /= F;
        sd[k] = sqrt((sd[k] / F) - avg[k] * avg[k]) / 255.0f; // :48-51
    }
    for (int f = 0; f < F; f++) {
        if (!resident) SF_CUDA(cudaMemcpyAsync(dev, seq[f]->c1, 3 * P * sizeof(float), cudaMemcpyHostToDevice, st));
        k_norm_apply<<<grid2d(g.W, g.H), dim3(32, 8), 0, st>>>(g, dev + (size_t)f * fstride, avg[0], avg[1], avg[2], sd[0], sd[1], sd[2]);
        SF_CUDA(cudaMemcpyAsync(seq[f]->c1, dev + (size_t)f * fstride, 3 * P * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    SF_CUDA(cudaGetLastError());
    SF_CUDA(cudaStreamSynchronize(st));
    for (int k = 0; k < 3; k++) {
        // the reference publishes the values through a stringstream with 6 significant digits (:72-84)
        char buf[64];
        snprintf(buf, sizeof(buf), "%.6g", avg[k]);
        params->img_norm_avg[k] = (float)atof(buf);
        snprintf(buf, sizeof(buf), "%.6g", sd[k]);
        params->img_norm_std[k] = (float)atof(buf);
    }
    c->prof_acc.kernel_launches += 2 * F;
    return SFGPU_OK;
}

// ---- input side of a window (SURVEY 8f rank 3): what slow_flow.cpp does to every frame before the solver sees it
int sfgpu_prescale_size(int width, int height, float scale, int *out_width, int *out_height) {
    if (width <= 0 || height <= 0 || !(scale > 0.0f) || !out_width || !out_height) {
        set_error("sfgpu_prescale_size: bad argument");
        return SFGPU_ERR_ARG;
    }
    // cv::resize(src, dst, Size(0,0), fx, fy): dsize = (cvRound(cols*fx), cvRound(rows*fy)), round half to even
    *out_width = (int)lrint((double)width * (double)scale);
    *out_height = (int)lrint((double)height * (double)scale);
    if (*out_width < 1 || *out_height < 1) {
        set_error("sfgpu_prescale_size: scaled image is empty");
        return SFGPU_ERR_ARG;
    }
    return SFGPU_OK;
}

int sfgpu_prescale(sfgpu_ctx *c, color_image_t *dst, const color_image_t *src, float scale) {
    if (!c) {
        set_error("sfgpu_prescale: null argument");
        return SFGPU_ERR_ARG;
    }
    Geom gs;
    if (!arg_geom("sfgpu_prescale: ", "src", src, gs)) return SFGPU_ERR_ARG;
    int dw = 0, dh = 0;
    int rc = sfgpu_prescale_size(gs.W, gs.H, scale, &dw, &dh);
    if (rc != SFGPU_OK) return rc;
    const Geom gd = make_geom(dw, dh); // what sfgpu_prescale_size reports
    if (!arg_is("sfgpu_prescale: ", "dst", dst, gd)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t Ps = gs.plane(), Pd = gd.plane();
    rc = c->ensure_io(9 * Ps + 3 * Pd);
    if (rc != SFGPU_OK) return rc;
    float *d_src = c->io, *d_tmp = c->io + 3 * Ps, *d_blur = c->io + 6 * Ps, *d_dst = c->io + 9 * Ps;
    SF_CUDA(cudaMemcpyAsync(d_src, src->c1, 3 * Ps * sizeof(float), cudaMemcpyHostToDevice, st));
    // GaussianBlur(img, img, Size(), 1/sqrt(2*scale), ..., BORDER_REPLICATE) then resize(..., scale, scale, INTER_LINEAR)
    // (slow_flow.cpp:539-542); the mapping of a resize by factor uses 1/fx, not the ratio of the rounded sizes
    const double sigma = 1.0 / sqrt((double)(2.0f * scale));
    const BlurTaps taps = make_taps(sigma);
    launch_blur(st, gs, d_src, d_tmp, d_blur, taps, 3);
    k_resize<<<resize_grid(gd), dim3(32, 8), 0, st>>>(gs, d_blur, gd, d_dst, 1.0 / (double)scale, 1.0 / (double)scale, 1.0f, 3);
    c->prof_acc.kernel_launches += 3;
    SF_CUDA(cudaMemcpyAsync(dst->c1, d_dst, 3 * Pd * sizeof(float), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    return SFGPU_OK;
}

int sfgpu_raw_weighting(sfgpu_ctx *c, color_image_t *weights, int red_x, int red_y, float weight) {
    Geom g;
    if (!c) {
        set_error("sfgpu_raw_weighting: bad argument");
        return SFGPU_ERR_ARG;
    }
    if (!arg_geom("sfgpu_raw_weighting: ", "weights", weights, g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t P = g.plane();
    int rc = c->ensure_io(3 * P);
    if (rc != SFGPU_OK) return rc;
    // the reference only writes the valid columns (utils/utils.cpp:1340-1372); the stride padding keeps the caller's values
    SF_CUDA(cudaMemcpyAsync(c->io, weights->c1, 3 * P * sizeof(float), cudaMemcpyHostToDevice, st));
    k_raw_weights<<<grid2d(g.W, g.H), dim3(32, 8), 0, st>>>(g, c->io, red_x, red_y, fminf(fmaxf(weight, 0.0f), 3.0f));
    c->prof_acc.kernel_launches++;
    SF_CUDA(cudaMemcpyAsync(weights->c1, c->io, 3 * P * sizeof(float), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    return SFGPU_OK;
}

// ---- operator twins of one level: the production kernels on uploaded level frames and flow
extern "C++" {
struct MtTwin { // device planes of one level and the LevelCtx the production helpers take
    float *base = nullptr;
    LevelCtx L{};
    ~MtTwin() { if (base) cudaFree(base); }
};

// checks the level arguments, uploads frames / flow / occlusion plane / channel weights and warps every frame
// (plus the reference frame's derivative planes when the all-terms pass is the data pass); `extra` planes follow
static int mt_twin_level(sfgpu_ctx *c, const char *at, const color_image_t *const *im, const image_t *wx, const image_t *wy,
                         const image_t *occ, const color_image_t *channel_w, const sf_mt_params_t *p, bool one_direction, int extra,
                         MtTwin &t, MtSystemTerms *sys, float **extra_planes) {
    const std::string who(at);
    if (!c || !im || !p) {
        set_error(who + "null argument");
        return SFGPU_ERR_ARG;
    }
    const int ref = p->S - 1, F = 2 * ref + 1;
    if (ref < 1 || ref > SF_MT_MAX_REF || p->smoothing < 0 || p->smoothing > 1) {
        set_error(who + "slow_flow_S or slow_flow_smoothing out of range");
        return SFGPU_ERR_ARG;
    }
    Geom g;
    if (!arg_geom(who, "wx", wx, g) || !arg_is(who, "wy", wy, g) || (occ && !arg_is(who, "occ", occ, g)) ||
        (channel_w && !arg_is(who, "channel_w", channel_w, g)))
        return SFGPU_ERR_ARG;
    for (int f = 0; f < F; f++)
        if (!arg_is(who, "im[" + std::to_string(f) + "]", im[f], g)) return SFGPU_ERR_ARG;
    if (g.W < 5 || g.H < 5) {
        set_error(who + "images smaller than 5x5 are not supported");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t P = g.plane();
    const bool fused = c->mt_data_variant == 0;
    const size_t planes = (size_t)F * 3 /*frames*/ + (size_t)F * 3 /*warped*/ + F /*masks*/ + (fused ? (size_t)F * 15 : 0) +
                          4 /*wx wy occ dpsis*/ + 3 /*channel weights*/ + extra;
    SF_CUDA(cudaMalloc(&t.base, planes * P * sizeof(float)));
    float *ptr = t.base;
    auto take = [&](size_t n) { float *r = ptr; ptr += n * P; return r; };
    LevelCtx &L = t.L;
    L.c = c; L.p = p; L.g = g; L.ref = ref;
    L.one_direction = one_direction;
    L.alpha = p->alpha;
    L.gamma_over3 = p->gamma / 3.0f;
    L.delta_over3 = p->delta / 3.0f;
    L.pc = make_penalty(p->robust_color, p->robust_color_eps, p->robust_color_truncation);
    L.pg = (p->robust_grad >= 0) ? make_penalty(p->robust_grad, p->robust_grad_eps, p->robust_grad_truncation) : L.pc;
    L.preg = make_penalty(p->robust_reg, p->robust_reg_eps, p->robust_reg_truncation);
    L.frames.assign(F, nullptr); L.warped.assign(F, nullptr); L.masks.assign(F, nullptr); L.derivs.assign(F, nullptr);
    for (int f = 0; f < F; f++) {
        L.frames[f] = take(3);
        SF_CUDA(cudaMemcpyAsync(L.frames[f], im[f]->c1, 3 * P * sizeof(float), cudaMemcpyHostToDevice, st));
        L.warped[f] = (f == ref) ? L.frames[f] : take(3);
        L.masks[f] = take(1);
        if (fused) L.derivs[f] = take(15);
    }
    L.fused_terms = fused;
    L.wx = take(1); L.wy = take(1); L.occ = take(1); L.dpsis = take(1);
    L.d0 = L.d1 = nullptr; L.uu = L.vv = L.odu = L.odv = nullptr;
    SF_CUDA(cudaMemcpyAsync(L.wx, wx->data, P * sizeof(float), cudaMemcpyHostToDevice, st));
    SF_CUDA(cudaMemcpyAsync(L.wy, wy->data, P * sizeof(float), cudaMemcpyHostToDevice, st));
    if (occ) SF_CUDA(cudaMemcpyAsync(L.occ, occ->data, P * sizeof(float), cudaMemcpyHostToDevice, st));
    float *chw = take(3);
    L.chw = nullptr;
    L.chw_pstride = P;
    if (channel_w) {
        SF_CUDA(cudaMemcpyAsync(chw, channel_w->c1, 3 * P * sizeof(float), cudaMemcpyHostToDevice, st));
        L.chw = chw;
    }
    L.work = nullptr;
    *extra_planes = take(extra);
    warp_all(L);
    if (sys) {
        launch_dpsis_weight(st, g, L.frames[ref], L.dpsis, 5.0f, p->img_norm_avg, p->img_norm_std, p->hbit ? 65535.0f : 255.0f);
        mt_system_setup(L, *sys);
    }
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}
} // extern "C++"

int sfgpu_mt_system(sfgpu_ctx *c, image_t *a11, image_t *a12, image_t *a22, image_t *b1, image_t *b2, image_t *psi_h, image_t *psi_v,
                    const color_image_t *const *im, const image_t *wx, const image_t *wy, const image_t *du, const image_t *dv,
                    const image_t *occ, const color_image_t *channel_w, const sf_mt_params_t *p) {
    const char *at = "sfgpu_mt_system: ";
    if ((du == nullptr) != (dv == nullptr) || !occ) {
        set_error("sfgpu_mt_system: du and dv must both be given or both be null, occ is required");
        return SFGPU_ERR_ARG;
    }
    Geom g;
    if (!arg_geom(at, "wx", wx, g) || (du && (!arg_is(at, "du", du, g) || !arg_is(at, "dv", dv, g))))
        return SFGPU_ERR_ARG;
    image_t *outs[7] = {a11, a12, a22, b1, b2, psi_h, psi_v}; // arena order SP_A11 .. SP_PV
    const char *names[7] = {"a11", "a12", "a22", "b1", "b2", "psi_h", "psi_v"};
    for (int k = 0; k < 7; k++)
        if (!arg_is(at, names[k], outs[k], g)) return SFGPU_ERR_ARG;
    MtTwin t;
    MtSystemTerms sys;
    float *A = nullptr;
    int rc = mt_twin_level(c, at, im, wx, wy, occ, channel_w, p, p && p->one_direction != 0, 11, t, &sys, &A);
    if (rc != SFGPU_OK) return rc;
    cudaStream_t st = c->stream;
    const size_t P = g.plane();
    float *uu = A + 7 * P, *vv = A + 8 * P, *ddu = A + 9 * P, *ddv = A + 10 * P;
    const float *su = t.L.wx, *sv = t.L.wy;
    std::vector<float> hu, hv;
    if (du) { // uu = wx + du (variational_mt.cpp:397-398)
        hu.resize(P); hv.resize(P);
        for (size_t k = 0; k < P; k++) { hu[k] = wx->data[k] + du->data[k]; hv[k] = wy->data[k] + dv->data[k]; }
        SF_CUDA(cudaMemcpyAsync(ddu, du->data, P * sizeof(float), cudaMemcpyHostToDevice, st));
        SF_CUDA(cudaMemcpyAsync(ddv, dv->data, P * sizeof(float), cudaMemcpyHostToDevice, st));
        SF_CUDA(cudaMemcpyAsync(uu, hu.data(), P * sizeof(float), cudaMemcpyHostToDevice, st));
        SF_CUDA(cudaMemcpyAsync(vv, hv.data(), P * sizeof(float), cudaMemcpyHostToDevice, st));
        su = uu; sv = vv;
    }
    SF_CUDA(cudaMemsetAsync(A, 0xff, 7 * P * sizeof(float), st)); // NaN pattern: every element must be written
    launch_mt_system(t.L, sys, g, su, sv, du ? ddu : nullptr, du ? ddv : nullptr, A);
    for (int k = 0; k < 7; k++)
        SF_CUDA(cudaMemcpyAsync(outs[k]->data, A + (size_t)k * P, P * sizeof(float), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_mt_occ_costs(sfgpu_ctx *c, image_t *d0, image_t *d1, const color_image_t *const *im, const image_t *wx, const image_t *wy,
                       const sf_mt_params_t *p) {
    const char *at = "sfgpu_mt_occ_costs: ";
    Geom g;
    if (!arg_geom(at, "wx", wx, g) || !arg_is(at, "d0", d0, g) || !arg_is(at, "d1", d1, g)) return SFGPU_ERR_ARG;
    MtTwin t;
    float *D = nullptr;
    int rc = mt_twin_level(c, at, im, wx, wy, nullptr, nullptr, p, false, 2, t, nullptr, &D);
    if (rc != SFGPU_OK) return rc;
    cudaStream_t st = c->stream;
    const size_t P = g.plane();
    SF_CUDA(cudaMemsetAsync(D, 0xff, 2 * P * sizeof(float), st)); // NaN pattern: the kernel writes the W x H pixels only
    k_occ_costs<<<grid2d(g.W, g.H), dim3(32, 8), 0, st>>>(g, occ_args(t.L), D, D + P, nullptr, p->graphcut_int_terms != 0 ? 1 : 0);
    SF_CUDA(cudaMemcpyAsync(d0->data, D, P * sizeof(float), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaMemcpyAsync(d1->data, D + P, P * sizeof(float), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_variational_mt(sfgpu_ctx *c, image_t *wx, image_t *wy, const color_image_t *const *im,
                         const sf_mt_params_t *p, const color_image_t *channel_w, image_t *occlusions_out,
                         float avg_change_out[2]) {
    if (!c || !im || !p) {
        set_error("sfgpu_variational_mt: null argument");
        return SFGPU_ERR_ARG;
    }
    const int ref = p->S - 1, F = 2 * ref + 1;
    if (ref < 1 || ref > SF_MT_MAX_REF) {
        set_error("sfgpu_variational_mt: slow_flow_S out of range");
        return SFGPU_ERR_ARG;
    }
    if (p->smoothing < 0 || p->smoothing > 1) {
        set_error("sfgpu_variational_mt: slow_flow_smoothing >= 2 is not supported (reference bug, SURVEY Q6)");
        return SFGPU_ERR_UNSUPPORTED;
    }
    if (p->layers < 1 || (p->layers > 1 && !(p->p_scale > 0.f && p->p_scale < 1.f))) {
        set_error("sfgpu_variational_mt: bad pyramid parameters");
        return SFGPU_ERR_ARG;
    }
    const char *at = "sfgpu_variational_mt: ";
    Geom flow_g;
    if (!arg_geom(at, "wx", wx, flow_g) || !arg_is(at, "wy", wy, flow_g) || (channel_w && !arg_is(at, "channel_w", channel_w, flow_g)) ||
        (occlusions_out && occlusions_out->data && !arg_is(at, "occlusions_out", occlusions_out, flow_g)))
        return SFGPU_ERR_ARG;
    for (int f = 0; f < F; f++)
        if (!arg_is(at, "im[" + std::to_string(f) + "]", im[f], flow_g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    memset(&c->mt_stats, 0, sizeof(c->mt_stats));
    const double t_call = now_ms();
    if (avg_change_out) avg_change_out[0] = avg_change_out[1] = 0.f;

    // ---- pyramid geometry (variational_mt.cpp:583-652): floor((float)w * p_scale); a level is dropped when
    // the NEXT one would be <= order+1 = floor(3 sigma)+2 pixels (:647-651)
    const float sigma = 1.0f / sqrtf(2.0f * p->p_scale);
    const int order = (int)floorf(3.0f * sigma) + 1;
    std::vector<Geom> geoms;
    int L = p->layers;
    for (int l = 0; l < L; l++) {
        if (l == 0) geoms.push_back(flow_g);
        else geoms.push_back(make_geom((int)floorf((float)geoms[l - 1].W * p->p_scale), (int)floorf((float)geoms[l - 1].H * p->p_scale)));
        if (floorf((float)geoms[l].W * p->p_scale) <= order + 1 || floorf((float)geoms[l].H * p->p_scale) <= order + 1) {
            L = l;
            break;
        }
    }
    if (L == 0) return SFGPU_OK; // the reference computes nothing in this case
    geoms.resize(L);
    c->mt_stats.levels = L;

    // ---- device memory: frames of all levels + per-level work planes sized for level 0
    const Geom g0 = geoms[0];
    const size_t P0 = g0.plane();
    // with the frame cache (sfgpu_mt_frame_cache) the level-0 frames live in the cache's own device buffers
    const bool cached = !c->mt_cache.empty() && (int)c->mt_cache.size() >= F;
    size_t frame_floats = 0;
    for (int l = cached ? 1 : 0; l < L; l++) frame_floats += (size_t)F * 3 * geoms[l].plane();
    const size_t work_planes = (size_t)(F - 1) * 3 + (F - 1) + 2 /*wx wy*/ + 2 /*wx,wy of next level*/ + 2 /*uu vv*/ + 2 /*odu odv*/ + 1 /*dpsis*/ +
                               1 /*occ*/ + 2 /*d0 d1*/ + 3 /*blur tmp*/ + (channel_w ? 3 : 0) +
                               (c->mt_data_variant == 0 ? (size_t)F * 15 /*per-frame derivative planes*/ : 0);
    if (!c->mtw) c->mtw = new MtWork();
    MtWork &work = *c->mtw;
    {
        const int rcw = work.reserve(frame_floats + work_planes * P0, (size_t)((g0.W + 31) / 32) * 64 * 4, (size_t)g0.W * g0.H);
        if (rcw != SFGPU_OK) return rcw;
    }
    float *ptr = work.pool;
    std::vector<MtLevel> levels(L);
    std::vector<bool> frame_resident(F, false); // level-0 frame already on the device (cache hit)
    for (int l = 0; l < L; l++) {
        levels[l].g = geoms[l];
        if (l == 0 && cached) {
            // slot per frame: the one that holds this host buffer, else the least recently used slot no frame of this call has
            const unsigned long long now = ++c->mt_cache_clock;
            const size_t want = 3 * P0;
            if (c->mt_cache_slot_floats != want) { // first use, or another geometry: one pool for all slots
                SF_CUDA(cudaStreamSynchronize(st));
                if (c->mt_cache_pool) cudaFree(c->mt_cache_pool);
                c->mt_cache_pool = nullptr;
                c->mt_cache_slot_floats = 0;
                SF_CUDA(cudaMalloc(&c->mt_cache_pool, c->mt_cache.size() * want * sizeof(float)));
                c->mt_cache_slot_floats = want;
                for (size_t k = 0; k < c->mt_cache.size(); k++) {
                    c->mt_cache[k] = sfgpu_ctx::MtFrameSlot();
                    c->mt_cache[k].dev = c->mt_cache_pool + k * want;
                    c->mt_cache[k].floats = want;
                }
            }
            for (int f = 0; f < F; f++) {
                sfgpu_ctx::MtFrameSlot *slot = nullptr;
                for (auto &e : c->mt_cache)
                    if (e.host == (const void *)im[f]->c1 && e.floats == want && e.stamp != now) { slot = &e; frame_resident[f] = true; break; }
                if (!slot) {
                    for (auto &e : c->mt_cache)
                        if (e.stamp != now && (!slot || e.stamp < slot->stamp)) slot = &e;
                    slot->host = im[f]->c1;
                    c->mt_cache_misses++;
                } else {
                    c->mt_cache_hits++;
                }
                slot->stamp = now;
                levels[0].frames.push_back(slot->dev);
            }
            continue;
        }
        for (int f = 0; f < F; f++) { levels[l].frames.push_back(ptr); ptr += 3 * geoms[l].plane(); }
    }
    auto take = [&](size_t planes) { float *r = ptr; ptr += planes * P0; return r; };
    std::vector<float *> warped(F, nullptr), masks(F, nullptr);
    for (int f = 0; f < F; f++)
        if (f != ref) { warped[f] = take(3); masks[f] = take(1); }
    float *wxa = take(1), *wya = take(1), *wxb = take(1), *wyb = take(1);
    float *uu = take(1), *vv = take(1), *odu = take(1), *odv = take(1), *dpsis = take(1), *occ = take(1), *d0 = take(1), *d1 = take(1);
    float *blur_tmp = take(3);
    float *chw = channel_w ? take(3) : nullptr;
    std::vector<float *> derivs(F, nullptr);
    if (c->mt_data_variant == 0)
        for (int f = 0; f < F; f++) derivs[f] = take(15);

    // ---- upload
    {
        std::vector<HostCopy> up;
        for (int f = 0; f < F; f++)
            if (!frame_resident[f]) up.push_back(HostCopy{levels[0].frames[f], im[f]->c1, 3 * P0 * sizeof(float)});
        up.push_back(HostCopy{wxa, wx->data, P0 * sizeof(float)});
        up.push_back(HostCopy{wya, wy->data, P0 * sizeof(float)});
        if (chw) up.push_back(HostCopy{chw, channel_w->c1, 3 * P0 * sizeof(float)});
        const int rcu = host_copies(c, up, true); // pageable caller frames: multi-threaded staging (sf_hostcopy.cu)
        if (rcu != SFGPU_OK) return rcu;
    }

    // ---- pyramid: GaussianBlur(sigma) + resize per frame and level (:604-614)
    if (L > 1) {
        const BlurTaps taps = make_taps((double)sigma);
        for (int l = 1; l < L; l++) {
            const Geom gs = geoms[l - 1], gd = geoms[l];
            for (int f = 0; f < F; f++) {
                // vertical pass writes into the (not yet used) warp scratch of frame slot 0/1
                float *tmp2 = warped[ref == 0 ? 1 : 0];
                launch_blur(st, gs, levels[l - 1].frames[f], blur_tmp, tmp2, taps, 3);
                k_resize<<<resize_grid(gd), dim3(32, 8), 0, st>>>(gs, tmp2, gd, levels[l].frames[f], (double)gs.W / gd.W,
                                                                  (double)gs.H / gd.H, 1.0f, 3);
                c->prof_acc.kernel_launches += 3;
            }
        }
    }

    // ---- coarse-to-fine (:662-762)
    float *cur_x = wxa, *cur_y = wya, *oth_x = wxb, *oth_y = wyb;
    Geom cur_g = g0;
    if (L > 1) {
        const Geom gd = geoms[L - 1];
        const float fx = (1.0f * gd.W) / g0.W, fy = (1.0f * gd.H) / g0.H;
        k_resize<<<resize_grid(gd), dim3(32, 8), 0, st>>>(g0, cur_x, gd, oth_x, (double)g0.W / gd.W, (double)g0.H / gd.H, fx, 1);
        k_resize<<<resize_grid(gd), dim3(32, 8), 0, st>>>(g0, cur_y, gd, oth_y, (double)g0.W / gd.W, (double)g0.H / gd.H, fy, 1);
        std::swap(cur_x, oth_x);
        std::swap(cur_y, oth_y);
        cur_g = gd;
        c->prof_acc.kernel_launches += 2;
    }
    float avg_change[2] = {0.f, 0.f};
    int rc = c->ensure_workspace(g0); // size the level workspace once for the finest level
    if (cudaStreamSynchronize(st) == cudaSuccess) c->mt_stats.setup_ms = now_ms() - t_call;
    for (int l = L - 1; l >= 0 && rc == SFGPU_OK; l--) {
        const Geom g = geoms[l];
        if (l < L - 1) { // up-sample the flow of level l+1 and scale the vectors (:687-722)
            const float fx = (1.0f * g.W) / cur_g.W, fy = (1.0f * g.H) / cur_g.H;
            k_resize<<<resize_grid(g), dim3(32, 8), 0, st>>>(cur_g, cur_x, g, oth_x, (double)cur_g.W / g.W, (double)cur_g.H / g.H, fx, 1);
            k_resize<<<resize_grid(g), dim3(32, 8), 0, st>>>(cur_g, cur_y, g, oth_y, (double)cur_g.W / g.W, (double)cur_g.H / g.H, fy, 1);
            std::swap(cur_x, oth_x);
            std::swap(cur_y, oth_y);
            cur_g = g;
            c->prof_acc.kernel_launches += 2;
        }
        rc = c->ensure_workspace(g);
        if (rc != SFGPU_OK) break;
        LevelCtx Lc;
        Lc.c = c; Lc.p = p; Lc.g = g; Lc.ref = ref;
        Lc.one_direction = p->one_direction != 0;
        Lc.alpha = p->alpha;
        Lc.gamma_over3 = p->gamma / 3.0f;
        Lc.delta_over3 = p->delta / 3.0f;
        Lc.pc = make_penalty(p->robust_color, p->robust_color_eps, p->robust_color_truncation);
        Lc.pg = (p->robust_grad >= 0) ? make_penalty(p->robust_grad, p->robust_grad_eps, p->robust_grad_truncation) : Lc.pc; // Q8
        Lc.preg = make_penalty(p->robust_reg, p->robust_reg_eps, p->robust_reg_truncation);
        Lc.frames = levels[l].frames;
        Lc.warped = warped;
        Lc.warped[ref] = levels[l].frames[ref];
        Lc.masks = masks;
        Lc.derivs = derivs;
        Lc.fused_terms = c->mt_data_variant == 0;
        Lc.wx = cur_x; Lc.wy = cur_y; Lc.uu = uu; Lc.vv = vv; Lc.odu = odu; Lc.odv = odv;
        Lc.dpsis = dpsis; Lc.occ = occ; Lc.d0 = d0; Lc.d1 = d1;
        Lc.chw = chw; Lc.chw_pstride = P0;
        Lc.work = &work;
        rc = compute_one_level(Lc, avg_change);
    }
    if (rc != SFGPU_OK) return rc;

    {
        std::vector<HostCopy> down;
        down.push_back(HostCopy{cur_x, wx->data, P0 * sizeof(float)});
        down.push_back(HostCopy{cur_y, wy->data, P0 * sizeof(float)});
        if (occlusions_out && occlusions_out->data)
            down.push_back(HostCopy{occ, occlusions_out->data, P0 * sizeof(float)});
        const int rcd = host_copies(c, down, false);
        if (rcd != SFGPU_OK) return rcd;
    }
    SF_CUDA(cudaStreamSynchronize(st));
    if (avg_change_out) { avg_change_out[0] = avg_change[0]; avg_change_out[1] = avg_change[1]; }
    c->mt_stats.total_ms = now_ms() - t_call;
    return SFGPU_OK;
}

} // extern "C"
