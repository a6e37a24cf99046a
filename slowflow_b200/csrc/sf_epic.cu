// sf_epic.cu -- EPIC sparse-to-dense interpolation on the device (SURVEY 8f rank 4): the step that produces the initial
// flow variational() refines (epicflow.cpp:125, adaptiveFR.cpp:568, slow_flow.cpp:819,979).  Replaces
//   epic()                          epic_flow_extended/epic.cpp:147-234  (+ rectify / saliency / consistency filters :13-127)
//   dist_trf_nnfield_subset()       epic_aux.cpp:350-401: geodesic distance transform with label propagation (:91-182),
//                                   neighbourhood graph of the seeds (:186-288), k nearest seeds on that graph (:47-85)
//   fit_nadarayawatson / fit_localaffine / apply_*   epic_aux.cpp:404-492
//   saliency()                      image.c:728-790
//
// What runs where.  Everything image-sized or per-seed runs on the GPU; the host only compacts the (small) match list
// after the two filters, in the reference's order.
//   * Distance transform: the reference sweeps the image in raster order in four directions (Gauss-Seidel: a pixel uses
//     the already updated left / upper neighbour of the SAME sweep).  The sweeps are reproduced exactly -- same operations,
//     same order per pixel, no FMA contraction -- as a pipeline of row strips: a warp owns 32 rows (lane = row) and
//     marches along the sweep direction with its wavefront in registers (left neighbour = own previous result, upper
//     neighbour = shuffle), the strip below follows ~70 columns behind on the published last row of the strip above.
//     The data-dependent number of sweeps (epic_aux.cpp:170-178) is decided on the device: all 40 sweep kernels are queued,
//     the ones beyond end_iter return at once.
//   * Neighbourhood graph: every label border emits (row, col, d) in both directions; radix sort by (row, col) and a
//     segmented minimum (CUB) give the CSR matrix in the reference's order (sorted by row, then column).
//   * k nearest seeds: one warp per seed runs the reference's Dijkstra with ITS heap discipline (libstdc++'s push_heap /
//     pop_heap, so ties pop in the same order); heap in shared memory, tentative distances in a per-warp global array.
//   * Locally-weighted affine fit: the reference hands a 2(nn+4) x 6 system to LAPACK's sgels; the system decouples into
//     two weighted 3-parameter fits with one design matrix, solved here per seed by normal equations in DOUBLE with
//     coordinates centred on the seed (parity unpinned at this call anyway: LAPACK is not part of the reference tree).
#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include <stdlib.h>

#include <string.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>

#include "sf_context.cuh"
#include "sf_stencil.cuh"

namespace sf {

constexpr int DT_TILE = 32;
constexpr int DT_MAX_SWEEPS = 40;
constexpr unsigned EPIC_UNSEEN = 0x7F7F7F7Fu; // memset(…, 0x7F, …) pattern of the reference: 3.39e38f

// ------------------------------------------------------------------------------------------ saliency (image.c:728-790)
struct ConvTaps { int order; float c[17]; }; // c[order + k] = weight of src[i + k]
// The image-sized kernels of a call cover all its items at once: blockIdx.z is the item, and the item's planes lie zs floats
// after those of the item before it (k_conv_any: src_zs in its source, which may be another buffer).
__global__ void __launch_bounds__(256) k_conv_any(Geom g, const float *__restrict__ src, float *__restrict__ dst, ConvTaps t, int vertical,
                                                  int planes, size_t zs, size_t src_zs) {
    const int i = blockIdx.x * 32 + threadIdx.x, j = blockIdx.y * 8 + threadIdx.y;
    if (i >= g.W || j >= g.H) return;
    const size_t P = g.plane();
    src += blockIdx.z * src_zs;
    dst += blockIdx.z * zs;
    for (int c = 0; c < planes; c++) {
        const float *s = src + c * P;
        float sum = 0.0f;
        for (int k = -t.order; k <= t.order; k++) {
            const float v = vertical ? s[(size_t)clampi(j + k, 0, g.H - 1) * g.S + i] : s[(size_t)j * g.S + clampi(i + k, 0, g.W - 1)];
            sum += t.c[t.order + k] * v;
        }
        dst[c * P + (size_t)j * g.S + i] = sum;
    }
}
__global__ void __launch_bounds__(256) k_autocorr(Geom g, const float *__restrict__ ix, const float *__restrict__ iy, float *__restrict__ xx,
                                                  float *__restrict__ xy, float *__restrict__ yy, size_t zs) {
    const int i = blockIdx.x * 32 + threadIdx.x, j = blockIdx.y * 8 + threadIdx.y;
    if (i >= g.W || j >= g.H) return;
    const size_t P = g.plane(), o = (size_t)j * g.S + i + blockIdx.z * zs;
    const float a0 = ix[o], a1 = ix[o + P], a2 = ix[o + 2 * P], b0 = iy[o], b1 = iy[o + P], b2 = iy[o + 2 * P];
    xx[o] = a0 * a0 + a1 * a1 + a2 * a2;
    xy[o] = a0 * b0 + a1 * b1 + a2 * b2;
    yy[o] = b0 * b0 + b1 * b1 + b2 * b2;
}
__global__ void __launch_bounds__(256) k_min_eig(Geom g, const float *__restrict__ xx, const float *__restrict__ xy, const float *__restrict__ yy,
                                                 float *__restrict__ out, size_t zs) {
    const int i = blockIdx.x * 32 + threadIdx.x, j = blockIdx.y * 8 + threadIdx.y;
    if (i >= g.W || j >= g.H) return;
    const size_t o = (size_t)j * g.S + i + blockIdx.z * zs;
    const float t = 0.5f * (xx[o] + yy[o]);
    out[o] = sqrtf(fmaxf(0.0f, t - sqrtf(fmaxf(0.0f, t * t + xy[o] * xy[o] - xx[o] * yy[o]))));
}
static ConvTaps gaussian_taps(float sigma) { // gaussian_filter + convolution_new(even) (image.c:310-398)
    ConvTaps t;
    memset(&t, 0, sizeof(t));
    int order = (int)floor(3 * sigma) + 1;
    if (order == 0) order = 1;
    if (order > 8) order = 8;
    t.order = order;
    const float alpha = 1.0f / (2.0f * sigma * sigma);
    float sum = 0.0f;
    for (int i = -order; i <= order; i++) {
        t.c[order + i] = (float)exp(-i * i * alpha);
        sum += t.c[order + i];
    }
    for (int i = -order; i <= order; i++) t.c[order + i] /= sum;
    return t;
}

// ------------------------------------------------------------------------------------------ small per-match kernels
// pos: (x, y, item) per match; the item's plane lies item * zs floats after `plane`
__global__ void k_gather_plane(int n, const int *__restrict__ pos, Geom g, const float *__restrict__ plane, size_t zs, float *__restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = plane[(size_t)pos[3 * k + 2] * zs + (size_t)pos[3 * k + 1] * g.S + pos[3 * k]];
}
__global__ void k_fill_u32(size_t n, unsigned *__restrict__ dst, unsigned v) {
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x) dst[k] = v;
}
// The seeds of the n items of a call carry global ids: item k owns off[k] .. off[k+1]-1, in its own order, and label maps
// hold global ids.  So the keys of the border list sort by item, one CSR covers all seeds and no graph edge crosses items.
struct SeedItems {
    const int *item; // per seed: its item
    const int *off;  // per item: its first seed
    const int *nns;  // per item: neighbours searched (min(nn, its seeds))
};
// seeds onto the distance / label maps (W x H = N pixels per item): dmap[p] = cost[p]; of several seeds on one pixel the
// LAST one wins (the reference writes them in order, epic_aux.cpp:319-323; ids of one item keep its order)
__global__ void k_dt_seed_labels(int ns, const int *__restrict__ seeds, const int *__restrict__ item, int W, size_t N, int *__restrict__ labels) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < ns) atomicMax(labels + item[k] * N + (size_t)seeds[2 * k + 1] * W + seeds[2 * k], k);
}
__global__ void k_dt_seed_dist(int ns, const int *__restrict__ seeds, const int *__restrict__ item, int W, size_t N, const float *__restrict__ cost,
                               float *__restrict__ dmap) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < ns) {
        const size_t p = item[k] * N + (size_t)seeds[2 * k + 1] * W + seeds[2 * k];
        dmap[p] = cost[p];
    }
}

// ------------------------------------------------------------------------------------------ distance transform sweeps
struct DtCtrl { // one per item
    int end_iter;                   // sweeps with index > end_iter are skipped (epic_aux.cpp:170-178)
    int sweeps_run;
    unsigned maxdiff[DT_MAX_SWEEPS + 1]; // float bits of the largest decrease of sweep k (non-negative: ordered like ints)
};
struct DtGroup { // one per group of items whose transforms run side by side
    int end_iter;                   // the largest end_iter of the group's items
    int ticket[DT_MAX_SWEEPS + 1];
};
struct DtSweepArgs {
    int W, H, NS, NB; // image, strips of 32 rows, blocks of 32 columns
    int n;            // items of the group: their planes follow each other (W x H each)
    const float *cost;
    float *A;
    int *L;
    int sx, sy;       // sweep direction (+1 / -1)
    int k;            // sweep index, 1-based
    DtCtrl *ctrl;     // per item
    DtGroup *grp;
    int *prog;        // per item and strip (in sweep order): k * 65536 + column blocks finished and stored in sweep k
};

__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(int *p, int v) { asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}

// one arg_sweep update (epic_aux.cpp:118-148), operation for operation, without FMA contraction.  Branch-free: this is
// the serial chain of the wavefront (one update per step and lane), so both forms of t0 are computed and one is
// selected; the label is the one of the smaller neighbour in either form.  The square root keeps IEEE rounding; lanes
// that take the "far apart" form feed it a harmless 1.0 so that its slow path (negative argument) is never entered.
__device__ __forceinline__ void dt_update(float t1, int l1, float t2, int l2, float C, float twoCC, float &a, int &l, float &maxdiff) {
    const float dt12 = fabsf(__fsub_rn(t1, t2));
    const bool lt = t1 < t2, far = dt12 > C;
    const float tmin = lt ? t1 : t2;
    const int l0 = lt ? l1 : l2;
    const float arg = __fsub_rn(twoCC, __fmul_rn(dt12, dt12)); // twoCC = (2 C) C
    const float r = sqrtf(far ? 1.0f : arg);
    const float tn = 0.5f * __fadd_rn(__fadd_rn(t1, t2), r);
    const float t0 = far ? __fadd_rn(tmin, C) : tn;
    if (t0 < a) {
        maxdiff = fmaxf(maxdiff, __fsub_rn(a, t0));
        a = t0;
        l = l0;
    }
}

// One raster sweep of arg_sweep as a pipeline of row strips.  In sweep coordinates (p along x, q along y, both in the
// direction of the sweep) pixel (p, q) needs (p-1, q) and (p, q-1) of the SAME sweep.  A warp owns a strip of 32 rows
// (lane = row) and marches along p: at step s lane l updates column s - l, so its left neighbour is its own previous
// result (a register) and its upper neighbour is what lane l-1 produced one step earlier (a shuffle) -- a 32-row
// wavefront that never leaves the register file.  The strip below follows about 70 columns behind: it takes the last row
// of this strip from global memory, block of 32 columns by block, as soon as the block has been stored and published
// (release / acquire on a per-strip progress word).  Strips are handed out in sweep order by an atomic ticket, so a strip
// only ever waits for one that is already running.  The tile data moves global -> shared with cp.async one block ahead
// and back with coalesced row stores two blocks behind; a 3-slot ring holds the blocks in flight.
// The sweep is latency-bound on the chain shuffle -> update -> shuffle of a step, so everything else is kept off it: the
// step's operands come from shared memory through a per-lane address that is advanced incrementally (no index
// arithmetic in front of the loads), the update is branch-free, and the last row of the strip above is fetched one block
// ahead whenever it is already published (its L2 latency then overlaps 32 steps instead of stalling the block change).
constexpr int DT_RING = 3;
// bounded spin on the progress word of the strip above: a protocol error traps instead of hanging the GPU
__device__ __forceinline__ void dt_wait(const int *flag, int need) {
    unsigned spins = 0;
    while (ld_acquire_gpu(flag) < need) {
        __nanosleep(32);
        if (++spins > (1u << 24)) __trap();
    }
}
__device__ __forceinline__ float lds_f32(unsigned addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ int lds_s32(unsigned addr) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(unsigned addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_s32(unsigned addr, int v) { asm volatile("st.shared.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }

// bounded spin on a shared-memory counter of the other warp of the CTA (a protocol error traps instead of hanging)
__device__ __forceinline__ void dt_wait_smem(const volatile int *cnt, int need) {
    unsigned spins = 0;
    while (*cnt < need)
        if (++spins > (1u << 26)) __trap();
}

// CTA = two warps on one strip.  Warp 0 runs the wavefront and nothing else; warp 1 (the mover) loads the blocks ahead of
// it, fetches the halo row of the strip above, and stores / publishes the blocks behind it -- the ~3000 clk of block
// moves per 32 steps (row stores, the fence of the publication, 96 cp.async) left the serial chain of the strip this way.
// The warps meet on two shared-memory counters: `full` = blocks ready for the wavefront (written by the mover),
// `done` = blocks the wavefront has left (written by warp 0).  Ring of 3 slots: block i goes into the slot block i-3
// was stored from.
//   mover, iteration i:  A  block i-1 has landed, its halo row is in place        -> full = i
//                        B  wait done >= i-2, store block i-3, publish             (strip below may read it)
//                        C  cp.async block i into slot i % 3
//   wavefront, step 32b: lane 31 has left block b-2 -> done = b-1;  wait full >= b+1;  32 steps of block b (lane 0)
// Shared-memory layout: per array (A, L, cost) every strip row keeps a circular window of DT_COLS = 3 x 32 columns
// (the three ring slots side by side), so the wavefront's per-lane cursor is one address that advances by a column per
// step and wraps once per 96 steps.  Row pitch 98 floats: lane l reads column (s - l) of row l at step s -> bank
// (2 l + s - l) % 32 = (l + s) % 32, conflict-free; the mover's row-wise accesses are conflict-free anyway.
constexpr int DT_COLS = DT_RING * DT_TILE, DT_ROWP = DT_COLS + 2, DT_ARR = DT_TILE * DT_ROWP;
// A group of items runs its sweeps in the same launches.  The strips of all its items share one ticket sequence in sweep
// order (ticket t = strip t / n of item t % n), so every strip still only waits for the strip above it in its own image,
// which holds a smaller ticket.  An item past its own end_iter returns at once, as a single transform does.
__global__ void __launch_bounds__(64) k_dt_sweep(DtSweepArgs a) {
    if (a.k > *reinterpret_cast<volatile int *>(&a.grp->end_iter)) return;
    // [A | L | cost] arrays, then the halo row (t, label) of the strip above in the same circular column index
    __shared__ __align__(16) float smem[3 * DT_ARR + 2 * DT_COLS];
    __shared__ int s_strip;
    __shared__ volatile int s_full, s_done;
    float *const sA = smem, *const sC = smem + 2 * DT_ARR;
    int *const sL = reinterpret_cast<int *>(smem + DT_ARR);
    float *const hT = smem + 3 * DT_ARR;
    int *const hL = reinterpret_cast<int *>(hT + DT_COLS);
    // byte offsets from an address in sA: the same element of L / cost; from lane 0's cursor (row 0): the halo entries
    constexpr unsigned OFF_L = DT_ARR * 4, OFF_C = 2 * DT_ARR * 4, OFF_HT = 3 * DT_ARR * 4, OFF_HL = (3 * DT_ARR + DT_COLS) * 4;
    const int lane = threadIdx.x & 31;
    const bool mover = threadIdx.x >= 32;
    const float INF = __int_as_float(0x7f800000);
    if (threadIdx.x == 0) {
        s_strip = atomicAdd(&a.grp->ticket[a.k], 1);
        s_full = 0;
        s_done = 0;
    }
    __syncthreads();
    const int ticket = s_strip;
    if (ticket >= a.NS * a.n) return;
    const int item = ticket % a.n, strip = ticket / a.n;
    DtCtrl *const ctrl = a.ctrl + item;
    if (a.k > *reinterpret_cast<volatile int *>(&ctrl->end_iter)) return;
    const int W = a.W, H = a.H, q0 = strip * DT_TILE, rows = min(DT_TILE, H - q0);
    const int NB = a.NB;
    const size_t item_off = (size_t)item * W * H;
    const float *const cost = a.cost + item_off;
    float *const gA = a.A + item_off;
    int *const gL = a.L + item_off;
    int *const prog = a.prog + item * a.NS;

    if (mover) {
        const int jtop = (a.sy > 0) ? q0 - 1 : H - q0; // image row of sweep row q0 - 1 (the last row of the strip above)
        const int base = a.k << 16;
        auto load_block = [&](int m) { // A, L, cost of columns 32m .. 32m+31, all rows of the strip: lane = column (coalesced)
            const int p = m * DT_TILE + lane;
            if (p < W) {
                const int i = a.sx > 0 ? p : W - 1 - p;
                const int e0 = (m % DT_RING) * DT_TILE + lane;
#pragma unroll 8
                for (int r = 0; r < rows; r++) {
                    const size_t o = (size_t)(a.sy > 0 ? q0 + r : H - 1 - (q0 + r)) * W + i;
                    const int e = r * DT_ROWP + e0;
                    cp_async4(&sA[e], gA + o);
                    cp_async4(&sL[e], gL + o);
                    cp_async4(&sC[e], cost + o);
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        // rows [r0, r1) of block m back to the image
        auto store_rows = [&](int m, int r0, int r1) {
            const int p = m * DT_TILE + lane;
            if (p < W) {
                const int i = a.sx > 0 ? p : W - 1 - p;
                const int e0 = (m % DT_RING) * DT_TILE + lane;
#pragma unroll 8
                for (int r = r0; r < r1; r++) {
                    const size_t o = (size_t)(a.sy > 0 ? q0 + r : H - 1 - (q0 + r)) * W + i;
                    const int e = r * DT_ROWP + e0;
                    gA[o] = sA[e];
                    gL[o] = sL[e];
                }
            }
        };
#pragma unroll 1
        for (int i = 0; i < NB + 3; i++) {
            if (i >= 1 && i <= NB) { // A: block i-1
                const int m = i - 1, p = m * DT_TILE + lane;
                float t = INF;
                int l = -1;
                if (strip > 0) {
                    if (lane == 0) dt_wait(prog + strip - 1, base + m + 1);
                    __syncwarp();
                    if (p < W) {
                        const int ii = a.sx > 0 ? p : W - 1 - p;
                        t = __ldcg(gA + (size_t)jtop * W + ii);
                        l = __ldcg(gL + (size_t)jtop * W + ii);
                    }
                }
                hT[(m % DT_RING) * DT_TILE + lane] = t;
                hL[(m % DT_RING) * DT_TILE + lane] = l;
                asm volatile("cp.async.wait_group 0;" ::: "memory"); // block i-1 has landed (the lanes' copies: next line)
                __syncwarp();
                __threadfence_block();
                if (lane == 0) s_full = i;
            }
            if (i >= 3) { // B: block i-3 (i - 3 < NB by the loop bound)
                if (lane == 0) dt_wait_smem(&s_done, i - 2);
                __syncwarp();
                __threadfence_block();
                // The strip below only reads the LAST row of this strip, and its start is the critical path of the sweep
                // (one hand-over per strip): that row goes out and is published first -- the fence of the release then has
                // two stores per lane to wait for instead of 64 -- the other rows follow.  The lanes' stores become
                // visible with lane 0's release: __syncwarp orders them before it, the release is cumulative.
                store_rows(i - 3, rows - 1, rows);
                __syncwarp();
                if (lane == 0) st_release_gpu(prog + strip, base + i - 2);
                store_rows(i - 3, 0, rows - 1);
            }
            if (i < NB) load_block(i); // C (after the store: the slot is the one block i-3 was read out of just now)
        }
        return;
    }

    // ---- the wavefront.  Lane l works on column p = s - l at step s; rows below the image never become valid.
    float cur_t = INF, maxdiff = 0.0f; // (left neighbour of column 0: INF / -1, the initial values)
    int cur_l = -1;
    const unsigned row_lo = (unsigned)__cvta_generic_to_shared(smem) + 4u * (unsigned)(lane * DT_ROWP), row_hi = row_lo + 4u * DT_COLS;
    unsigned addr = lane ? row_hi - 4u * (unsigned)lane : row_lo; // cursor: element (row l, column p mod 96) of A
    int p = (lane < rows) ? -lane : -(1 << 30);
    const int nsteps = W + DT_TILE - 1;
#pragma unroll 1
    for (int b = 0; b * DT_TILE < nsteps; b++) {
        // lane 0 enters block b now; lane 31 left block b-2 in the previous step
        __syncwarp();
        if (b >= 2 && b - 2 < NB) {
            __threadfence_block();
            if (lane == 0) s_done = b - 1;
        }
        if (b < NB) {
            if (lane == 0) dt_wait_smem(&s_full, b + 1);
            __syncwarp();
            __threadfence_block();
        }
        const int jn = min(DT_TILE, nsteps - b * DT_TILE);
#pragma unroll 1
        for (int j = 0; j < jn; j++, p++) {
            float up_t = __shfl_up_sync(0xffffffffu, cur_t, 1);
            int up_l = __shfl_up_sync(0xffffffffu, cur_l, 1);
            if ((unsigned)p < (unsigned)W) {
                float av = lds_f32(addr);
                int lv = lds_s32(addr + OFF_L);
                const float C = lds_f32(addr + OFF_C);
                if (lane == 0) { // (row_lo of lane 0 is the start of the array: the cursor doubles as the halo index)
                    up_t = lds_f32(addr + OFF_HT);
                    up_l = lds_s32(addr + OFF_HL);
                }
                dt_update(up_t, up_l, cur_t, cur_l, C, __fmul_rn(__fmul_rn(2.0f, C), C), av, lv, maxdiff);
                sts_f32(addr, av);
                sts_s32(addr + OFF_L, lv);
                cur_t = av;
                cur_l = lv;
            }
            addr += 4u;
            if (addr == row_hi) addr = row_lo;
        }
    }
    __syncwarp();
    __threadfence_block();
    if (lane == 0) s_done = NB; // every block may be stored now
    for (int off = 16; off > 0; off >>= 1) maxdiff = fmaxf(maxdiff, __shfl_xor_sync(0xffffffffu, maxdiff, off));
    if (lane == 0 && maxdiff > 0.0f) atomicMax(&ctrl->maxdiff[a.k], __float_as_uint(maxdiff));
}
// the loop control of weighted_distance_transform (epic_aux.cpp:170-178) after sweep k; one thread per item of the group
__global__ void k_dt_control(DtCtrl *ctrl, DtGroup *grp, int n, int k, float min_change, int max_iter) {
    if ((int)threadIdx.x >= n) return;
    DtCtrl *c = ctrl + threadIdx.x;
    if (k > c->end_iter) return;
    c->sweeps_run = k;
    if (__uint_as_float(c->maxdiff[k]) > min_change) {
        c->end_iter = min(max_iter, k + 3);
        atomicMax(&grp->end_iter, c->end_iter);
    }
}

// ------------------------------------------------------------------------------------------ neighbourhood graph of the seeds
// (ngh_labels_to_spmat, epic_aux.cpp:226-288): for every pixel with i >= 1 and j >= 1 whose left / upper neighbour carries
// another label, the edge (l0, l1) with cost dis[p] + dis[q]; emitted in both directions with key = (row << 32) | col.
// blockIdx.z is the item (maps of W x H each); the labels are global seed ids, so one list serves all items.
__global__ void __launch_bounds__(256) k_border_emit(int W, int H, const int *__restrict__ lab, const float *__restrict__ dis,
                                                     unsigned long long *__restrict__ keys, float *__restrict__ vals, int *__restrict__ count, int cap) {
    const int i = blockIdx.x * 32 + threadIdx.x, j = blockIdx.y * 8 + threadIdx.y;
    int n = 0;
    unsigned long long k0 = 0, k1 = 0;
    float d0 = 0.f, d1 = 0.f;
    if (i >= 1 && j >= 1 && i < W && j < H) {
        const size_t o = (size_t)j * W + i + (size_t)blockIdx.z * W * H;
        const int l0 = lab[o], l1 = lab[o - 1], l2 = lab[o - W];
        if (l0 != l1 && l0 >= 0 && l1 >= 0) { k0 = ((unsigned long long)(unsigned)l0 << 32) | (unsigned)l1; d0 = dis[o] + dis[o - 1]; n = 1; }
        if (l0 != l2 && l0 >= 0 && l2 >= 0) { k1 = ((unsigned long long)(unsigned)l0 << 32) | (unsigned)l2; d1 = dis[o] + dis[o - W]; n |= 2; }
    }
    const int mine = 2 * ((n & 1) + ((n >> 1) & 1));
    // warp-aggregated append
    int pre = mine;
    const int lane = (threadIdx.y * 32 + threadIdx.x) & 31;
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, pre, off);
        if (lane >= off) pre += v;
    }
    const int total = __shfl_sync(0xffffffffu, pre, 31);
    int base = 0;
    if (lane == 31 && total > 0) base = atomicAdd(count, total);
    base = __shfl_sync(0xffffffffu, base, 31);
    int at = base + pre - mine;
    auto put = [&](unsigned long long k, float d) {
        if (at + 1 < cap) {
            keys[at] = k; vals[at] = d;
            keys[at + 1] = (k << 32) | (k >> 32); vals[at + 1] = d;
        }
        at += 2;
    };
    if (n & 1) put(k0, d0);
    if (n & 2) put(k1, d1);
}
__global__ void k_csr_rows(int ns, int nedges, const unsigned long long *__restrict__ keys, int *__restrict__ indptr, int *__restrict__ indices) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r <= ns) { // indptr[r] = first edge whose row is >= r
        int lo = 0, hi = nedges;
        const unsigned long long key = (unsigned long long)(unsigned)r << 32;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (keys[mid] < key) lo = mid + 1; else hi = mid;
        }
        indptr[r] = lo;
    }
    for (int e = r; e < nedges; e += ns + 1) indices[e] = (int)(keys[e] & 0xffffffffu);
}

// ------------------------------------------------------------------------------------------ k nearest seeds on the graph
// find_nn_graph_arr (epic_aux.cpp:47-85): Dijkstra with std::priority_queue<current_t, vector, smallest_on_top>.  The heap
// below performs exactly libstdc++'s push_heap / pop_heap moves, so entries with equal distance leave it in the same order.
constexpr int KNN_HEAP = 2048;
struct HeapItem { int node; float dis; };
__device__ __forceinline__ bool heap_less(const HeapItem &x, const HeapItem &y) { return x.dis > y.dis; } // comp(a, b): a.dis > b.dis
__device__ void heap_push(HeapItem *h, int &len, HeapItem v) {
    int hole = len++;
    int parent = (hole - 1) / 2;
    while (hole > 0 && heap_less(h[parent], v)) {
        h[hole] = h[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    h[hole] = v;
}
__device__ HeapItem heap_pop(HeapItem *h, int &len) { // pop_heap + pop_back
    const HeapItem top = h[0];
    const HeapItem v = h[len - 1];
    len--;
    if (len == 0) return top;
    int hole = 0, child = 0;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (heap_less(h[child], h[child - 1])) child--;
        h[hole] = h[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        h[hole] = h[child - 1];
        hole = child - 1;
    }
    int parent = (hole - 1) / 2;
    while (hole > 0 && heap_less(h[parent], v)) {
        h[hole] = h[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    h[hole] = v;
    return top;
}
// one warp per seed (lane 0 runs the search, the warp restores the tentative-distance array afterwards).  Rows of nnf / dis
// are `ld` entries apart, and a seed fills the first nns of its item.  A search never leaves its seed's item, so the
// per-warp tentative distances are indexed by the node's index within the item: done_all holds `nsmax` (the largest item's
// seed count) entries per warp.
__global__ void __launch_bounds__(256) k_knn_graph(int ns, int ld, int nsmax, SeedItems si, const int *__restrict__ indptr, const int *__restrict__ indices,
                                                   const float *__restrict__ data, unsigned *__restrict__ done_all, int *__restrict__ touched_all,
                                                   int *__restrict__ nnf, float *__restrict__ dis, int *__restrict__ overflow, int heap_cap) {
    extern __shared__ HeapItem heaps[];
    const int warp_in_block = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gwarp = blockIdx.x * (blockDim.x >> 5) + warp_in_block, nwarps = gridDim.x * (blockDim.x >> 5);
    HeapItem *h = heaps + warp_in_block * heap_cap; // heap_cap <= KNN_HEAP entries of shared memory per warp
    unsigned *const done_w = done_all + (size_t)gwarp * nsmax; // float bits; EPIC_UNSEEN = not reached (memset 0x7F in the reference)
    int *touched = touched_all + (size_t)gwarp * KNN_HEAP * 2;   // (indices within the item)
    for (int seed = gwarp; seed < ns; seed += nwarps) {
        int ntouched = 0, n = 0;
        if (lane == 0) {
            const int it = si.item[seed], nn = si.nns[it];
            unsigned *const done = done_w - si.off[it]; // done[node] for the global ids of this item
            int len = 0;
            heap_push(h, len, HeapItem{seed, 0.0f});
            done[seed] = __float_as_uint(0.0f);
            touched[ntouched++] = seed - si.off[it];
            while (len > 0) {
                const HeapItem cur = heap_pop(h, len);
                if (cur.dis > __uint_as_float(done[cur.node])) continue;
                nnf[(size_t)seed * ld + n] = cur.node;
                dis[(size_t)seed * ld + n] = cur.dis;
                n++;
                if (n >= nn) break;
                for (int e = indptr[cur.node]; e < indptr[cur.node + 1]; e++) {
                    const int ngh = indices[e];
                    const float nd = cur.dis + data[e];
                    if (nd >= __uint_as_float(done[ngh])) continue;
                    if (len >= heap_cap || ntouched >= 2 * KNN_HEAP) { atomicExch(overflow, 1); continue; }
                    heap_push(h, len, HeapItem{ngh, nd});
                    if (done[ngh] == EPIC_UNSEEN) touched[ntouched++] = ngh - si.off[it];
                    done[ngh] = __float_as_uint(nd);
                }
            }
            for (int k = n; k < nn; k++) { // not enough results: 0xFF / 0x7F patterns like the reference's memsets
                nnf[(size_t)seed * ld + k] = -1;
                dis[(size_t)seed * ld + k] = __uint_as_float(EPIC_UNSEEN);
            }
        }
        ntouched = __shfl_sync(0xffffffffu, ntouched, 0);
        __syncwarp();
        for (int k = lane; k < ntouched; k += 32) done_w[touched[k]] = EPIC_UNSEEN;
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------ per-seed fits, per-pixel apply
// query point = seed i: neighbours of the seed that owns its pixel, distances + the pixel's own distance, then the kernel
// exp(-coef d) + 1e-08 (dist_trf_nnfield_subset :385-394, epic.cpp:96-98, 203-205)
// (rows of ld entries, the first nns of the seed's item used, like nnf / dis; maps of W x H = N pixels per item)
__global__ void k_query_weights(int ns, int ld, SeedItems si, const int *__restrict__ seeds, int W, size_t N, const int *__restrict__ labels,
                                const float *__restrict__ dmap, const int *__restrict__ nnf, const float *__restrict__ dis, float coef, int *__restrict__ qnn,
                                float *__restrict__ qw) {
    const int i = blockIdx.x, j = threadIdx.x;
    if (i >= ns) return;
    const int it = si.item[i], nn = si.nns[it];
    const size_t p = it * N + (size_t)seeds[2 * i + 1] * W + seeds[2 * i];
    const int s = labels[p];
    const float d = dmap[p];
    for (int k = j; k < nn; k += blockDim.x) {
        qnn[(size_t)i * ld + k] = nnf[(size_t)s * ld + k];
        const float dist = d + dis[(size_t)s * ld + k];
        qw[(size_t)i * ld + k] = (coef < 0.0f) ? dist : (float)((double)expf(-coef * dist) + 1e-08); // coef < 0: raw distances (operator twin)
    }
}
// fit_nadarayawatson (epic_aux.cpp:410-428): sequential float sums in neighbour order
__global__ void k_fit_nw(int ns, int ld, SeedItems si, const int *__restrict__ qnn, const float *__restrict__ qw, const float *__restrict__ vects,
                         float *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    const int nn = si.nns[si.item[i]];
    float u = 0.0f, v = 0.0f, s = 0.0f;
    for (int j = 0; j < nn; j++) {
        const float d = qw[(size_t)i * ld + j];
        const int jj = qnn[(size_t)i * ld + j];
        if (jj < 0) continue;
        u = __fadd_rn(u, __fmul_rn(d, vects[2 * jj]));
        v = __fadd_rn(v, __fmul_rn(d, vects[2 * jj + 1]));
        s = __fadd_rn(s, d);
    }
    out[2 * i] = u / s;
    out[2 * i + 1] = v / s;
}
__global__ void k_prefilter_flags(int ns, const float *__restrict__ est, const float *__restrict__ vects, float th2, unsigned char *__restrict__ keep) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    const float a = est[2 * i] - vects[2 * i], b = est[2 * i + 1] - vects[2 * i + 1];
    keep[i] = (__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)) < th2) ? 1 : 0;
}
// fit_localaffine (epic_aux.cpp:438-481).  Rows of the reference's system are (x c, y c, c | (x + wx) c) and the same for y:
// two weighted least-squares fits (weights c^2) of x' and y' over [x y 1].  Normal equations in double, centred on the seed.
__global__ void k_fit_la(int ns, int ld, SeedItems si, const int *__restrict__ qnn, const float *__restrict__ qw, const int *__restrict__ seeds,
                         const float *__restrict__ vects, float *__restrict__ aff) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    const int nn = si.nns[si.item[i]];
    const double xi = seeds[2 * i], yi = seeds[2 * i + 1];
    double sxx = 0, sxy = 0, sx = 0, syy = 0, sy = 0, s1 = 0, bx0 = 0, bx1 = 0, bx2 = 0, by0 = 0, by1 = 0, by2 = 0;
    auto add = [&](double x, double y, double wx, double wy, float cf) {
        // the reference forms the row entries in float: (x)*(c), (y)*(c), ((x)+(wx))*(c)
        const double c2 = (double)cf * (double)cf;
        const double dx = x - xi, dy = y - yi;          // centred design
        const double tx = (x + wx) - xi, ty = (y + wy) - yi; // centred targets
        sxx += c2 * dx * dx; sxy += c2 * dx * dy; sx += c2 * dx; syy += c2 * dy * dy; sy += c2 * dy; s1 += c2;
        bx0 += c2 * dx * tx; bx1 += c2 * dy * tx; bx2 += c2 * tx;
        by0 += c2 * dx * ty; by1 += c2 * dy * ty; by2 += c2 * ty;
    };
    float coefi = 0.0f;
    for (int j = 0; j < nn; j++) {
        const int s = qnn[(size_t)i * ld + j];
        if (s < 0) continue;
        float coef = qw[(size_t)i * ld + j];
        if (s == i) { coefi = 0.01f * coef; coef *= 0.96f; }
        add((double)seeds[2 * s], (double)seeds[2 * s + 1], (double)vects[2 * s], (double)vects[2 * s + 1], coef);
    }
    const double ui = vects[2 * i], vi = vects[2 * i + 1];
    add((double)((float)xi + 0.1f), yi, ui, vi, coefi);
    add(xi, (double)((float)yi + 0.1f), ui, vi, coefi);
    add((double)((float)xi - 0.1f), yi, ui, vi, coefi);
    add(xi, (double)((float)yi - 0.1f), ui, vi, coefi);
    // solve the symmetric 3x3 system [sxx sxy sx; sxy syy sy; sx sy s1] p = b (cofactors)
    const double c00 = syy * s1 - sy * sy, c01 = sx * sy - sxy * s1, c02 = sxy * sy - syy * sx;
    const double c11 = sxx * s1 - sx * sx, c12 = sxy * sx - sxx * sy, c22 = sxx * syy - sxy * sxy;
    const double det = sxx * c00 + sxy * c01 + sx * c02;
    const double inv = 1.0 / det;
    const double a0 = (c00 * bx0 + c01 * bx1 + c02 * bx2) * inv, a1 = (c01 * bx0 + c11 * bx1 + c12 * bx2) * inv,
                 a2 = (c02 * bx0 + c12 * bx1 + c22 * bx2) * inv;
    const double a3 = (c00 * by0 + c01 * by1 + c02 * by2) * inv, a4 = (c01 * by0 + c11 * by1 + c12 * by2) * inv,
                 a5 = (c02 * by0 + c12 * by1 + c22 * by2) * inv;
    // back to absolute coordinates: x' = a0 (x - xi) + a1 (y - yi) + a2 + xi
    float *m = aff + (size_t)6 * i;
    m[0] = (float)a0; m[1] = (float)a1; m[2] = (float)(a2 + xi - a0 * xi - a1 * yi);
    m[3] = (float)a3; m[4] = (float)a4; m[5] = (float)(a5 + yi - a3 * xi - a4 * yi);
}
// apply_localaffine / apply_nadarayawatson (epic_aux.cpp:430-436, 483-492) straight into the flow planes (stride S);
// blockIdx.z is the item: its label map is W x H further on, its flow planes zs floats
__global__ void __launch_bounds__(256) k_apply(Geom g, const int *__restrict__ labels, const float *__restrict__ model, int affine, float *__restrict__ fx,
                                               float *__restrict__ fy, size_t zs) {
    const int i = blockIdx.x * 32 + threadIdx.x, j = blockIdx.y * 8 + threadIdx.y;
    if (i >= g.W || j >= g.H) return;
    const int s = labels[(size_t)j * g.W + i + (size_t)blockIdx.z * g.W * g.H];
    const size_t o = (size_t)j * g.S + i + blockIdx.z * zs;
    if (s < 0) { fx[o] = 0.0f; fy[o] = 0.0f; return; }
    if (affine) {
        const float *m = model + (size_t)6 * s;
        fx[o] = __fsub_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], (float)i), __fmul_rn(m[1], (float)j)), m[2]), (float)i);
        fy[o] = __fsub_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[3], (float)i), __fmul_rn(m[4], (float)j)), m[5]), (float)j);
    } else {
        fx[o] = model[2 * s];
        fy[o] = model[2 * s + 1];
    }
}

// ------------------------------------------------------------------------------------------ host side
// All device memory of a call comes from ONE grow-only arena kept by the context (cudaMalloc / cudaFree per buffer cost
// more than the kernels: 390 ms per call against 20 ms of GPU work at 1024x436).  Buffers are bump-allocated views;
// mark() / release() give stack discipline to the scratch of a phase.  A call that does not fit reports it, the entry
// point grows the arena to the recorded high-water mark and runs the call again.
struct EpicArena {
    char *base = nullptr;
    size_t cap = 0, off = 0, high = 0;
    bool overflow = false;
    void *take(size_t bytes) {
        const size_t at = (off + 255) & ~(size_t)255;
        high = std::max(high, at + bytes);
        if (at + bytes > cap) {
            overflow = true;
            return nullptr;
        }
        off = at + bytes;
        return base + at;
    }
    size_t mark() const { return off; }
    void release(size_t m) { off = m; }
};
void epic_arena_free(EpicArena *a) {
    if (!a) return;
    if (a->base) cudaFree(a->base);
    delete a;
}
static thread_local EpicArena *g_arena = nullptr; // the arena of the call running on this host thread
struct DevBuf { // a view into the arena (named like the owning buffer it replaced)
    void *p = nullptr;
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
    bool alloc(size_t bytes) {
        p = g_arena->take(bytes ? bytes : 4);
        if (!p) set_error("sfgpu_epic: workspace arena too small (the call is repeated with a larger one)");
        return p != nullptr;
    }
};
struct ArenaScope { // releases everything a phase allocated when it ends
    size_t m;
    ArenaScope() : m(g_arena->mark()) {}
    ~ArenaScope() { g_arena->release(m); }
};
static dim3 grid2(int w, int h) { return dim3((w + 31) / 32, (h + 7) / 8); }

// phase timer for SLOWFLOW_GPU_TRACE=1 (stderr); synchronises the stream when tracing, otherwise free
struct EpicTrace {
    bool on;
    cudaStream_t st;
    std::chrono::steady_clock::time_point t0;
    explicit EpicTrace(cudaStream_t s) : on(getenv("SLOWFLOW_GPU_TRACE") != nullptr), st(s), t0(std::chrono::steady_clock::now()) {}
    void mark(const char *what) {
        if (!on) return;
        cudaStreamSynchronize(st);
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "  epic: %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

struct EpicGeo {
    int W, H;
};

// The seeds of the n items of one call, host side of SeedItems: item k owns the global ids off[k] .. off[k+1]-1 and
// searches nns[k] neighbours.
struct EpicItems {
    int n = 0;
    std::vector<int> off, nns, item;
    SeedItems d{};
    int ns() const { return off[n]; }
    int nnmax() const { return *std::max_element(nns.begin(), nns.end()); }
    int nsmax() const {
        int m = 0;
        for (int k = 0; k < n; k++) m = std::max(m, off[k + 1] - off[k]);
        return m;
    }
    int upload(cudaStream_t st) { // the device copies, in the arena
        item.resize(ns());
        for (int k = 0; k < n; k++) std::fill(item.begin() + off[k], item.begin() + off[k + 1], k);
        DevBuf di, doff, dnns;
        if (!di.alloc(item.size() * 4) || !doff.alloc((size_t)(n + 1) * 4) || !dnns.alloc((size_t)n * 4)) return SFGPU_ERR_CUDA;
        if (!item.empty()) SF_CUDA(cudaMemcpyAsync(di.p, item.data(), item.size() * 4, cudaMemcpyHostToDevice, st));
        SF_CUDA(cudaMemcpyAsync(doff.p, off.data(), (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, st));
        SF_CUDA(cudaMemcpyAsync(dnns.p, nns.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
        d = SeedItems{di.as<int>(), doff.as<int>(), dnns.as<int>()};
        return SFGPU_OK;
    }
};

// dist_trf_nnfield_subset with the seeds as query points, followed by the kernel weights, for all items of `it` at once:
// fills qnn / qw (rows of it.nnmax() entries, the first nns of the seed's item used) and leaves the label maps (W x H per
// item, global seed ids) in `labels`.  Everything is queued on the context's stream; returns after one sync.
static int nn_field(sfgpu_ctx *c, const EpicGeo &eg, const float *d_cost, const EpicItems &it, const int *d_seeds, float coef, int *d_labels,
                    float *d_dmap, int *d_qnn, float *d_qw, int *sweeps_out) {
    cudaStream_t st = c->stream;
    EpicTrace tr(st);
    ArenaScope scope; // (the caller's buffers were allocated before; the stream is idle when the scratch is released)
    const int W = eg.W, H = eg.H, n = it.n, ns = it.ns(), ld = it.nnmax();
    const size_t N = (size_t)W * H;
    const int NS = (H + DT_TILE - 1) / DT_TILE, NB = (W + DT_TILE - 1) / DT_TILE;
    // One block of two warps and 40 KB of shared memory per strip of 32 rows; every strip must be resident together with the
    // one above it (tickets hand the strips out in sweep order), and 4 blocks per SM always fit.  So the transforms of a
    // batch run in groups of items whose strips number at most 4 per SM, one group after the other.
    if (NS > c->num_sms * 4) {
        set_error("sfgpu_epic: image too tall for the strip pipeline of the distance transform");
        return SFGPU_ERR_UNSUPPORTED;
    }
    const int per_group = std::min(n, c->num_sms * 4 / NS), ngroups = (n + per_group - 1) / per_group;
    DevBuf ctrl, grp, prog;
    if (!ctrl.alloc((size_t)n * sizeof(DtCtrl)) || !grp.alloc((size_t)ngroups * sizeof(DtGroup)) || !prog.alloc((size_t)n * NS * sizeof(int)))
        return SFGPU_ERR_CUDA;
    std::vector<DtCtrl> h_ctrl((size_t)n);
    std::vector<DtGroup> h_grp((size_t)ngroups);
    memset(h_ctrl.data(), 0, h_ctrl.size() * sizeof(DtCtrl));
    memset(h_grp.data(), 0, h_grp.size() * sizeof(DtGroup));
    for (auto &x : h_ctrl) x.end_iter = 4; // (:168)
    for (auto &x : h_grp) x.end_iter = 4;
    SF_CUDA(cudaMemcpyAsync(ctrl.p, h_ctrl.data(), h_ctrl.size() * sizeof(DtCtrl), cudaMemcpyHostToDevice, st));
    SF_CUDA(cudaMemcpyAsync(grp.p, h_grp.data(), h_grp.size() * sizeof(DtGroup), cudaMemcpyHostToDevice, st));
    SF_CUDA(cudaMemsetAsync(prog.p, 0, (size_t)n * NS * sizeof(int), st));
    k_fill_u32<<<592, 256, 0, st>>>(n * N, reinterpret_cast<unsigned *>(d_dmap), EPIC_UNSEEN);
    k_fill_u32<<<592, 256, 0, st>>>(n * N, reinterpret_cast<unsigned *>(d_labels), 0xFFFFFFFFu);
    k_dt_seed_labels<<<(ns + 255) / 256, 256, 0, st>>>(ns, d_seeds, it.d.item, W, N, d_labels);
    k_dt_seed_dist<<<(ns + 255) / 256, 256, 0, st>>>(ns, d_seeds, it.d.item, W, N, d_cost, d_dmap);
    // sweeps i = 1 .. : direction (x[i % 4], y[i % 4]) with x = {-1, 1, 1, -1}, y = {1, 1, -1, -1} (:165-172)
    static const int dx[4] = {-1, 1, 1, -1}, dy[4] = {1, 1, -1, -1};
    for (int g0 = 0, gi = 0; g0 < n; g0 += per_group, gi++) {
        const int gn = std::min(per_group, n - g0);
        for (int k = 1; k <= DT_MAX_SWEEPS; k++) {
            DtSweepArgs a;
            a.W = W; a.H = H; a.NS = NS; a.NB = NB; a.n = gn;
            a.cost = d_cost + g0 * N; a.A = d_dmap + g0 * N; a.L = d_labels + g0 * N;
            a.sx = dx[k % 4]; a.sy = dy[k % 4];
            a.k = k;
            a.ctrl = ctrl.as<DtCtrl>() + g0;
            a.grp = grp.as<DtGroup>() + gi;
            a.prog = prog.as<int>() + (size_t)g0 * NS;
            k_dt_sweep<<<gn * NS, 64, 0, st>>>(a);
            // default dt_params: max_iter 40, min_change 1 (:151-154)
            k_dt_control<<<1, gn, 0, st>>>(ctrl.as<DtCtrl>() + g0, grp.as<DtGroup>() + gi, gn, k, 1.0f, DT_MAX_SWEEPS);
        }
    }
    c->prof_acc.kernel_launches += 4 + 2 * DT_MAX_SWEEPS * ngroups;
    tr.mark("distance transform");

    // ---- neighbourhood graph
    // label borders: every border pixel pair emits two entries; ~6 sqrt(N ns) per item in practice, 4 N at worst
    size_t cap_all = 0;
    for (int k = 0; k < n; k++) cap_all += std::min<size_t>(4 * N, (size_t)(32.0 * sqrt((double)N * (double)(it.off[k + 1] - it.off[k]))) + ((size_t)1 << 20));
    const int cap = (int)std::min<size_t>(cap_all, (size_t)1 << 30);
    DevBuf keys, vals, keys2, vals2, count, ukeys, uvals, nruns, tmp;
    if (!keys.alloc((size_t)cap * 8) || !vals.alloc((size_t)cap * 4) || !keys2.alloc((size_t)cap * 8) || !vals2.alloc((size_t)cap * 4) ||
        !count.alloc(8) || !nruns.alloc(8))
        return SFGPU_ERR_CUDA;
    SF_CUDA(cudaMemsetAsync(count.p, 0, 8, st));
    dim3 bgrid = grid2(W, H);
    bgrid.z = n;
    k_border_emit<<<bgrid, dim3(32, 8), 0, st>>>(W, H, d_labels, d_dmap, keys.as<unsigned long long>(), vals.as<float>(), count.as<int>(), cap);
    int h_count = 0;
    SF_CUDA(cudaMemcpyAsync(&h_count, count.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaMemcpyAsync(h_ctrl.data(), ctrl.p, h_ctrl.size() * sizeof(DtCtrl), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    int most_sweeps = 0;
    for (int k = 0; k < n; k++) {
        if (sweeps_out) sweeps_out[k] = h_ctrl[k].sweeps_run;
        most_sweeps = std::max(most_sweeps, h_ctrl[k].sweeps_run);
    }
    if (tr.on)
        fprintf(stderr, "  epic: (distance transform: %d item(s) in %d group(s), up to %d sweeps, %d strips x %d blocks per item)\n", n, ngroups,
                most_sweeps, NS, NB);
    tr.mark("border emit (+allocs)");
    if (h_count + 1 >= cap) {
        set_error("sfgpu_epic: label border list overflow (more than 32 sqrt(N ns) + 1M border entries)");
        return SFGPU_ERR_UNSUPPORTED;
    }
    int nedges = 0;
    DevBuf indptr, indices;
    if (!indptr.alloc((size_t)(ns + 1) * sizeof(int))) return SFGPU_ERR_CUDA;
    if (h_count > 0) {
        size_t tb1 = 0, tb2 = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tb1, keys.as<unsigned long long>(), keys2.as<unsigned long long>(), vals.as<float>(), vals2.as<float>(), h_count, 0, 64, st);
        if (!ukeys.alloc((size_t)h_count * 8) || !uvals.alloc((size_t)h_count * 4)) return SFGPU_ERR_CUDA;
        cub::DeviceReduce::ReduceByKey(nullptr, tb2, keys2.as<unsigned long long>(), ukeys.as<unsigned long long>(), vals2.as<float>(), uvals.as<float>(),
                                       nruns.as<int>(), cub::Min(), h_count, st);
        if (!tmp.alloc(std::max(tb1, tb2))) return SFGPU_ERR_CUDA;
        size_t tb = std::max(tb1, tb2);
        SF_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tb, keys.as<unsigned long long>(), keys2.as<unsigned long long>(), vals.as<float>(), vals2.as<float>(),
                                                h_count, 0, 64, st));
        tb = std::max(tb1, tb2);
        SF_CUDA(cub::DeviceReduce::ReduceByKey(tmp.p, tb, keys2.as<unsigned long long>(), ukeys.as<unsigned long long>(), vals2.as<float>(), uvals.as<float>(),
                                               nruns.as<int>(), cub::Min(), h_count, st));
        SF_CUDA(cudaMemcpyAsync(&nedges, nruns.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        SF_CUDA(cudaStreamSynchronize(st));
    }
    if (!indices.alloc((size_t)std::max(nedges, 1) * sizeof(int))) return SFGPU_ERR_CUDA;
    k_csr_rows<<<(ns + 1 + 255) / 256, 256, 0, st>>>(ns, nedges, ukeys.as<unsigned long long>(), indptr.as<int>(), indices.as<int>());
    tr.mark("sort + reduce + csr");

    // ---- k nearest seeds of every seed, then the query step.  The search is one serial thread per seed, i.e. bound by the
    // latency of its dependent loads: what counts is how many searches are in flight.  The heap lives in shared memory, so
    // its capacity sets the residency: first a pass with 1024 entries per warp (3 blocks of 8 warps per SM; a search for
    // nn = 100 neighbours on the planar seed graph keeps a few hundred entries open), and only if a heap overflowed the
    // pass with the full 2048 entries (1 block per SM).  An overflow reruns the search of every item.
    const int warps_per_block = 8;
    int blocks_per_sm = 3;
    int blocks = std::min((ns + warps_per_block - 1) / warps_per_block, c->num_sms * blocks_per_sm);
    // the per-warp tentative-distance arrays: one entry per seed of the largest item per resident warp (bounded to 1 GB)
    const int nsmax = it.nsmax();
    while (blocks > 1 && (size_t)blocks * warps_per_block * nsmax * 4 > ((size_t)1 << 30)) blocks /= 2;
    DevBuf done_all, touched, nnf, dis, overflow;
    const size_t nwarps = (size_t)blocks * warps_per_block;
    if (!done_all.alloc(nwarps * nsmax * 4) || !touched.alloc(nwarps * KNN_HEAP * 2 * 4) || !nnf.alloc((size_t)ns * ld * 4) ||
        !dis.alloc((size_t)ns * ld * 4) || !overflow.alloc(4))
        return SFGPU_ERR_CUDA;
    k_fill_u32<<<592, 256, 0, st>>>(nwarps * nsmax, done_all.as<unsigned>(), EPIC_UNSEEN);
    SF_CUDA(cudaMemsetAsync(overflow.p, 0, 4, st));
    tr.mark("knn allocs + fill");
    SF_CUDA(cudaFuncSetAttribute(k_knn_graph, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)warps_per_block * KNN_HEAP * sizeof(HeapItem))));
    int h_over = 0;
    for (int heap_cap = KNN_HEAP / 2; heap_cap <= KNN_HEAP; heap_cap *= 2) {
        const size_t smem = (size_t)warps_per_block * heap_cap * sizeof(HeapItem);
        const int nblocks = heap_cap == KNN_HEAP ? std::min(blocks, c->num_sms) : blocks; // (a retry: every entry of done_all is EPIC_UNSEEN again)
        k_knn_graph<<<nblocks, warps_per_block * 32, smem, st>>>(ns, ld, nsmax, it.d, indptr.as<int>(), indices.as<int>(), uvals.as<float>(),
                                                                 done_all.as<unsigned>(), touched.as<int>(), nnf.as<int>(), dis.as<float>(), overflow.as<int>(),
                                                                 heap_cap);
        c->prof_acc.kernel_launches++;
        SF_CUDA(cudaMemcpyAsync(&h_over, overflow.p, 4, cudaMemcpyDeviceToHost, st));
        SF_CUDA(cudaStreamSynchronize(st));
        if (!h_over) break;
        if (heap_cap < KNN_HEAP) SF_CUDA(cudaMemsetAsync(overflow.p, 0, 4, st));
    }
    k_query_weights<<<ns, 128, 0, st>>>(ns, ld, it.d, d_seeds, W, N, d_labels, d_dmap, nnf.as<int>(), dis.as<float>(), coef, d_qnn, d_qw);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    c->prof_acc.kernel_launches += 5;
    tr.mark("knn search + query");
    if (h_over) {
        set_error("sfgpu_epic: neighbour search heap overflow (a seed with more than 2048 open graph nodes)");
        return SFGPU_ERR_NOMEM;
    }
    return SFGPU_OK;
}

} // namespace sf

using namespace sf;

extern "C" {

void epic_params_default(epic_params_t *params) { // epic.cpp:131-140
    if (!params) return;
    strcpy(params->method, "LA");
    params->saliency_th = 0.045f;
    params->pref_nn = 25;
    params->pref_th = 5.0f;
    params->nn = 100;
    params->coef_kernel = 0.8f;
    params->euc = 0.001f;
    params->verbose = 0;
}

} // extern "C"

// runs `body` with the context's arena installed, growing the arena and repeating the call while it does not fit
template <typename F> static int with_arena(sfgpu_ctx *c, size_t first_guess, F body) {
    if (!c->epic_arena) c->epic_arena = new EpicArena();
    EpicArena *ar = c->epic_arena;
    for (int attempt = 0; attempt < 4; attempt++) {
        // first call: the estimate; after an overflow: the recorded high-water mark plus a margin.  A call that fits
        // never touches the allocation.
        const size_t want = ar->overflow ? ar->high + ar->high / 4 : std::max(ar->cap, first_guess);
        if (want > ar->cap) {
            SF_CUDA(cudaStreamSynchronize(c->stream));
            if (ar->base) cudaFree(ar->base);
            ar->base = nullptr;
            ar->cap = 0;
            SF_CUDA(cudaMalloc(&ar->base, want));
            ar->cap = want;
        }
        ar->off = 0;
        ar->high = 0;
        ar->overflow = false;
        g_arena = ar;
        const int rc = body();
        g_arena = nullptr;
        if (!ar->overflow) return rc;
    }
    set_error("sfgpu_epic: workspace arena could not be sized");
    return SFGPU_ERR_NOMEM;
}

// epic() on n items of one geometry on device planes (the checks of epic_check_args have passed, euc is in the edge costs).
// Every step runs over all items at once; the host filters and compacts each item's match list in the reference's order.
// d_cost: the items' W x H edge costs one after another; d_lab: their Lab images, 3 planes of g each (only the saliency
// filter reads them; null when it is off); d_flow: item k's flow x at 2 k P, flow y at (2 k + 1) P, written whole (padding
// zeroed).  Runs with the arena installed; the flow kernels are left queued on the context's stream.  sstat: n entries.
static int epic_core(sfgpu_ctx *c, int n, Geom g, const float *d_cost_in, const float *d_lab, const float_image *const *input_matches,
                     const epic_params_t *params, float *d_flow, sfgpu_epic_stats_t *sstat, const Caller &who) {
    const int W = g.W, H = g.H;
    const bool la = strcmp(params->method, "LA") == 0;
    cudaStream_t st = c->stream;
    EpicTrace trace(st);
    const size_t N = (size_t)W * H, P = g.plane();
    memset(sstat, 0, (size_t)n * sizeof(sfgpu_epic_stats_t));

    // ---- rectify_corres (epic.cpp:13-27)
    std::vector<std::vector<float>> m4((size_t)n);
    std::vector<int> nm((size_t)n);
    for (int k = 0; k < n; k++) {
        const float_image *in = input_matches[k];
        nm[k] = in->ty;
        m4[k].resize((size_t)in->ty * 4);
        for (int i = 0; i < nm[k]; i++) {
            const float *r = in->pixels + (size_t)i * in->tx;
            m4[k][4 * i + 0] = std::max(0.0f, std::min(r[0], (float)(W - 1)));
            m4[k][4 * i + 1] = std::max(0.0f, std::min(r[1], (float)(H - 1)));
            m4[k][4 * i + 2] = std::max(0.0f, std::min(r[2], (float)(W - 1)));
            m4[k][4 * i + 3] = std::max(0.0f, std::min(r[3], (float)(H - 1)));
        }
        sstat[k].matches_in = nm[k];
    }
    DevBuf d_labels, d_dmap;
    if (!d_labels.alloc(n * N * 4) || !d_dmap.alloc(n * N * 4)) return SFGPU_ERR_CUDA;

    EpicGeo eg;
    eg.W = W; eg.H = H;

    auto compact = [&](int k, const unsigned char *keep) {
        int ii = 0;
        for (int i = 0; i < nm[k]; i++)
            if (keep[i]) {
                if (ii != i) memcpy(&m4[k][4 * (size_t)ii], &m4[k][4 * (size_t)i], 4 * sizeof(float));
                ii++;
            }
        nm[k] = ii;
    };
    auto all_have_matches = [&]() {
        for (int k = 0; k < n; k++)
            if (nm[k] <= 0) {
                set_error(who.at(k) + "no match survived the filters");
                return false;
            }
        return true;
    };

    // ---- saliency filter (epic.cpp:60-77) on the Lab planes; an item's 13 work planes follow those of the item before it
    if (params->saliency_th) {
        ArenaScope sal_scope;
        DevBuf work;
        const size_t zs = 13 * P;
        if (!work.alloc(n * zs * 4)) return SFGPU_ERR_CUDA;
        float *d_tmp = work.as<float>(), *d_sm = d_tmp + 3 * P, *d_ix = d_tmp + 6 * P, *d_iy = d_tmp + 9 * P;
        float *d_xx = d_tmp + 12 * P; // xy, yy reuse d_tmp / d_sm planes below
        const ConvTaps pre = gaussian_taps(0.8f), post = gaussian_taps(1.0f);
        ConvTaps der;
        memset(&der, 0, sizeof(der));
        der.order = 1; der.c[0] = -0.5f; der.c[1] = 0.0f; der.c[2] = 0.5f; // convolution_new(1, {0, -0.5}, odd)
        dim3 grid = grid2(W, H);
        grid.z = n;
        k_conv_any<<<grid, dim3(32, 8), 0, st>>>(g, d_lab, d_tmp, pre, 0, 3, zs, 3 * P);
        k_conv_any<<<grid, dim3(32, 8), 0, st>>>(g, d_tmp, d_sm, pre, 1, 3, zs, zs);
        k_conv_any<<<grid, dim3(32, 8), 0, st>>>(g, d_sm, d_ix, der, 0, 3, zs, zs);
        k_conv_any<<<grid, dim3(32, 8), 0, st>>>(g, d_sm, d_iy, der, 1, 3, zs, zs);
        float *d_xy = d_tmp, *d_yy = d_tmp + P, *d_t = d_tmp + 2 * P, *d_sal = d_sm;
        k_autocorr<<<grid, dim3(32, 8), 0, st>>>(g, d_ix, d_iy, d_xx, d_xy, d_yy, zs);
        float *planes[3] = {d_xx, d_xy, d_yy};
        for (int k = 0; k < 3; k++) {
            k_conv_any<<<grid, dim3(32, 8), 0, st>>>(g, planes[k], d_t, post, 0, 1, zs, zs);
            k_conv_any<<<grid, dim3(32, 8), 0, st>>>(g, d_t, planes[k], post, 1, 1, zs, zs);
        }
        k_min_eig<<<grid, dim3(32, 8), 0, st>>>(g, d_xx, d_xy, d_yy, d_sal, zs);
        c->prof_acc.kernel_launches += 12;
        std::vector<int> pos;
        for (int k = 0; k < n; k++)
            for (int i = 0; i < nm[k]; i++) { // the reference indexes with (int)(y * stride + x) on the float coordinates
                const int idx = (int)(m4[k][4 * i + 1] * (float)g.S + m4[k][4 * i]);
                pos.push_back(idx % g.S);
                pos.push_back(idx / g.S);
                pos.push_back(k);
            }
        const int total = (int)(pos.size() / 3);
        DevBuf d_pos, d_val;
        if (!d_pos.alloc(pos.size() * 4 + 4) || !d_val.alloc((size_t)total * 4 + 4)) return SFGPU_ERR_CUDA;
        std::vector<float> sal((size_t)total);
        if (total > 0) {
            SF_CUDA(cudaMemcpyAsync(d_pos.p, pos.data(), pos.size() * 4, cudaMemcpyHostToDevice, st));
            k_gather_plane<<<(total + 255) / 256, 256, 0, st>>>(total, d_pos.as<int>(), g, d_sal, zs, d_val.as<float>());
            SF_CUDA(cudaMemcpyAsync(sal.data(), d_val.p, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
        }
        SF_CUDA(cudaStreamSynchronize(st));
        std::vector<unsigned char> keep((size_t)total);
        for (int i = 0; i < total; i++) keep[i] = sal[i] >= params->saliency_th;
        for (int k = 0, at = 0; k < n; k++) {
            const int before = nm[k];
            compact(k, keep.data() + at);
            at += before;
        }
    }
    for (int k = 0; k < n; k++) sstat[k].matches_after_saliency = nm[k];
    trace.mark("[rectify + saliency filter]");
    if (!all_have_matches()) return SFGPU_ERR_ARG;

    // the match lists of all items, concatenated: seed ids are global (EpicItems)
    std::vector<int> seeds;
    std::vector<float> vects;
    EpicItems items;
    DevBuf d_seeds, d_vects, d_qnn, d_qw, d_est, d_keep;
    const size_t match_mark = g_arena->mark();
    auto upload_matches = [&](int nn) -> int { // nns = min(nn, the item's matches) per item
        g_arena->release(match_mark); // the buffers of the previous (larger) match lists
        items.n = n;
        items.off.assign(1, 0);
        items.nns.clear();
        seeds.clear();
        vects.clear();
        for (int k = 0; k < n; k++) { // matches_to_seeds / matches_to_vects (:30-57)
            items.off.push_back(items.off.back() + nm[k]);
            items.nns.push_back(std::min(nn, nm[k]));
            for (int i = 0; i < nm[k]; i++) {
                const float *r = &m4[k][4 * (size_t)i];
                seeds.push_back((int)r[0]);
                seeds.push_back((int)r[1]);
                vects.push_back(r[2] - r[0]);
                vects.push_back(r[3] - r[1]);
            }
        }
        const size_t ns = (size_t)items.ns(), ld = (size_t)items.nnmax();
        if (!d_seeds.alloc(ns * 8) || !d_vects.alloc(ns * 8) || !d_qnn.alloc(ns * ld * 4) || !d_qw.alloc(ns * ld * 4) || !d_est.alloc(ns * 6 * 4) ||
            !d_keep.alloc(ns + 4))
            return SFGPU_ERR_CUDA;
        const int rcu = items.upload(st);
        if (rcu != SFGPU_OK) return rcu;
        SF_CUDA(cudaMemcpyAsync(d_seeds.p, seeds.data(), ns * 8, cudaMemcpyHostToDevice, st));
        SF_CUDA(cudaMemcpyAsync(d_vects.p, vects.data(), ns * 8, cudaMemcpyHostToDevice, st));
        return SFGPU_OK;
    };
    std::vector<int> sweeps((size_t)n);

    // ---- consistency filter (prefiltering, epic.cpp:80-127)
    if (params->pref_nn) {
        int rc = upload_matches(params->pref_nn + 1);
        if (rc != SFGPU_OK) return rc;
        const int ns = items.ns(), ld = items.nnmax();
        rc = nn_field(c, eg, d_cost_in, items, d_seeds.as<int>(), params->coef_kernel, d_labels.as<int>(), d_dmap.as<float>(), d_qnn.as<int>(),
                      d_qw.as<float>(), sweeps.data());
        if (rc != SFGPU_OK) return rc;
        for (int k = 0; k < n; k++) sstat[k].sweeps_prefilter = sweeps[k];
        k_fit_nw<<<(ns + 127) / 128, 128, 0, st>>>(ns, ld, items.d, d_qnn.as<int>(), d_qw.as<float>(), d_vects.as<float>(), d_est.as<float>());
        k_prefilter_flags<<<(ns + 127) / 128, 128, 0, st>>>(ns, d_est.as<float>(), d_vects.as<float>(), params->pref_th * params->pref_th,
                                                          d_keep.as<unsigned char>());
        c->prof_acc.kernel_launches += 2;
        std::vector<unsigned char> keep((size_t)ns);
        SF_CUDA(cudaMemcpyAsync(keep.data(), d_keep.p, (size_t)ns, cudaMemcpyDeviceToHost, st));
        SF_CUDA(cudaStreamSynchronize(st));
        for (int k = 0; k < n; k++) compact(k, keep.data() + items.off[k]);
    }
    for (int k = 0; k < n; k++) sstat[k].matches_after_consistency = nm[k];
    trace.mark("[consistency filter total]");
    if (!all_have_matches()) return SFGPU_ERR_ARG;

    // ---- interpolation (epic.cpp:184-219)
    int rc = upload_matches(params->nn);
    if (rc != SFGPU_OK) return rc;
    const int ns = items.ns(), ld = items.nnmax();
    rc = nn_field(c, eg, d_cost_in, items, d_seeds.as<int>(), params->coef_kernel, d_labels.as<int>(), d_dmap.as<float>(), d_qnn.as<int>(),
                  d_qw.as<float>(), sweeps.data());
    if (rc != SFGPU_OK) return rc;
    for (int k = 0; k < n; k++) sstat[k].sweeps_interpolation = sweeps[k];
    SF_CUDA(cudaMemsetAsync(d_flow, 0, n * 2 * P * 4, st));
    if (la)
        k_fit_la<<<(ns + 127) / 128, 128, 0, st>>>(ns, ld, items.d, d_qnn.as<int>(), d_qw.as<float>(), d_seeds.as<int>(), d_vects.as<float>(),
                                                   d_est.as<float>());
    else k_fit_nw<<<(ns + 127) / 128, 128, 0, st>>>(ns, ld, items.d, d_qnn.as<int>(), d_qw.as<float>(), d_vects.as<float>(), d_est.as<float>());
    dim3 grid = grid2(W, H);
    grid.z = n;
    k_apply<<<grid, dim3(32, 8), 0, st>>>(g, d_labels.as<int>(), d_est.as<float>(), la ? 1 : 0, d_flow, d_flow + P, 2 * P);
    c->prof_acc.kernel_launches += 2;
    trace.mark("[interpolation total]");
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

// sfgpu_epic / sfgpu_epic_batch: the caller's edge costs and Lab images go up, the flows come down
static int epic_host(sfgpu_ctx *c, int n, image_t *const *flowx, image_t *const *flowy, const color_image_t *const *im,
                     const float_image *const *input_matches, float_image *const *edges, const epic_params_t *params, sfgpu_epic_stats_t *stats,
                     const Caller &who) {
    const Geom g{im[0]->width, im[0]->height, flowx[0]->stride};
    const size_t N = (size_t)g.W * g.H, P = g.plane();
    const bool sal = params->saliency_th != 0;
    DevBuf d_cost, d_lab, d_flow;
    if (!d_cost.alloc(n * N * 4) || !d_flow.alloc(n * 2 * P * 4) || (sal && !d_lab.alloc(n * 3 * P * 4))) return SFGPU_ERR_CUDA;
    {   // (pageable caller arrays go through the multi-threaded staging path, sf_hostcopy.cu: 30+ instead of 11 GB/s)
        std::vector<HostCopy> up;
        for (int k = 0; k < n; k++) up.push_back({d_cost.as<float>() + k * N, edges[k]->pixels, N * 4});
        if (sal)
            for (int k = 0; k < n; k++) up.push_back({d_lab.as<float>() + k * 3 * P, im[k]->c1, 3 * P * 4});
        const int rcu = host_copies(c, up, true);
        if (rcu != SFGPU_OK) return rcu;
    }
    std::vector<sfgpu_epic_stats_t> sstat((size_t)n);
    int rc = epic_core(c, n, g, d_cost.as<float>(), sal ? d_lab.as<float>() : nullptr, input_matches, params, d_flow.as<float>(), sstat.data(), who);
    if (rc != SFGPU_OK) return rc;
    EpicTrace trace(c->stream);
    // every check has passed: only now are the caller's flow planes written
    std::vector<HostCopy> down;
    for (int k = 0; k < n; k++) {
        down.push_back({d_flow.as<float>() + 2 * k * P, flowx[k]->data, P * 4});
        down.push_back({d_flow.as<float>() + (2 * k + 1) * P, flowy[k]->data, P * 4});
    }
    rc = host_copies(c, down, false);
    if (rc != SFGPU_OK) return rc;
    SF_CUDA(cudaStreamSynchronize(c->stream));
    trace.mark("[flow download]");
    SF_CUDA(cudaGetLastError());
    if (stats)
        for (int k = 0; k < n; k++) stats[k] = sstat[k];
    return SFGPU_OK;
}

namespace sf {

int epic_check_args(sfgpu_ctx *c, int n, image_t *const *flowx, image_t *const *flowy, const color_image_t *const *im,
                    const float_image *const *input_matches, float_image *const *edges, const epic_params_t *params, const Caller &who,
                    const char *const names[3], Geom &g) {
    if (n < 1) {
        set_error(std::string(who.fn) + ": no item (n < 1)");
        return SFGPU_ERR_ARG;
    }
    if (!c || !flowx || !flowy || !im || !input_matches || !edges || !params) {
        set_error(std::string(who.fn) + ": null argument");
        return SFGPU_ERR_ARG;
    }
    for (int k = 0; k < n; k++)
        if (!flowx[k] || !flowy[k] || !im[k] || !input_matches[k] || !edges[k] || !input_matches[k]->pixels || !edges[k]->pixels) {
            set_error(who.at(k) + "null argument");
            return SFGPU_ERR_ARG;
        }
    if (!arg_geom(who.at(0), names[2], im[0], g)) return SFGPU_ERR_ARG;
    for (int k = 0; k < n; k++) {
        if (!arg_is(who.at(k), names[0], flowx[k], g) || !arg_is(who.at(k), names[1], flowy[k], g)) return SFGPU_ERR_ARG;
        if (edges[k]->tx != g.W || edges[k]->ty != g.H) {
            set_error(who.at(k) + "edges: must have the image's width x height (" + std::to_string(g.W) + "x" + std::to_string(g.H) + ")");
            return SFGPU_ERR_ARG;
        }
        if (input_matches[k]->tx < 4) {
            set_error(who.at(k) + "input_matches: need >= 4 columns (x1 y1 x2 y2)");
            return SFGPU_ERR_ARG;
        }
    }
    if (strcmp(params->method, "LA") != 0 && strcmp(params->method, "NW") != 0) {
        set_error(std::string(who.fn) + ": method " + params->method + " not recognized");
        return SFGPU_ERR_ARG;
    }
    return SFGPU_OK;
}

void epic_add_euc(int n, float_image *const *edges, float euc) {
    if (!euc) return;
    for (int k = 0; k < n; k++) {
        const size_t N = (size_t)edges[k]->tx * edges[k]->ty;
        for (size_t i = 0; i < N; i++) edges[k]->pixels[i] += euc;
    }
}

size_t epic_arena_guess(int n, size_t N) { return n * N * 4 * 24 + ((size_t)64 << 20); }

int epic_device(sfgpu_ctx *c, int n, Geom g, const float *d_cost, const float *d_lab, const float_image *const *input_matches,
                const epic_params_t *params, float *d_flow, sfgpu_epic_stats_t *stats, const Caller &who) {
    return with_arena(c, epic_arena_guess(n, (size_t)g.W * g.H),
                      [&]() { return epic_core(c, n, g, d_cost, d_lab, input_matches, params, d_flow, stats, who); });
}

} // namespace sf

// the argument checks of epic() on n items, all before anything is touched; then edges += euc in every caller's array, like
// the reference (epic.cpp:155-163), once whatever the arena does below
static int epic_batch(sfgpu_ctx *c, int n, image_t *const *flowx, image_t *const *flowy, const color_image_t *const *im,
                      const float_image *const *input_matches, float_image *const *edges, const epic_params_t *params, sfgpu_epic_stats_t *stats,
                      const Caller &who) {
    const char *const names[3] = {"flowx", "flowy", "im"};
    Geom g;
    const int rc = epic_check_args(c, n, flowx, flowy, im, input_matches, edges, params, who, names, g);
    if (rc != SFGPU_OK) return rc;
    for (int k = 1; k < n; k++) // im[0] gave g
        if (!arg_is(who.at(k), "im", im[k], g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    epic_add_euc(n, edges, params->euc);
    return with_arena(c, epic_arena_guess(n, (size_t)im[0]->width * im[0]->height),
                      [&]() { return epic_host(c, n, flowx, flowy, im, input_matches, edges, params, stats, who); });
}

extern "C" {

int sfgpu_epic(sfgpu_ctx *c, image_t *flowx, image_t *flowy, const color_image_t *im, const float_image *input_matches, float_image *edges,
               const epic_params_t *params, sfgpu_epic_stats_t *stats) {
    return epic_batch(c, 1, &flowx, &flowy, &im, &input_matches, &edges, params, stats, Caller{"sfgpu_epic", nullptr, 0});
}

int sfgpu_epic_batch(sfgpu_ctx *c, int n, image_t *const *flowx, image_t *const *flowy, const color_image_t *const *im,
                     const float_image *const *input_matches, float_image *const *edges, const epic_params_t *params, sfgpu_epic_stats_t *stats) {
    return epic_batch(c, n, flowx, flowy, im, input_matches, edges, params, stats, Caller{"sfgpu_epic_batch", "item", 0});
}

} // extern "C"

// operator twin of dist_trf_nnfield_subset (epic_aux.cpp:350) with the seeds as query points: labels (W*H), best and dist
// (ns x nn; dist BEFORE the exp kernel) for operator-level parity tests
static int nnfield_impl(sfgpu_ctx *c, int *best, float *dist, int *labels, const int *seeds, int ns, int nn, const float *cost, int w, int h,
                        int *sweeps) {
    if (!c || !best || !dist || !labels || !seeds || !cost || ns < 1 || nn < 1 || nn > ns || w < 1 || h < 1) {
        set_error("sfgpu_epic_nnfield: bad argument");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t N = (size_t)w * h;
    EpicGeo eg;
    eg.W = w; eg.H = h;
    EpicItems items;
    items.n = 1;
    items.off = {0, ns};
    items.nns = {nn};
    DevBuf d_cost, d_labels, d_dmap, d_seeds, d_qnn, d_qw;
    if (!d_cost.alloc(N * 4) || !d_labels.alloc(N * 4) || !d_dmap.alloc(N * 4) || !d_seeds.alloc((size_t)ns * 8) || !d_qnn.alloc((size_t)ns * nn * 4) ||
        !d_qw.alloc((size_t)ns * nn * 4))
        return SFGPU_ERR_CUDA;
    int rc = items.upload(st);
    if (rc != SFGPU_OK) return rc;
    SF_CUDA(cudaMemcpyAsync(d_cost.p, cost, N * 4, cudaMemcpyHostToDevice, st));
    SF_CUDA(cudaMemcpyAsync(d_seeds.p, seeds, (size_t)ns * 8, cudaMemcpyHostToDevice, st));
    rc = nn_field(c, eg, d_cost.as<float>(), items, d_seeds.as<int>(), -1.0f /* raw distances */, d_labels.as<int>(), d_dmap.as<float>(), d_qnn.as<int>(),
                  d_qw.as<float>(), sweeps);
    if (rc != SFGPU_OK) return rc;
    SF_CUDA(cudaMemcpyAsync(labels, d_labels.p, N * 4, cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaMemcpyAsync(best, d_qnn.p, (size_t)ns * nn * 4, cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaMemcpyAsync(dist, d_qw.p, (size_t)ns * nn * 4, cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    return SFGPU_OK;
}


extern "C" {

int sfgpu_epic_nnfield(sfgpu_ctx *c, int *best, float *dist, int *labels, const int *seeds, int ns, int nn, const float *cost, int w, int h,
                       int *sweeps) {
    if (!c || w < 1 || h < 1) {
        set_error("sfgpu_epic_nnfield: bad argument");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(c->device));
    return with_arena(c, (size_t)w * h * 4 * 16 + ((size_t)64 << 20), [&]() { return nnfield_impl(c, best, dist, labels, seeds, ns, nn, cost, w, h, sweeps); });
}

} // extern "C"

