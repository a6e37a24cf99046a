// sf_internal.cuh -- internal declarations shared by the CUDA translation units of libslowflow_gpu.so.
// Nothing here is part of the ABI (see include/slowflow_gpu.h).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "slowflow_gpu.h"

namespace sf {

// ---------------------------------------------------------------------------------------------
// geometry of one pyramid level: W valid columns, H rows, S = ceil4(W) floats per row (image.c:25).
// Device planes use exactly the host layout, so a plane moves with one cudaMemcpyAsync.
// skip: optional device flag.  When it is set every kernel of the refinement chain returns at once: this is how the
// data-dependent early exit of the multi-frame outer loop (variational_mt.cpp:436-437) works without a host round trip --
// the host queues all outer iterations of an alternation, the reduction kernel that closes an iteration raises the flag,
// and the launches queued behind it fall through (sf_mt.cu).  NULL everywhere else.
struct Geom {
    int W, H, S;
    const int *skip = nullptr;
    __host__ __device__ size_t plane() const { return (size_t)S * H; }
#ifdef __CUDACC__
    __device__ __forceinline__ bool cancelled() const { return skip != nullptr && *reinterpret_cast<const volatile int *>(skip) != 0; }
#endif
};
static inline Geom make_geom(int w, int h) { return Geom{w, h, ((w + 3) / 4) * 4}; }

// thread-local error string behind sfgpu_last_error()
void set_error(const std::string &msg);
bool cuda_ok(cudaError_t e, const char *what);
#define SF_CUDA(call)                                         \
    do {                                                      \
        if (!::sf::cuda_ok((call), #call)) return SFGPU_ERR_CUDA; \
    } while (0)

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (sm_90+): every kernel of the refinement chain starts with pdl_enter() -- it lets the
// NEXT launch of the stream become resident while this grid drains, then waits until the PREVIOUS grid has completed
// and flushed its memory -- and is launched through launch_pdl().  A field is ~50 dependent launches of 10-140 us; the
// launch latency between them (about 2 us each) is what this hides.  Nothing above pdl_enter() may touch global memory.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

// ---------------------------------------------------------------------------------------------
// robust penalties (penalty_functions/*.h), selected at run time inside the kernels by a small POD
struct Penalty {
    int type;        // SF_ROBUST_*
    float eps_sq_f;  // epsilon_vec_sq / float epsilon_sq
    double eps_sq_d; // double epsilon_sq (ModL1, Lorentzian, Geman-McClure keep it in double)
    float trunc;     // TruncModifiedL1Norm::truncation
};
Penalty make_penalty(int type, float eps, float trunc);

// ---------------------------------------------------------------------------------------------
// kernel launchers (all asynchronous on `st`)

// K0: smoothness weight 0.5*exp(-coef*|grad lum|) (variational_aux.c:183 ; variational_aux_mt.cpp:673)
void launch_dpsis_weight(cudaStream_t st, Geom g, const float *im3, float *out, float coef, const float avg[3],
                         const float stdv[3], float divisor);
// K1: bilinear warp with integer time factor (variational_aux.c:18 ; variational_aux_mt.cpp:722)
void launch_warp(cudaStream_t st, Geom g, const float *src3, const float *wx, const float *wy, int factor,
                 float *dst3, float *mask /*nullable*/);
// K3: smoothness diffusivities.  reg.type < 0: two-frame form (variational_aux.c:84), else MT modes 0/1.
void launch_smoothness(cudaStream_t st, Geom g, const float *uu, const float *vv, const float *w, float alpha_factor,
                       Penalty reg, int mode, float *ph, float *pv);
// K3 fused with the flow update: smoothness of (wx + du, wy + dv), which is also stored to (wx_out, wy_out)
void launch_update_smoothness(cudaStream_t st, Geom g, const float *wx, const float *wy, const float *du, const float *dv,
                              const float *w, float alpha_factor, Penalty reg, int mode, float *wx_out, float *wy_out,
                              float *ph, float *pv);
// K2: derivatives + robust data term of ONE term, fused (sf_data.cu).  A term pairs two colour images:
//   m = 0.5*(B + A) (spatial derivatives are taken on it), z = zsign>0 ? B - A : A - B (temporal difference).
enum DataKind { DK_TWO_FRAME = 0, DK_MT_SUCC = 1, DK_MT_REF = 2, DK_DERIVS = 3 };
struct DataTermDesc {
    const float *A, *B; // 3-plane images
    int zsign;
    const float *mask;  // raw in-bounds mask of the warp
    int kind;           // DataKind
    float wd, wg;       // weights of the colour / gradient constancy parts (already scaled by rho/omega for MT)
    float s;            // MT time factor
    int dir;            // MT occlusion handling: 0 past term, 1 future term, -1 none
};
struct DataCommon {
    const float *du, *dv; // current increment (nullable: 0)
    const float *chw;     // channel weights, 3 planes (nullable: 1)
    size_t chw_pstride;   // floats between the channel-weight planes (full-resolution plane size, SURVEY Q14)
    const float *occ;     // occlusion labels -1/0/+1 (nullable)
    float data_norm;      // sum_s rho_s + omega_s (variational_mt.cpp:223-226)
    int dt_norm;          // slow_flow_dataterm
    Penalty pc, pg;       // psi_color, psi_grad
    bool accumulate;      // add to the existing a11..b2 instead of starting from 0
    // fuse_system: also add div(psi grad lap_u/lap_v) (variational_aux.c:153) and store the inverted 2x2
    // blocks exactly as sor_coupled's first sweep would (solver.c:101-106)
    bool fuse_system;
    const float *ph, *pv, *lap_u, *lap_v;
    float *a11, *a12, *a22, *b1, *b2;
};
void launch_data_term(cudaStream_t st, Geom g, const DataTermDesc &t, const DataCommon &cm);

// Multi-frame data pass in two kernels (sf_data.cu), replacing one launch_data_term per term:
//   launch_frame_derivs: the five spatial derivative images Ix Iy Ixx Ixy Iyy of ONE (warped) frame, 15 planes
//                        [derivative][channel], computed once per frame and outer iteration (the reference frame: once
//                        per level) with the filters and border rules of get_derivatives (variational_mt.cpp:87-166);
//   launch_mt_terms:     every term of variational_mt.cpp:343-361 in one pointwise pass.  A term's derivatives are linear
//                        in its two frames -- m = (A + B)/2, z = A - B -- so they are formed from the per-frame planes:
//                        Ix = (Ix_A + Ix_B)/2, Ixz = Ix_A - Ix_B, ...; A,b are accumulated in registers and the Laplacian
//                        and block inverse of fuse_system close the pass.
constexpr int MT_MAX_FRAMES = 2 * SF_MT_MAX_REF + 1, MT_MAX_TERMS = 4 * SF_MT_MAX_REF;
struct MtTerm {
    int fa, fb;        // frame indices of A and B (z = A - B)
    int mask_frame;    // frame whose warp mask gates the term
    int kind;          // DK_MT_SUCC / DK_MT_REF
    int dir;           // occlusion handling: 0 past term, 1 future term
    float wd, wg, s;
};
struct MtTermsArgs {
    int nterms;
    MtTerm term[MT_MAX_TERMS];
    const float *I[MT_MAX_FRAMES];    // warped frames (3 planes); the reference frame unwarped
    const float *D[MT_MAX_FRAMES];    // their derivative planes (15)
    const float *mask[MT_MAX_FRAMES]; // warp masks
};
void launch_frame_derivs(cudaStream_t st, Geom g, const float *image3, float *derivs15);
// launch_warp + launch_frame_derivs of ONE frame in one marching pass (sf_wderivs.cu)
void launch_warp_derivs(cudaStream_t st, Geom g, int num_sms, const float *src3, const float *wx, const float *wy, int factor,
                        float *warped3, float *mask, float *derivs15);
// ... of all warped frames of a window in ONE launch (they share the flow of the reference frame)
void launch_warp_derivs_batch(cudaStream_t st, Geom g, int num_sms, const float *wx, const float *wy, int nframes,
                              const float *const *src3, const int *factor, float *const *warped3, float *const *mask,
                              float *const *derivs15);
// force_scalar: the one-column-per-thread form with run-time penalty switch (A/B switch of the tests; also taken when a
// plane is not 8-byte aligned) instead of the packed two-columns-per-thread kernel
void launch_mt_terms(cudaStream_t st, Geom g, const MtTermsArgs &ta, const DataCommon &cm, bool force_scalar = false);
// K1+K2 fused, marching form (sf_prep.cu): warp + derivatives + two-frame data term + Laplacian + block inverse.
// Writes the same five planes as launch_warp + launch_data_term(fuse_system) without the warped image in HBM.
void launch_prep_two_frame(cudaStream_t st, Geom g, int num_sms, const float *im1, const float *im2, const float *wx, const float *wy, const float *du, const float *dv, const float *ph, const float *pv,
                           float half_delta_over3, float half_gamma_over3, float *a11, float *a12, float *a22, float *b1,
                           float *b2);
// One outer iteration of the two-frame loop with niter_inner == 1 in one pass (sf_prep.cu): launch_update_smoothness
// (du != nullptr: the flow is wx + du, stored to wx_out / wy_out) or launch_smoothness (du == nullptr) with the two-frame
// penalty and mode 1, followed by launch_prep_two_frame on that flow and its diffusivities (also stored to ph / pv) at
// a zero increment.  The same planes as the two launches, bit for bit.
void launch_prep_fused(cudaStream_t st, Geom g, int num_sms, const float *im1, const float *im2, const float *wx, const float *wy,
                       const float *du, const float *dv, const float *dpsis, float half_alpha, float half_delta_over3,
                       float half_gamma_over3, float *wx_out, float *wy_out, float *ph, float *pv, float *a11, float *a12,
                       float *a22, float *b1, float *b2);
// convolve_horiz / convolve_vert over `planes` planes (operator twins; order 1 = 3 taps, 2 = 5 taps)
void launch_convolve(cudaStream_t st, Geom g, const float *src, float *dst, bool vertical, int order, const float *coeffs,
                     int planes);
void launch_mean_diff(cudaStream_t st, size_t n, const float *im1, const float *im2, float *mean, float *dt);
// sub_laplacian as a gather (operator twin)
void launch_sub_laplacian(cudaStream_t st, Geom g, float *dst, const float *src, const float *ph, const float *pv);
// in-place inverse of the 2x2 blocks (operator twin of the first SOR sweep's prologue)
void launch_invert_blocks(cudaStream_t st, Geom g, float *a11, float *a12, float *a22, const float *ph, const float *pv);
// K5: dst = a + b over the whole plane (variational.c:60-65)
void launch_add(cudaStream_t st, Geom g, float *dst, const float *a, const float *b);
void launch_fill(cudaStream_t st, float *dst, size_t n, float v);

// ---------------------------------------------------------------------------------------------
// input side of the multi-frame path: what slow_flow.cpp does to every frame before the solver sees it
// packed 8-/16-bit frame (cv::Mat rows of `step` bytes, 1 or 3 interleaved channels) -> planar fp32 of g, exact, stride
// padding zeroed (mat2colorImg / colorMat2colorImg, utils/utils.h:122-160; sf_sequence.cu)
void launch_unpack_frame(cudaStream_t st, Geom g, const unsigned char *raw, size_t step, int channels, int bits, float *dst);
// separable Gaussian of cv::GaussianBlur (replicate border) and its taps (cv::getGaussianKernel) (sf_mt.cu)
struct BlurTaps { int r; float k[17]; }; // k[0] centre, k[i] at distance i
BlurTaps make_taps(double sigma);
void launch_blur(cudaStream_t st, Geom g, const float *src, float *tmp, float *dst, const BlurTaps &t, int planes);
// the pre-scaling of slow_flow.cpp:538-542 from src (gs) into dst (gd = sfgpu_prescale_size); tmp, blur: 3 planes of gs
void launch_prescale(cudaStream_t st, Geom gs, const float *src, float *tmp, float *blur, Geom gd, float *dst, float scale);
// normalize() (variational_mt.cpp:17-85) in four steps: per frame the block partials of the channel sums (norm_blocks(g) x 6
// doubles), from a planar fp32 frame or from the packed integer frame that unpacks to it (same partials); the statistics
// of F frames from their partials, in a fixed order on the host; the in-place normalisation of a frame (a channel with
// std <= 0 is left as it is); the values the reference publishes (6 significant digits) into p->img_norm_*.
int norm_blocks(Geom g);
void launch_norm_sums(cudaStream_t st, Geom g, const float *im, double *sums);
void launch_norm_sums_packed(cudaStream_t st, Geom g, const unsigned char *raw, size_t step, int channels, int bits, double *sums);
void norm_statistics(const double *partials, int F, Geom g, double avg[3], double sd[3]);
void launch_norm_apply(cudaStream_t st, Geom g, float *im, const double avg[3], const double sd[3]);
void norm_publish(const double avg[3], const double sd[3], sf_mt_params_t *p);

// ---------------------------------------------------------------------------------------------
// K4: red-black SOR on the coupled 2x2-block 5-point system (solver.c:63, re-ordered).
// The SOR arena is 11 consecutive planes: a11' a12' a22' b1 b2 psi_h psi_v duA dvA duB dvB.
enum SorPlane { SP_A11 = 0, SP_A12, SP_A22, SP_B1, SP_B2, SP_PH, SP_PV, SP_DUA, SP_DVA, SP_DUB, SP_DVB, SP_COUNT };

struct SorPlan {
    Geom g{0, 0, 0};
    float *arena = nullptr; // SP_COUNT planes
    CUtensorMap tmap;       // 3-D (x, y, plane) views of the arena: box = a tile of the first 4 coefficient planes,
    CUtensorMap tmap_gb;    //   ... of the other 3,
    CUtensorMap tmap_iter;  //   ... of a du,dv plane pair,
    CUtensorMap tmap_row;   //   ... one row of one plane
    CUtensorMap tmap_s_coef, tmap_s_iter, tmap_s_row; // the same three views with the boxes of the streaming kernel
    bool tmap_valid = false;
    int num_sms = 0;
    // device words of the tiled kernel's multi-pass launches: [0] ticket counter, [1] CTAs that have left, [2] generation,
    // [4 + tile] generation + passes the tile has completed.  Owned by the plan (sor_plan_release); a plan serves one
    // stream at a time.
    static constexpr size_t SYNC_TILES = 1 << 16;
    unsigned *sync = nullptr;
    size_t sync_tiles = 0;
};
// per-device kernel attributes (dynamic shared memory opt-in); called once per context on its device
bool sor_device_init();
bool data_term_device_init();
// Encode the TMA descriptor for an arena.  Returns false (and sets the error) on failure.
bool sor_plan_init(SorPlan &plan, Geom g, float *arena, int num_sms);
void sor_plan_release(SorPlan &plan);
// Runs `iterations` sweeps; the iterate starts in (duA,dvA) when *cur==0 or (duB,dvB) when *cur==1 and
// *cur is updated to the buffer holding the result.  zero_init: treat the initial iterate as 0.
// variant 0: tiled / temporally blocked (fuse sweeps per launch), variant 1: one launch per half sweep,
// variant 2: streaming wavefront (sf_sor_stream.cu).
// Returns the number of kernel launches issued (negative on error).
int launch_sor(cudaStream_t st, SorPlan &plan, int iterations, float omega, int variant, int fuse, int *cur,
               bool zero_init);
bool sor_stream_device_init();
void sor_stream_boxes(unsigned boxes[3][3]);
int launch_sor_stream(cudaStream_t st, SorPlan &plan, int iterations, float omega, int fuse, int *cur, bool zero_init);

} // namespace sf
