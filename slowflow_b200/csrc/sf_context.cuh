// sf_context.cuh -- the per-thread / per-device context behind sfgpu_ctx.
#pragma once
#include <vector>

#include "sf_internal.cuh"

namespace sf {
struct MtWork; // multi-frame workspace (sf_mt.cu), kept between calls
void mt_work_free(MtWork *w);
struct EpicArena; // workspace of the EPIC interpolation (sf_epic.cu)
void epic_arena_free(EpicArena *a);
struct DeviceCut; // device-side grid min-cut workspace (sf_mincut.cu)
void device_cut_free(DeviceCut *d);
struct HostStager; // pinned bounce buffers for pageable caller memory (sf_hostcopy.cu)
void host_stager_free(HostStager *h);
struct HostCopy {
    void *dev;
    void *host;
    size_t bytes;
};
} // namespace sf

struct sfgpu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int num_sms = 148;

    int sor_variant = 0; // 0 tiled, 1 per-half-sweep launches
    int data_variant = 0; // 0 fused marching data pass, 1 separate warp + tile kernel, 2 as 0 with a separate smoothness pass (env SLOWFLOW_GPU_DATA_VARIANT)
    int sor_fuse = 0;    // 0 = auto
    int mt_warp_variant = 0; // 0: fused warp + per-frame derivatives (sf_wderivs.cu), 1: k_warp + k_data_term<DK_DERIVS> (env SLOWFLOW_GPU_MT_WARP_VARIANT)
    bool mt_terms_scalar = false; // env SLOWFLOW_GPU_MT_TERMS_SCALAR: one column per thread in the all-terms pass (A/B switch)
    int mt_data_variant = 0; // 0: per-frame derivative planes + one pointwise all-terms pass, 1: one fused kernel per term (env SLOWFLOW_GPU_MT_DATA_VARIANT)

    // ---- level workspace (one allocation, re-made when the geometry grows)
    sf::Geom g{0, 0, 0};
    float *ws = nullptr;
    size_t ws_floats = 0;
    sf::SorPlan sor;
    float *wim = nullptr;   // 3 planes: warped second image (two-frame)
    float *mask = nullptr;  // 1 plane
    float *uu = nullptr, *vv = nullptr;
    float *dpsis = nullptr;

    // ---- host-API staging (device copies of caller buffers)
    float *io = nullptr; // im1(3) im2(3) wx wy   [+ ring for the sequence API]
    size_t io_floats = 0;

    // ---- copy pipeline (CopyPipeline, sf_hostcopy.cu; created at first use) and sequence frames (sf_sequence.cu)
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t copy_ev[3][4] = {}; // rings of "uploaded" / "compute passed" / "drained" events
    unsigned char *seq_raw = nullptr; // 3 slots of packed 8-/16-bit frames awaiting their on-device conversion
    size_t seq_raw_bytes = 0;        // bytes per slot
    sf::Geom seq_geom{0, 0, 0};      // geometry of the frame ring left by the last sequence call
    int seq_last_slot = -1;          // ring slot that holds the last frame of that call (-1: none)

    // ---- multi-frame frame cache (sfgpu_mt_frame_cache): device copies of level-0 frames keyed by the caller's host
    // pointer, for callers that solve many windows over one immutable sequence (consecutive windows share frames, the
    // backward window of a jet reads the frames of its forward window)
    struct MtFrameSlot { const void *host = nullptr; size_t floats = 0; float *dev = nullptr; unsigned long long stamp = 0; };
    std::vector<MtFrameSlot> mt_cache;
    float *mt_cache_pool = nullptr; // ONE allocation for all slots (cudaMalloc / cudaFree per frame cost tens of ms each next to registered host memory)
    size_t mt_cache_slot_floats = 0;
    unsigned long long mt_cache_clock = 0;
    unsigned long long mt_cache_hits = 0, mt_cache_misses = 0;

    // ---- profiling
    bool prof = false;
    struct EvPair { cudaEvent_t a, b; int kind; };
    std::vector<EvPair> ev_pending;
    std::vector<cudaEvent_t> ev_free;
    sfgpu_profile_t prof_acc{};

    sfgpu_mt_stats_t mt_stats{};
    sf::MtWork *mtw = nullptr;
    sf::HostStager *stager = nullptr;
    sf::DeviceCut *cut = nullptr;
    sf::EpicArena *epic_arena = nullptr;
    bool host_mincut = false; // env SLOWFLOW_GPU_HOST_MINCUT=1: occlusion labelling on the host (sf_gridcut.hpp), A/B only
    bool staged_host_copies = true; // env SLOWFLOW_GPU_STAGED_COPIES=0 switches the multi-threaded staging off

    // helpers
    int ensure_workspace(sf::Geom geom);
    int ensure_io(size_t floats);
    cudaEvent_t get_event();
    void prof_begin(int kind, cudaEvent_t &a);
    void prof_end(int kind, cudaEvent_t a);
    int prof_collect();
};

namespace sf {
// copies between caller (host) buffers and the device for one call, one direction (sf_hostcopy.cu)
int host_copies(sfgpu_ctx *c, const std::vector<HostCopy> &list, bool h2d);
// The copies of a call that streams caller memory stage by stage (0, 1, 2, ...: pairs, chunks) while the compute stream
// works (sf_hostcopy.cu).  start() decides once: if any caller buffer is pageable, every copy is a host_copies() on the
// compute stream in program order and the ordering calls do nothing.  Otherwise uploads and downloads run on their own
// streams, ordered by rings of 4 events per kind (stage & 3), so a stage waited for must be one of the last 4 of its kind.
// A stage argument < 0 means no wait.
class CopyPipeline {
  public:
    explicit CopyPipeline(sfgpu_ctx *c) : c(c) {}
    // buffers: every caller buffer of the call.  The first upload comes after the work already on the compute stream.
    int start(const std::vector<const void *> &buffers);
    // stage k's uploads, after compute has passed stage `passed` and stage `drained`'s downloads have finished
    int upload(int k, const std::vector<HostCopy> &list, int passed = -1, int drained = -1);
    int wait(int uploaded, int drained = -1); // the compute stream waits for these stages' uploads / downloads
    int pass(int k);                          // compute has passed stage k with the work queued so far
    // stage k's downloads, after compute has passed it (the last pass(k)); may be called several times per stage
    int download(int k, const std::vector<HostCopy> &list);
    int finish(int status); // drains all three streams; returns `status` if it is an error, else the first error met

  private:
    sfgpu_ctx *c;
    bool pageable = false;
};
// two-frame refinement on device planes (variational.c:19-82 + :101-143)
int run_two_frame(sfgpu_ctx *c, Geom g, float *d_wx, float *d_wy, const float *d_im1, const float *d_im2,
                  const variational_params_t *params);

// ---- image arguments of the host-buffer entries (the container contract of slowflow_gpu.h:30-44).  An entry copies whole
// planes of P = stride * height floats (3 P from a colour image's c1), with P from the call's one geometry.
// Names the entry point in error messages, and in a batch or sequence the item ("item" / "pair" numbered from `first`;
// null: none): at(k) is "<fn>: " or "<fn>: <item> <first + k>: ".  With per > 1, per consecutive k share an item and
// part names them: "<fn>: <item> <first + k / per> <part[k % per]>: " (the two windows of a jet).
struct Caller {
    const char *fn;
    const char *item;
    int first;
    int per = 1;
    const char *const *part = nullptr;
    std::string at(int k) const;
};
// A failed check sets "<at><name>: <what>" and returns false; the entry then returns SFGPU_ERR_ARG before it touches the
// device or any caller buffer.
// arg_geom: the call's geometry g from argument `name`: non-null data, width and height >= 1, stride = ceil4(width), and
// a colour image planar and contiguous (c2 = c1 + P, c3 = c2 + P).
bool arg_geom(const std::string &at, const std::string &name, const image_t *a, Geom &g);
bool arg_geom(const std::string &at, const std::string &name, const color_image_t *a, Geom &g);
// arg_is: argument `name` has non-null data and exactly the geometry g (a colour image: also planar and contiguous)
bool arg_is(const std::string &at, const std::string &name, const image_t *a, Geom g);
bool arg_is(const std::string &at, const std::string &name, const color_image_t *a, Geom g);

// arg_frame_int: an integer frame (sf_frame_int_t) of `bits` 8 or 16 with non-null data, width x height of g, 1 or 3
// channels and a row step of at least width * channels samples that is a multiple of the sample size
bool arg_frame_int(const std::string &at, const std::string &name, const sf_frame_int_t &q, Geom g, int bits);

// One window of Variational_MT::variational (variational_mt.cpp:526-784) on device planes (sf_mt.cu), in three steps:
//   mt_window_layout  pyramid geometry and the planes of the context's multi-frame workspace.  own_frames0: the level-0
//                     frames are workspace planes too (else the caller sets frames[0][f] to its own device frames);
//                     chw_plane: 3 planes for channel weights (chw points at them; the caller may point it elsewhere).
//                     levels == 0: the reference computes nothing and nothing else may be called.
//   mt_window_build   after the caller has filled frames[0], wx, wy (and chw): the coarser levels' frames, the initial
//                     flow on the coarsest level, the level workspace
//   mt_window_solve   coarse-to-fine; the flow of level 0 is left in wx, wy, the occlusion labels in occ.  Synchronises the
//                     context's stream once per level.
struct MtWindow {
    int levels = 0, ref = 0;
    float sigma = 0.f;
    std::vector<Geom> geoms;                  // per level
    std::vector<std::vector<float *>> frames; // [level][frame], 3 planes each
    std::vector<float *> warped, masks, derivs;
    float *wx = nullptr, *wy = nullptr, *wxb = nullptr, *wyb = nullptr, *uu = nullptr, *vv = nullptr, *odu = nullptr,
          *odv = nullptr, *dpsis = nullptr, *occ = nullptr, *d0 = nullptr, *d1 = nullptr, *blur_tmp = nullptr, *chw_plane = nullptr;
    const float *chw = nullptr;
};
int mt_window_layout(sfgpu_ctx *c, const sf_mt_params_t *p, Geom g0, bool own_frames0, bool chw_plane, MtWindow &w);
int mt_window_build(sfgpu_ctx *c, MtWindow &w);
int mt_window_solve(sfgpu_ctx *c, const sf_mt_params_t *p, bool one_direction, MtWindow &w, float avg_change[2]);

// exact binary Potts min-cut on the device (sf_mincut.cu); results in occ / device_cut_labels(), status after a stream sync
int device_grid_mincut(sfgpu_ctx *c, DeviceCut *&cut, int W, int H, long long *tr_dev, long long pair_cap, float *occ, int S);
const int *device_cut_status(const DeviceCut *cut);       // {0 = converged, phases, grid-wide passes}
const unsigned char *device_cut_labels(const DeviceCut *cut); // dense W*H labels (device memory)
// one sor_coupled call on the context's SOR arena (profiled)
int run_sor(sfgpu_ctx *c, int iterations, float omega, int *cur, bool zero_init);

// ---- EPIC interpolation (sf_epic.cu)
// The argument checks of sfgpu_epic_batch on n items: null pointers, the call's geometry g from im[0], flows and edges of
// that geometry, >= 4 match columns, the method.  Touches nothing.  names: of flowx, flowy and im[0] in the caller's
// signature.  The callers check the other images against g: the batch its im[k], sfgpu_epicflow_sequence frame k + 1
// under pair k, the first pair that reads it.
int epic_check_args(sfgpu_ctx *c, int n, image_t *const *flowx, image_t *const *flowy, const color_image_t *const *im,
                    const float_image *const *input_matches, float_image *const *edges, const epic_params_t *params, const Caller &who,
                    const char *const names[3], Geom &g);
// edges[k] += euc in the caller's arrays (epic.cpp:155-163)
void epic_add_euc(int n, float_image *const *edges, float euc);
// epic() on n items of one geometry on device planes, after epic_check_args and epic_add_euc.  d_cost: the items' W x H
// edge costs one after another; d_lab: their Lab images, 3 planes of g each (read by the saliency filter only; may be null
// when it is off); d_flow: item k's flow x at 2 k P and flow y at (2 k + 1) P, whole planes with zeroed padding.  stats: n
// entries.  The last kernels are left queued on the context's stream; on an error d_flow is not fully written.
int epic_device(sfgpu_ctx *c, int n, Geom g, const float *d_cost, const float *d_lab, const float_image *const *input_matches,
                const epic_params_t *params, float *d_flow, sfgpu_epic_stats_t *stats, const Caller &who);
// rgb_to_lab (image.c:694) of the 3 planes of P floats at src into dst on the context's stream (sf_epicflow.cu)
void launch_rgb_to_lab(sfgpu_ctx *c, size_t P, const float *src, float *dst);
} // namespace sf
