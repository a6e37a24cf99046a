// sf_context.cu -- context management, the two-frame driver and the C ABI of include/slowflow_gpu.h
// (two-frame, sequence, operator twins, profiling).  The multi-frame driver lives in sf_mt.cu.
#include <utility>

#include "sf_context.cuh"

#include <stdlib.h>
#include <string.h>

namespace sf {

static thread_local std::string g_last_error;
void set_error(const std::string &msg) { g_last_error = msg; }
bool cuda_ok(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return true;
    g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return false;
}

Penalty make_penalty(int type, float eps, float trunc) {
    Penalty p;
    p.type = type;
    const float e2 = eps * eps; // the reference squares in float, then widens (modified_l1_norm.h:15)
    p.eps_sq_f = e2;
    p.eps_sq_d = (double)e2;
    p.trunc = trunc;
    return p;
}

// the 5-tap derivative filter of the two-frame path (image.c:425)
static bool at_least_5x5(const std::string &at, Geom g) {
    if (g.W >= 5 && g.H >= 5) return true;
    set_error(at + "image must be at least 5x5 (5-tap derivative filter, image.c:425)");
    return false;
}

} // namespace sf

using namespace sf;

// ------------------------------------------------------------------------------------------ context
enum { PROF_SOR = 0, PROF_DATA = 1, PROF_CUT = 2 };

int sfgpu_ctx::ensure_workspace(Geom geom) {
    if (!at_least_5x5("", geom)) return SFGPU_ERR_ARG;
    const size_t P = geom.plane();
    const size_t need = (size_t)(SP_COUNT + 3 + 1 + 2 + 1) * P;
    if (need > ws_floats) {
        if (ws) cudaFree(ws);
        ws = nullptr;
        ws_floats = 0;
        SF_CUDA(cudaMalloc(&ws, need * sizeof(float)));
        ws_floats = need;
        g = Geom{0, 0, 0};
    }
    if (geom.W != g.W || geom.H != g.H || geom.S != g.S) {
        g = geom;
        float *p = ws;
        float *arena = p; p += (size_t)SP_COUNT * P;
        wim = p;   p += 3 * P;
        mask = p;  p += P;
        uu = p;    p += P;
        vv = p;    p += P;
        dpsis = p; p += P;
        if (!sor_plan_init(sor, g, arena, num_sms)) {
            // no TMA descriptor: only the per-half-sweep variant can run; report it loudly
            return SFGPU_ERR_CUDA;
        }
    }
    return SFGPU_OK;
}

int sfgpu_ctx::ensure_io(size_t floats) {
    seq_last_slot = -1; // every user of the io area overwrites the frame ring a sequence call may have left there
    if (floats <= io_floats) return SFGPU_OK;
    if (io) cudaFree(io);
    io = nullptr;
    io_floats = 0;
    SF_CUDA(cudaMalloc(&io, floats * sizeof(float)));
    io_floats = floats;
    return SFGPU_OK;
}

cudaEvent_t sfgpu_ctx::get_event() {
    if (!ev_free.empty()) {
        cudaEvent_t e = ev_free.back();
        ev_free.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
void sfgpu_ctx::prof_begin(int kind, cudaEvent_t &a) {
    a = nullptr;
    if (!prof) return;
    a = get_event();
    cudaEventRecord(a, stream);
}
void sfgpu_ctx::prof_end(int kind, cudaEvent_t a) {
    if (!prof || !a) return;
    cudaEvent_t b = get_event();
    cudaEventRecord(b, stream);
    ev_pending.push_back(EvPair{a, b, kind});
}
int sfgpu_ctx::prof_collect() {
    SF_CUDA(cudaStreamSynchronize(stream));
    for (auto &p : ev_pending) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            if (p.kind == PROF_SOR) prof_acc.sor_ms += ms;
            else if (p.kind == PROF_CUT) prof_acc.graphcut_ms += ms;
            else prof_acc.data_ms += ms;
        }
        ev_free.push_back(p.a);
        ev_free.push_back(p.b);
    }
    ev_pending.clear();
    return SFGPU_OK;
}

static int auto_fuse(const sfgpu_ctx *c) { return c->sor_fuse > 0 ? c->sor_fuse : 4; }

// ------------------------------------------------------------------------------------------ two-frame driver
namespace sf {

// shared by the two-frame and multi-frame drivers: one sor_coupled call on the context's arena
int run_sor(sfgpu_ctx *c, int iterations, float omega, int *cur, bool zero_init) {
    cudaEvent_t ev;
    c->prof_begin(PROF_SOR, ev);
    const int n = launch_sor(c->stream, c->sor, iterations, omega, c->sor_variant, auto_fuse(c), cur, zero_init);
    c->prof_end(PROF_SOR, ev);
    if (n < 0) return SFGPU_ERR_CUDA;
    c->prof_acc.sor_launches += n;
    c->prof_acc.kernel_launches += n;
    c->prof_acc.sor_calls += 1;
    c->prof_acc.sor_pixel_sweeps += (long long)c->g.W * c->g.H * iterations;
    return SFGPU_OK;
}

int run_two_frame(sfgpu_ctx *c, Geom g, float *d_wx, float *d_wy, const float *d_im1, const float *d_im2,
                  const variational_params_t *params) {
    variational_params_t defaults;
    if (!params) {
        variational_params_default(&defaults);
        params = &defaults;
    }
    int rc = c->ensure_workspace(g);
    if (rc != SFGPU_OK) return rc;
    cudaStream_t st = c->stream;
    const size_t P = g.plane();
    float *A = c->sor.arena;
    // variational.c:114-116
    const float half_alpha = 0.5f * params->alpha;
    const float half_gamma_over3 = params->gamma * 0.5f / 3.0f;
    const float half_delta_over3 = params->delta * 0.5f / 3.0f;
    const float avg0[3] = {0.f, 0.f, 0.f}, std1[3] = {1.f, 1.f, 1.f};
    Penalty two_frame_reg;
    two_frame_reg.type = -1; two_frame_reg.eps_sq_f = 0.f; two_frame_reg.eps_sq_d = 0.0; two_frame_reg.trunc = 0.f;

    launch_dpsis_weight(st, g, d_im1, c->dpsis, 5.0f, avg0, std1, 255.0f); // variational.c:34
    c->prof_acc.kernel_launches++;

    // 0: marching data pass (k_prep_fused / k_prep_two_frame), 1: separate warp kernel + tile-based data-term kernel,
    // 2: as 0 but the default loop keeps the smoothness pass separate (k_flow_smooth + k_prep_two_frame); 1 and 2 are the
    // A/B references of the tests and benchmarks
    const bool fused_prep = c->data_variant == 0 || c->data_variant == 2;
    if (fused_prep && params->niter_inner == 1 && params->niter_solver > 0) {
        // Default shape of the loop (one inner iteration): per outer iteration the flow update of the previous
        // iteration (variational.c:60-69 collapsed to w += du) and the smoothness pass are folded into the data pass,
        // so an outer iteration is {update+smoothness+warp+derivatives+data term+Laplacian+block inverse, SOR launches}.
        // The flow ping-pongs between the caller's planes and (uu, vv); the last update lands in the caller's.
        const bool fused_psi = c->data_variant == 0;
        float *fx = d_wx, *fy = d_wy, *ax = c->uu, *ay = c->vv;
        const float *pdu = nullptr, *pdv = nullptr;
        for (int outer = 0; outer < params->niter_outer; outer++) {
            cudaEvent_t ev;
            if (fused_psi) {
                c->prof_begin(PROF_DATA, ev);
                launch_prep_fused(st, g, c->num_sms, d_im1, d_im2, fx, fy, pdu, pdv, c->dpsis, half_alpha, half_delta_over3,
                                  half_gamma_over3, ax, ay, A + SP_PH * P, A + SP_PV * P, A + SP_A11 * P, A + SP_A12 * P,
                                  A + SP_A22 * P, A + SP_B1 * P, A + SP_B2 * P);
                c->prof_end(PROF_DATA, ev);
                if (outer > 0) {
                    std::swap(fx, ax);
                    std::swap(fy, ay);
                }
                c->prof_acc.kernel_launches += 1;
            } else {
                if (outer == 0) {
                    launch_smoothness(st, g, fx, fy, c->dpsis, half_alpha, two_frame_reg, 1, A + SP_PH * P, A + SP_PV * P);
                } else {
                    launch_update_smoothness(st, g, fx, fy, pdu, pdv, c->dpsis, half_alpha, two_frame_reg, 1, ax, ay,
                                             A + SP_PH * P, A + SP_PV * P);
                    std::swap(fx, ax);
                    std::swap(fy, ay);
                }
                c->prof_begin(PROF_DATA, ev);
                launch_prep_two_frame(st, g, c->num_sms, d_im1, d_im2, fx, fy, nullptr, nullptr, A + SP_PH * P, A + SP_PV * P,
                                      half_delta_over3, half_gamma_over3, A + SP_A11 * P, A + SP_A12 * P, A + SP_A22 * P,
                                      A + SP_B1 * P, A + SP_B2 * P);
                c->prof_end(PROF_DATA, ev);
                c->prof_acc.kernel_launches += 2;
            }
            c->prof_acc.data_launches++;
            c->prof_acc.data_pixels += (long long)g.W * g.H;
            int cur = 0;
            rc = run_sor(c, params->niter_solver, params->sor_omega, &cur, true); // variational.c:57
            if (rc != SFGPU_OK) return rc;
            pdu = A + (size_t)(cur ? SP_DUB : SP_DUA) * P;
            pdv = A + (size_t)(cur ? SP_DVB : SP_DVA) * P;
        }
        if (pdu) {
            launch_add(st, g, d_wx, fx, pdu);
            launch_add(st, g, d_wy, fy, pdv);
            c->prof_acc.kernel_launches += 2;
        }
        SF_CUDA(cudaGetLastError());
        return SFGPU_OK;
    }
    for (int outer = 0; outer < params->niter_outer; outer++) {
        if (!fused_prep) {
            launch_warp(st, g, d_im2, d_wx, d_wy, 1, c->wim, c->mask); // variational.c:40
            c->prof_acc.kernel_launches++;
        }
        int cur = 0;
        for (int inner = 0; inner < params->niter_inner; inner++) {
            const bool first = (inner == 0), last = (inner == params->niter_inner - 1);
            const float *uu = first ? d_wx : c->uu, *vv = first ? d_wy : c->vv;
            launch_smoothness(st, g, uu, vv, c->dpsis, half_alpha, two_frame_reg, 1, A + SP_PH * P, A + SP_PV * P);
            const float *du = first ? nullptr : A + (size_t)(cur ? SP_DUB : SP_DUA) * P;
            const float *dv = first ? nullptr : A + (size_t)(cur ? SP_DVB : SP_DVA) * P;
            cudaEvent_t ev;
            c->prof_begin(PROF_DATA, ev);
            // variational.c:53-55 + the block inverse of solver.c:101-106, one pass
            DataTermDesc term{d_im1, c->wim, +1, c->mask, DK_TWO_FRAME, half_delta_over3, half_gamma_over3, 1.0f, -1};
            DataCommon cm{};
            cm.du = du; cm.dv = dv; cm.chw = nullptr; cm.occ = nullptr; cm.data_norm = 1.0f; cm.dt_norm = 1;
            cm.pc = two_frame_reg; cm.pg = two_frame_reg; cm.accumulate = false; cm.fuse_system = true;
            cm.ph = A + SP_PH * P; cm.pv = A + SP_PV * P; cm.lap_u = d_wx; cm.lap_v = d_wy;
            cm.a11 = A + SP_A11 * P; cm.a12 = A + SP_A12 * P; cm.a22 = A + SP_A22 * P; cm.b1 = A + SP_B1 * P;
            cm.b2 = A + SP_B2 * P;
            if (fused_prep)
                launch_prep_two_frame(st, g, c->num_sms, d_im1, d_im2, d_wx, d_wy, du, dv, cm.ph, cm.pv, half_delta_over3,
                                      half_gamma_over3, cm.a11, cm.a12, cm.a22, cm.b1, cm.b2);
            else
                launch_data_term(st, g, term, cm);
            c->prof_end(PROF_DATA, ev);
            c->prof_acc.data_launches++;
            c->prof_acc.data_pixels += (long long)g.W * g.H;
            c->prof_acc.kernel_launches += 2;
            rc = run_sor(c, params->niter_solver, params->sor_omega, &cur, first); // variational.c:57
            if (rc != SFGPU_OK) return rc;
            const float *ndu = A + (size_t)(cur ? SP_DUB : SP_DUA) * P, *ndv = A + (size_t)(cur ? SP_DVB : SP_DVA) * P;
            if (last) { // variational.c:60-69 collapsed: wx = wx + du
                launch_add(st, g, d_wx, d_wx, ndu);
                launch_add(st, g, d_wy, d_wy, ndv);
            } else {
                launch_add(st, g, c->uu, d_wx, ndu);
                launch_add(st, g, c->vv, d_wy, ndv);
            }
            c->prof_acc.kernel_launches += 2;
        }
    }
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

// ------------------------------------------------------------------------------------------ argument checks
std::string Caller::at(int k) const {
    if (!item) return std::string(fn) + ": ";
    return std::string(fn) + ": " + item + " " + std::to_string(first + k / per) + (part ? std::string(" ") + part[k % per] : "") + ": ";
}

static float *data_of(const image_t *a) { return a->data; }
static float *data_of(const color_image_t *a) { return a->c1; }
static bool contiguous(const image_t *) { return true; }
static bool contiguous(const color_image_t *a) { // image.c:80-87; the geometry has been checked
    const size_t P = (size_t)a->stride * a->height;
    return a->c2 == a->c1 + P && a->c3 == a->c2 + P;
}
static std::string dims(int w, int h, int s) { return std::to_string(w) + "x" + std::to_string(h) + " stride " + std::to_string(s); }

// sets_g: `a` gives the call's geometry g, else it must have it
template <typename Image>
static bool check_image(const std::string &at, const std::string &name, const Image *a, Geom &g, bool sets_g) {
    std::string what;
    if (!a || !data_of(a))
        what = "null image";
    else if (!sets_g && (a->width != g.W || a->height != g.H || a->stride != g.S))
        what = "different geometry (" + dims(a->width, a->height, a->stride) + "; the images of a call share width/height/stride, here " +
               dims(g.W, g.H, g.S) + ")";
    else if (a->width < 1 || a->height < 1)
        what = "width and height must be >= 1 (" + dims(a->width, a->height, a->stride) + ")";
    else if (a->stride != (((long long)a->width + 3) / 4) * 4)
        what = "stride must be ceil4(width) (image.c:25), not " + dims(a->width, a->height, a->stride);
    else if (!contiguous(a))
        what = "colour images must be planar and contiguous (image.c:80-87)";
    if (!what.empty()) {
        set_error(at + name + ": " + what);
        return false;
    }
    if (sets_g) g = make_geom(a->width, a->height);
    return true;
}

bool arg_geom(const std::string &at, const std::string &name, const image_t *a, Geom &g) { return check_image(at, name, a, g, true); }
bool arg_geom(const std::string &at, const std::string &name, const color_image_t *a, Geom &g) { return check_image(at, name, a, g, true); }
bool arg_is(const std::string &at, const std::string &name, const image_t *a, Geom g) { return check_image(at, name, a, g, false); }
bool arg_is(const std::string &at, const std::string &name, const color_image_t *a, Geom g) { return check_image(at, name, a, g, false); }

bool arg_frame_int(const std::string &at, const std::string &name, const sf_frame_int_t &q, Geom g, int bits) {
    const size_t sample = bits / 8;
    if (!q.data || q.width != g.W || q.height != g.H || (q.channels != 1 && q.channels != 3) ||
        q.step < (size_t)q.width * q.channels * sample || (q.step % sample) != 0) {
        set_error(at + name + ": integer frames must match the call's geometry (" + std::to_string(g.W) + "x" + std::to_string(g.H) +
                  "), have 1 or 3 channels and step >= width*channels*bytes");
        return false;
    }
    return true;
}

} // namespace sf

// ------------------------------------------------------------------------------------------ ABI: basics
extern "C" {

const char *sfgpu_version(void) { return "slowflow_gpu 0.1 (sm_100a)"; }
const char *sfgpu_last_error(void) { return g_last_error.c_str(); }

int sfgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int sfgpu_create(int device, void *stream, sfgpu_ctx **out) {
    if (!out) {
        set_error("sfgpu_create: out is NULL");
        return SFGPU_ERR_ARG;
    }
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        set_error("sfgpu_create: no CUDA device available (this library has no CPU fallback)");
        return SFGPU_ERR_CUDA;
    }
    if (device == -1 && cudaGetDevice(&device) != cudaSuccess) device = 0; // -1: the calling thread's current device
    if (device < 0 || device >= n) {
        set_error("sfgpu_create: device index out of range");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    SF_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("sfgpu_create: device is not sm_100 class (kernels are built for sm_100a only)");
        return SFGPU_ERR_UNSUPPORTED;
    }
    if (!sor_device_init() || !data_term_device_init()) {
        set_error("sfgpu_create: cudaFuncSetAttribute failed (dynamic shared memory opt-in)");
        return SFGPU_ERR_CUDA;
    }
    sfgpu_ctx *c = new sfgpu_ctx();
    c->device = device;
    if (const char *e = getenv("SLOWFLOW_GPU_DATA_VARIANT")) c->data_variant = atoi(e); // A/B switch for benchmarking
    if (const char *e = getenv("SLOWFLOW_GPU_STAGED_COPIES")) c->staged_host_copies = atoi(e) != 0;
    if (const char *e = getenv("SLOWFLOW_GPU_HOST_MINCUT")) c->host_mincut = atoi(e) != 0;
    if (const char *e = getenv("SLOWFLOW_GPU_MT_DATA_VARIANT")) c->mt_data_variant = atoi(e);
    if (const char *e = getenv("SLOWFLOW_GPU_MT_TERMS_SCALAR")) c->mt_terms_scalar = atoi(e) != 0;
    if (const char *e = getenv("SLOWFLOW_GPU_MT_WARP_VARIANT")) c->mt_warp_variant = atoi(e);
    c->num_sms = prop.multiProcessorCount;
    if (stream) {
        c->stream = (cudaStream_t)stream;
        c->own_stream = false;
    } else {
        if (!cuda_ok(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking), "cudaStreamCreate")) {
            delete c;
            return SFGPU_ERR_CUDA;
        }
        c->own_stream = true;
    }
    *out = c;
    return SFGPU_OK;
}

void sfgpu_destroy(sfgpu_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto &p : c->ev_pending) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    for (auto e : c->ev_free) cudaEventDestroy(e);
    if (c->mt_cache_pool) cudaFree(c->mt_cache_pool);
    if ((c->mt_cache_hits || c->mt_cache_misses) && getenv("SLOWFLOW_GPU_TRACE"))
        fprintf(stderr, "multi-frame frame cache: %llu frames found on the device, %llu uploaded\n", c->mt_cache_hits, c->mt_cache_misses);
    if (c->mtw) sf::mt_work_free(c->mtw);
    if (c->stager) sf::host_stager_free(c->stager);
    if (c->cut) sf::device_cut_free(c->cut);
    if (c->epic_arena) sf::epic_arena_free(c->epic_arena);
    if (c->ws) cudaFree(c->ws);
    sf::sor_plan_release(c->sor);
    if (c->io) cudaFree(c->io);
    for (auto &ring : c->copy_ev)
        for (auto e : ring)
            if (e) cudaEventDestroy(e);
    if (c->seq_raw) cudaFree(c->seq_raw);
    if (c->h2d) cudaStreamDestroy(c->h2d);
    if (c->d2h) cudaStreamDestroy(c->d2h);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

int sfgpu_mt_frame_cache(sfgpu_ctx *c, int max_frames) {
    if (!c || max_frames < 0 || max_frames > 64) {
        set_error("sfgpu_mt_frame_cache: bad argument");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(c->device));
    SF_CUDA(cudaStreamSynchronize(c->stream)); // nothing in flight reads a slot that is dropped here
    if ((size_t)max_frames != c->mt_cache.size()) { // another capacity: the pool is re-made at the next call
        if (c->mt_cache_pool) cudaFree(c->mt_cache_pool);
        c->mt_cache_pool = nullptr;
        c->mt_cache_slot_floats = 0;
        c->mt_cache.assign((size_t)max_frames, sfgpu_ctx::MtFrameSlot());
    }
    for (auto &e : c->mt_cache) e.host = nullptr; // enabling (again) starts from an empty cache: the caller may have changed frames
    return SFGPU_OK;
}

int sfgpu_synchronize(sfgpu_ctx *c) {
    if (!c) return SFGPU_ERR_ARG;
    SF_CUDA(cudaStreamSynchronize(c->stream));
    return SFGPU_OK;
}

int sfgpu_set_sor_variant(sfgpu_ctx *c, int variant) {
    if (!c || variant < 0 || variant > 2) return SFGPU_ERR_ARG;
    c->sor_variant = variant;
    return SFGPU_OK;
}
int sfgpu_set_sor_fuse(sfgpu_ctx *c, int n) {
    if (!c || n < 0 || n > 7) return SFGPU_ERR_ARG;
    c->sor_fuse = n;
    return SFGPU_OK;
}

int sfgpu_profile_enable(sfgpu_ctx *c, int on) {
    if (!c) return SFGPU_ERR_ARG;
    c->prof = on != 0;
    return SFGPU_OK;
}
int sfgpu_profile_reset(sfgpu_ctx *c) {
    if (!c) return SFGPU_ERR_ARG;
    int rc = c->prof_collect();
    memset(&c->prof_acc, 0, sizeof(c->prof_acc));
    return rc;
}
int sfgpu_profile_get(sfgpu_ctx *c, sfgpu_profile_t *out) {
    if (!c || !out) return SFGPU_ERR_ARG;
    int rc = c->prof_collect();
    *out = c->prof_acc;
    return rc;
}

int sfgpu_host_register(void *ptr, unsigned long long bytes) {
    SF_CUDA(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable)); // pinned for every device's context
    return SFGPU_OK;
}
int sfgpu_host_unregister(void *ptr) {
    SF_CUDA(cudaHostUnregister(ptr));
    return SFGPU_OK;
}

// ------------------------------------------------------------------------------------------ ABI: two-frame
void variational_params_default(variational_params_t *params) {
    if (!params) {
        fprintf(stderr, "Error optical_flow_params_default: argument is null\n");
        exit(1);
    }
    params->alpha = 1.0f;
    params->gamma = 0.71f;
    params->delta = 0.0f;
    params->sigma = 1.00f;
    params->niter_outer = 5;
    params->niter_inner = 1;
    params->niter_solver = 30;
    params->sor_omega = 1.9f;
}

int sfgpu_variational_dev(sfgpu_ctx *c, float *d_wx, float *d_wy, const float *d_im1, const float *d_im2, int width,
                          int height, int stride, const variational_params_t *params) {
    if (!c || !d_wx || !d_wy || !d_im1 || !d_im2) {
        set_error("sfgpu_variational_dev: null argument");
        return SFGPU_ERR_ARG;
    }
    if (stride != make_geom(width, height).S) {
        set_error("stride must be ceil4(width)");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(c->device));
    return run_two_frame(c, Geom{width, height, stride}, d_wx, d_wy, d_im1, d_im2, params);
}

int sfgpu_variational(sfgpu_ctx *c, image_t *wx, image_t *wy, const color_image_t *im1, const color_image_t *im2,
                      const variational_params_t *params) {
    const char *at = "sfgpu_variational: ";
    Geom g;
    if (!c || !arg_geom(at, "wx", wx, g) || !arg_is(at, "wy", wy, g) || !arg_is(at, "im1", im1, g) || !arg_is(at, "im2", im2, g))
        return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    int rc = c->ensure_io(8 * P);
    if (rc != SFGPU_OK) return rc;
    float *d_im1 = c->io, *d_im2 = c->io + 3 * P, *d_wx = c->io + 6 * P, *d_wy = c->io + 7 * P;
    cudaStream_t st = c->stream;
    // ordinary malloc'ed caller images (image.c:17-33) take the multi-threaded staged path of sf_hostcopy.cu
    rc = host_copies(c, {{d_im1, im1->c1, 3 * P * sizeof(float)}, {d_im2, im2->c1, 3 * P * sizeof(float)},
                         {d_wx, wx->data, P * sizeof(float)}, {d_wy, wy->data, P * sizeof(float)}}, true);
    if (rc != SFGPU_OK) return rc;
    rc = run_two_frame(c, g, d_wx, d_wy, d_im1, d_im2, params);
    if (rc != SFGPU_OK) return rc;
    rc = host_copies(c, {{d_wx, wx->data, P * sizeof(float)}, {d_wy, wy->data, P * sizeof(float)}}, false);
    if (rc != SFGPU_OK) return rc;
    SF_CUDA(cudaStreamSynchronize(st));
    return SFGPU_OK;
}

// legacy drop-in: thread-local default context on the current device, abort on error
void variational(image_t *wx, image_t *wy, const color_image_t *im1, const color_image_t *im2,
                 variational_params_t *params) {
    struct Holder {
        sfgpu_ctx *c = nullptr;
        ~Holder() { if (c) sfgpu_destroy(c); }
    };
    static thread_local Holder holder;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    if (holder.c && holder.c->device != dev) {
        sfgpu_destroy(holder.c);
        holder.c = nullptr;
    }
    if (!holder.c && sfgpu_create(dev, nullptr, &holder.c) != SFGPU_OK) {
        fprintf(stderr, "error in variational(): %s\n", sfgpu_last_error());
        exit(1);
    }
    if (sfgpu_variational(holder.c, wx, wy, im1, im2, params) != SFGPU_OK) {
        fprintf(stderr, "error in variational(): %s\n", sfgpu_last_error());
        exit(1);
    }
}

// ------------------------------------------------------------------------------------------ ABI: operator twins
struct DevPlanes { // scratch device planes for the operator twins
    float *p = nullptr;
    ~DevPlanes() { if (p) cudaFree(p); }
    int alloc(size_t floats) { SF_CUDA(cudaMalloc(&p, floats * sizeof(float))); return SFGPU_OK; }
};
#define H2D(dst, src, n) SF_CUDA(cudaMemcpyAsync((dst), (src), (n) * sizeof(float), cudaMemcpyHostToDevice, st))
#define D2H(dst, src, n) SF_CUDA(cudaMemcpyAsync((dst), (src), (n) * sizeof(float), cudaMemcpyDeviceToHost, st))

int sfgpu_image_warp(sfgpu_ctx *c, color_image_t *dst, image_t *mask, const color_image_t *src, const image_t *wx,
                     const image_t *wy, int factor) {
    const char *at = "sfgpu_image_warp: ";
    Geom g;
    if (!c || !arg_geom(at, "src", src, g) || !arg_is(at, "dst", dst, g) || !arg_is(at, "wx", wx, g) || !arg_is(at, "wy", wy, g) ||
        (mask && !arg_is(at, "mask", mask, g)))
        return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    DevPlanes d;
    int rc = d.alloc(9 * P);
    if (rc) return rc;
    float *s3 = d.p, *fx = d.p + 3 * P, *fy = d.p + 4 * P, *o3 = d.p + 5 * P, *m = d.p + 8 * P;
    H2D(s3, src->c1, 3 * P); H2D(fx, wx->data, P); H2D(fy, wy->data, P);
    launch_warp(st, g, s3, fx, fy, factor, o3, mask ? m : nullptr);
    D2H(dst->c1, o3, 3 * P);
    if (mask) D2H(mask->data, m, P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_warp_frame_derivs(sfgpu_ctx *c, const color_image_t *src, const image_t *wx, const image_t *wy, int factor, int variant,
                            color_image_t *warped, image_t *mask, color_image_t *dx, color_image_t *dy, color_image_t *dxx,
                            color_image_t *dxy, color_image_t *dyy) {
    const char *at = "sfgpu_warp_frame_derivs: ";
    if (!c || variant < 0 || variant > 1) {
        set_error("sfgpu_warp_frame_derivs: bad argument");
        return SFGPU_ERR_ARG;
    }
    Geom g;
    if (!arg_geom(at, "src", src, g) || !arg_is(at, "wx", wx, g) || !arg_is(at, "wy", wy, g) || !arg_is(at, "mask", mask, g))
        return SFGPU_ERR_ARG;
    color_image_t *outs[6] = {warped, dx, dy, dxx, dxy, dyy};
    const char *names[6] = {"warped", "dx", "dy", "dxx", "dxy", "dyy"};
    for (int k = 0; k < 6; k++)
        if (!arg_is(at, names[k], outs[k], g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    DevPlanes d;
    int rc = d.alloc(24 * P);
    if (rc) return rc;
    float *s3 = d.p, *fx = s3 + 3 * P, *fy = fx + P, *o3 = fy + P, *m = o3 + 3 * P, *dv = m + P;
    H2D(s3, src->c1, 3 * P); H2D(fx, wx->data, P); H2D(fy, wy->data, P);
    // NaN pre-fill: every element the kernel leaves untouched shows up in the test
    SF_CUDA(cudaMemsetAsync(o3, 0xff, 19 * P * sizeof(float), st));
    if (variant == 0) {
        launch_warp_derivs(st, g, c->num_sms, s3, fx, fy, factor, o3, m, dv);
    } else {
        launch_warp(st, g, s3, fx, fy, factor, o3, m);
        launch_frame_derivs(st, g, o3, dv);
    }
    D2H(warped->c1, o3, 3 * P);
    D2H(mask->data, m, P);
    for (int k = 0; k < 5; k++) D2H(outs[k + 1]->c1, dv + (size_t)k * 3 * P, 3 * P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

extern "C++" { // Image: image_t (planes = 1) or color_image_t (planes = 3)
template <typename Image>
static int convolve_planes(sfgpu_ctx *c, Image *dst, const Image *src, int planes, int horder, const float *hc, int vorder,
                           const float *vc, const char *what) {
    const std::string at = std::string(what) + ": ";
    Geom g;
    if (!arg_geom(at, "src", src, g) || !arg_is(at, "dst", dst, g)) return SFGPU_ERR_ARG;
    if (!c || (!hc && !vc) || (hc && (horder < 1 || horder > 2)) || (vc && (vorder < 1 || vorder > 2))) {
        set_error(at + "bad argument (order 1 = 3 taps, 2 = 5 taps)");
        return SFGPU_ERR_ARG;
    }
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane(), n = (size_t)planes * P;
    int rc = c->ensure_io(3 * n);
    if (rc != SFGPU_OK) return rc;
    cudaStream_t st = c->stream;
    float *d_src = c->io, *d_tmp = c->io + n, *d_dst = c->io + 2 * n;
    SF_CUDA(cudaMemcpyAsync(d_src, data_of(src), n * sizeof(float), cudaMemcpyHostToDevice, st));
    if (hc && vc) { // image.c:665-680: horizontal into a temporary, then vertical
        launch_convolve(st, g, d_src, d_tmp, false, horder, hc, planes);
        launch_convolve(st, g, d_tmp, d_dst, true, vorder, vc, planes);
        c->prof_acc.kernel_launches += 2;
    } else {
        launch_convolve(st, g, d_src, d_dst, vc != nullptr, hc ? horder : vorder, hc ? hc : vc, planes);
        c->prof_acc.kernel_launches++;
    }
    SF_CUDA(cudaMemcpyAsync(data_of(dst), d_dst, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    return SFGPU_OK;
}
} // extern "C++"

int sfgpu_convolve_horiz(sfgpu_ctx *c, image_t *dst, const image_t *src, int order, const float *coeffs) {
    return convolve_planes(c, dst, src, 1, order, coeffs, 0, nullptr, "sfgpu_convolve_horiz");
}
int sfgpu_convolve_vert(sfgpu_ctx *c, image_t *dst, const image_t *src, int order, const float *coeffs) {
    return convolve_planes(c, dst, src, 1, 0, nullptr, order, coeffs, "sfgpu_convolve_vert");
}
int sfgpu_color_image_convolve_hv(sfgpu_ctx *c, color_image_t *dst, const color_image_t *src, int horiz_order, const float *horiz_coeffs,
                                  int vert_order, const float *vert_coeffs) {
    return convolve_planes(c, dst, src, 3, horiz_order, horiz_coeffs, vert_order, vert_coeffs, "sfgpu_color_image_convolve_hv");
}

// get_derivatives (variational_aux.c:55-78) with the 5-tap derivative filter of variational.c:118-119
int sfgpu_get_derivatives(sfgpu_ctx *c, const color_image_t *im1, const color_image_t *im2, color_image_t *dx, color_image_t *dy,
                          color_image_t *dt, color_image_t *dxx, color_image_t *dxy, color_image_t *dyy, color_image_t *dxt,
                          color_image_t *dyt) {
    const char *at = "sfgpu_get_derivatives: ";
    Geom g;
    if (!c) { set_error("sfgpu_get_derivatives: null argument"); return SFGPU_ERR_ARG; }
    if (!arg_geom(at, "im1", im1, g) || !arg_is(at, "im2", im2, g)) return SFGPU_ERR_ARG;
    color_image_t *outs[8] = {dx, dy, dt, dxx, dxy, dyy, dxt, dyt};
    const char *names[8] = {"dx", "dy", "dt", "dxx", "dxy", "dyy", "dxt", "dyt"};
    for (int k = 0; k < 8; k++)
        if (!arg_is(at, names[k], outs[k], g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t n = 3 * g.plane();
    int rc = c->ensure_io(11 * n);
    if (rc != SFGPU_OK) return rc;
    cudaStream_t st = c->stream;
    float *d1 = c->io, *d2 = d1 + n, *mean = d2 + n, *o[8];
    for (int k = 0; k < 8; k++) o[k] = mean + (size_t)(k + 1) * n;
    const float c5[5] = {1.0f / 12.0f, -8.0f / 12.0f, -0.0f, 8.0f / 12.0f, -(1.0f / 12.0f)};
    SF_CUDA(cudaMemcpyAsync(d1, im1->c1, n * sizeof(float), cudaMemcpyHostToDevice, st));
    SF_CUDA(cudaMemcpyAsync(d2, im2->c1, n * sizeof(float), cudaMemcpyHostToDevice, st));
    launch_mean_diff(st, n, d1, d2, mean, o[2]);
    launch_convolve(st, g, mean, o[0], false, 2, c5, 3); // dx
    launch_convolve(st, g, mean, o[1], true, 2, c5, 3);  // dy
    launch_convolve(st, g, o[0], o[3], false, 2, c5, 3); // dxx
    launch_convolve(st, g, o[0], o[4], true, 2, c5, 3);  // dxy
    launch_convolve(st, g, o[1], o[5], true, 2, c5, 3);  // dyy
    launch_convolve(st, g, o[2], o[6], false, 2, c5, 3); // dxt
    launch_convolve(st, g, o[2], o[7], true, 2, c5, 3);  // dyt
    c->prof_acc.kernel_launches += 8;
    for (int k = 0; k < 8; k++) SF_CUDA(cudaMemcpyAsync(outs[k]->c1, o[k], n * sizeof(float), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    return SFGPU_OK;
}

int sfgpu_compute_dpsis_weight(sfgpu_ctx *c, image_t *dst, const color_image_t *im, float coef, const float *avg3,
                               const float *std3, int hbit) {
    const char *at = "sfgpu_compute_dpsis_weight: ";
    Geom g;
    if (!c || !arg_geom(at, "im", im, g) || !arg_is(at, "dst", dst, g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    DevPlanes d;
    int rc = d.alloc(4 * P);
    if (rc) return rc;
    const float a0[3] = {0.f, 0.f, 0.f}, s1[3] = {1.f, 1.f, 1.f};
    H2D(d.p, im->c1, 3 * P);
    launch_dpsis_weight(st, g, d.p, d.p + 3 * P, coef, avg3 ? avg3 : a0, std3 ? std3 : s1, hbit ? 65535.0f : 255.0f);
    D2H(dst->data, d.p + 3 * P, P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_compute_smoothness(sfgpu_ctx *c, image_t *dst_horiz, image_t *dst_vert, const image_t *uu, const image_t *vv,
                             const image_t *w, float alpha_factor, int robust_reg, float reg_eps, float reg_trunc,
                             int mode) {
    const char *at = "sfgpu_compute_smoothness: ";
    Geom g;
    if (!c || !arg_geom(at, "uu", uu, g) || !arg_is(at, "vv", vv, g) || !arg_is(at, "dpsis_weight", w, g) ||
        !arg_is(at, "dst_horiz", dst_horiz, g) || !arg_is(at, "dst_vert", dst_vert, g))
        return SFGPU_ERR_ARG;
    if (mode < 0 || mode > 1) {
        set_error("smoothing modes >= 2 are not supported (reference bug Q6)");
        return SFGPU_ERR_UNSUPPORTED;
    }
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    DevPlanes d;
    int rc = d.alloc(5 * P);
    if (rc) return rc;
    H2D(d.p, uu->data, P); H2D(d.p + P, vv->data, P); H2D(d.p + 2 * P, w->data, P);
    Penalty reg = make_penalty(robust_reg, reg_eps, reg_trunc);
    launch_smoothness(st, g, d.p, d.p + P, d.p + 2 * P, alpha_factor, reg, mode, d.p + 3 * P, d.p + 4 * P);
    D2H(dst_horiz->data, d.p + 3 * P, P); D2H(dst_vert->data, d.p + 4 * P, P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_compute_data_and_match(sfgpu_ctx *c, image_t *a11, image_t *a12, image_t *a22, image_t *b1, image_t *b2,
                                 const image_t *mask, const image_t *du, const image_t *dv, const color_image_t *im1,
                                 const color_image_t *im2w, float half_delta_over3, float half_gamma_over3) {
    const char *at = "sfgpu_compute_data_and_match: ";
    Geom g;
    if (!c || !arg_geom(at, "im1", im1, g) || !arg_is(at, "im2w", im2w, g) || !arg_is(at, "mask", mask, g) || !arg_is(at, "du", du, g) ||
        !arg_is(at, "dv", dv, g) || !arg_is(at, "a11", a11, g) || !arg_is(at, "a12", a12, g) || !arg_is(at, "a22", a22, g) ||
        !arg_is(at, "b1", b1, g) || !arg_is(at, "b2", b2, g) || !at_least_5x5(at, g))
        return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    DevPlanes d;
    int rc = d.alloc(14 * P);
    if (rc) return rc;
    float *i1 = d.p, *i2 = d.p + 3 * P, *m = d.p + 6 * P, *u = d.p + 7 * P, *v = d.p + 8 * P, *o = d.p + 9 * P;
    H2D(i1, im1->c1, 3 * P); H2D(i2, im2w->c1, 3 * P); H2D(m, mask->data, P); H2D(u, du->data, P); H2D(v, dv->data, P);
    DataTermDesc term{i1, i2, +1, m, DK_TWO_FRAME, half_delta_over3, half_gamma_over3, 1.0f, -1};
    DataCommon cm{};
    cm.du = u; cm.dv = v; cm.data_norm = 1.0f; cm.dt_norm = 1; cm.pc = make_penalty(1, 0.001f, 0.5f); cm.pg = cm.pc;
    cm.accumulate = false; cm.fuse_system = false;
    cm.a11 = o; cm.a12 = o + P; cm.a22 = o + 2 * P; cm.b1 = o + 3 * P; cm.b2 = o + 4 * P;
    launch_data_term(st, g, term, cm);
    D2H(a11->data, o, P); D2H(a12->data, o + P, P); D2H(a22->data, o + 2 * P, P); D2H(b1->data, o + 3 * P, P);
    D2H(b2->data, o + 4 * P, P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_prep_two_frame(sfgpu_ctx *c, image_t *a11, image_t *a12, image_t *a22, image_t *b1, image_t *b2, const color_image_t *im1,
                         const color_image_t *im2, const image_t *wx, const image_t *wy, const image_t *du, const image_t *dv,
                         const image_t *ph, const image_t *pv, float half_delta_over3, float half_gamma_over3) {
    const char *at = "sfgpu_prep_two_frame: ";
    Geom g;
    if (!c || (du == nullptr) != (dv == nullptr)) {
        set_error("sfgpu_prep_two_frame: null argument");
        return SFGPU_ERR_ARG;
    }
    if (!arg_geom(at, "wx", wx, g) || !arg_is(at, "wy", wy, g) || !arg_is(at, "im1", im1, g) || !arg_is(at, "im2", im2, g) ||
        (du && (!arg_is(at, "du", du, g) || !arg_is(at, "dv", dv, g))) || !arg_is(at, "dpsis_horiz", ph, g) ||
        !arg_is(at, "dpsis_vert", pv, g) || !arg_is(at, "a11", a11, g) || !arg_is(at, "a12", a12, g) || !arg_is(at, "a22", a22, g) ||
        !arg_is(at, "b1", b1, g) || !arg_is(at, "b2", b2, g) || !at_least_5x5(at, g))
        return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    DevPlanes d;
    int rc = d.alloc(17 * P);
    if (rc) return rc;
    float *i1 = d.p, *i2 = d.p + 3 * P, *fx = d.p + 6 * P, *fy = d.p + 7 * P, *u = d.p + 8 * P, *v = d.p + 9 * P,
          *dh = d.p + 10 * P, *dvv = d.p + 11 * P, *o = d.p + 12 * P;
    H2D(i1, im1->c1, 3 * P); H2D(i2, im2->c1, 3 * P); H2D(fx, wx->data, P); H2D(fy, wy->data, P);
    H2D(dh, ph->data, P); H2D(dvv, pv->data, P);
    if (du) { H2D(u, du->data, P); H2D(v, dv->data, P); }
    SF_CUDA(cudaMemsetAsync(o, 0xff, 5 * P * sizeof(float), st)); // NaN pattern: every element must be written by the kernel
    launch_prep_two_frame(st, g, c->num_sms, i1, i2, fx, fy, du ? u : nullptr, du ? v : nullptr, dh, dvv, half_delta_over3,
                          half_gamma_over3, o, o + P, o + 2 * P, o + 3 * P, o + 4 * P);
    c->prof_acc.kernel_launches++;
    D2H(a11->data, o, P); D2H(a12->data, o + P, P); D2H(a22->data, o + 2 * P, P); D2H(b1->data, o + 3 * P, P);
    D2H(b2->data, o + 4 * P, P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_sub_laplacian(sfgpu_ctx *c, image_t *dst, const image_t *src, const image_t *wh, const image_t *wv) {
    const char *at = "sfgpu_sub_laplacian: ";
    Geom g;
    if (!c || !arg_geom(at, "src", src, g) || !arg_is(at, "dst", dst, g) || !arg_is(at, "weight_horiz", wh, g) ||
        !arg_is(at, "weight_vert", wv, g))
        return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    DevPlanes d;
    int rc = d.alloc(4 * P);
    if (rc) return rc;
    H2D(d.p, dst->data, P); H2D(d.p + P, src->data, P); H2D(d.p + 2 * P, wh->data, P); H2D(d.p + 3 * P, wv->data, P);
    launch_sub_laplacian(st, g, d.p, d.p + P, d.p + 2 * P, d.p + 3 * P);
    D2H(dst->data, d.p, P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

int sfgpu_sor_coupled(sfgpu_ctx *c, image_t *du, image_t *dv, image_t *a11, image_t *a12, image_t *a22,
                      const image_t *b1, const image_t *b2, const image_t *ph, const image_t *pv, int iterations,
                      float omega) {
    const char *at = "sfgpu_sor_coupled: ";
    Geom g;
    if (!c || !arg_geom(at, "du", du, g) || !arg_is(at, "dv", dv, g) || !arg_is(at, "a11", a11, g) || !arg_is(at, "a12", a12, g) ||
        !arg_is(at, "a22", a22, g) || !arg_is(at, "b1", b1, g) || !arg_is(at, "b2", b2, g) || !arg_is(at, "dpsis_horiz", ph, g) ||
        !arg_is(at, "dpsis_vert", pv, g))
        return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    int rc = c->ensure_workspace(g);
    if (rc != SFGPU_OK) return rc;
    const size_t P = g.plane();
    cudaStream_t st = c->stream;
    float *A = c->sor.arena;
    H2D(A + SP_A11 * P, a11->data, P); H2D(A + SP_A12 * P, a12->data, P); H2D(A + SP_A22 * P, a22->data, P);
    H2D(A + SP_B1 * P, b1->data, P); H2D(A + SP_B2 * P, b2->data, P); H2D(A + SP_PH * P, ph->data, P);
    H2D(A + SP_PV * P, pv->data, P); H2D(A + SP_DUA * P, du->data, P); H2D(A + SP_DVA * P, dv->data, P);
    launch_invert_blocks(st, g, A + SP_A11 * P, A + SP_A12 * P, A + SP_A22 * P, A + SP_PH * P, A + SP_PV * P);
    int cur = 0;
    rc = run_sor(c, iterations, omega, &cur, false);
    if (rc != SFGPU_OK) return rc;
    D2H(du->data, A + (size_t)(cur ? SP_DUB : SP_DUA) * P, P);
    D2H(dv->data, A + (size_t)(cur ? SP_DVB : SP_DVA) * P, P);
    D2H(a11->data, A + SP_A11 * P, P); D2H(a12->data, A + SP_A12 * P, P); D2H(a22->data, A + SP_A22 * P, P);
    SF_CUDA(cudaStreamSynchronize(st));
    SF_CUDA(cudaGetLastError());
    return SFGPU_OK;
}

} // extern "C"
