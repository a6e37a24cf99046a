// sf_jets.cu -- the jet loop of Slow Flow (slow_flow.cpp:706-1030, deep_matching = 0) over one sequence of integer frames
// on the device: sfgpu_slow_flow_jets.
//
// Pass 1 streams every frame's packed 8-/16-bit samples through a raw ring and reduces them to the block partials of
// normalize() (variational_mt.cpp:17-85) -- straight from the packed samples, or after the pre-scaling of
// slow_flow.cpp:538-542 -- so that the statistics cover all n_frames like the reference's one normalize() call.
// Pass 2 uploads the frames of the requested jets a second time (1-2 bytes per sample: cheaper than keeping fp32 frames
// resident, and device memory stays bounded by the window) and turns each into a normalised level-0 frame of a device
// ring.  Jet j reads frames j*steps .. j*steps + 3*steps: its forward window is the first 2*steps + 1 of them, its
// backward window the last 2*steps + 1 in reverse order (slow_flow.cpp:865-911, 1018-1030).  Each window runs the
// window core of sfgpu_variational_mt (sf_mt.cu) on ring pointers; its flow, multiplied by steps, and its occlusion
// labels go to download planes that the D2H stream drains while the next window computes.
//
// Copies go through CopyPipeline (sf_hostcopy.cu).  Pass 2's stage k = jet first_jet + k: its new frames go up right
// after stage k - 1 has converted its own, so they cross PCIe while jet k - 1 solves.
#include <string.h>

#include <cmath>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "sf_context.cuh"

namespace sf {

struct NormCoef {
    double avg[3], sd[3];
};

// k_unpack_frame (sf_sequence.cu) followed by k_norm_apply (sf_mt.cu) in one pass, with their arithmetic: the exact
// integer -> float conversion, then (float)((v - avg) / std) in double for a channel with std > 0.  The stride padding
// is zeroed.
template <typename T>
__global__ void __launch_bounds__(256) k_unpack_normalize(Geom g, const unsigned char *__restrict__ raw, size_t step, int channels,
                                                          NormCoef n, float *__restrict__ dst) {
    const int i = blockIdx.x * 32 + threadIdx.x, j = blockIdx.y * 8 + threadIdx.y;
    if (i >= g.S || j >= g.H) return;
    float v[3] = {0.f, 0.f, 0.f};
    if (i < g.W) {
        const T *row = reinterpret_cast<const T *>(raw + (size_t)j * step);
#pragma unroll
        for (int c = 0; c < 3; c++) {
            v[c] = (float)row[channels == 1 ? i : 3 * i + c];
            if (n.sd[c] > 0) v[c] = (float)(((double)v[c] - n.avg[c]) / n.sd[c]);
        }
    }
    const size_t P = g.plane(), o = (size_t)j * g.S + i;
    dst[o] = v[0];
    dst[o + P] = v[1];
    dst[o + 2 * P] = v[2];
}

// the outputs of one window: flow x steps in fp32 (slow_flow.cpp:907-911, 1026-1030), occlusion labels copied (occ may be
// null), whole planes
__global__ void __launch_bounds__(256) k_jet_out(size_t P, const float *__restrict__ wx, const float *__restrict__ wy,
                                                 const float *__restrict__ occ, float steps, float *__restrict__ ox,
                                                 float *__restrict__ oy, float *__restrict__ oocc) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    ox[i] = wx[i] * steps;
    oy[i] = wy[i] * steps;
    if (occ) oocc[i] = occ[i];
}

static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct JetOutputs {
    image_t *const *fwd_x, *const *fwd_y, *const *back_x, *const *back_y, *const *occ;
};

// The arguments have been checked.  gf: the frames' geometry, g: the (pre-scaled) geometry of the windows and outputs.
static int run_jets(sfgpu_ctx *c, int n_frames, const sf_frame_int_t *frames, int bits, float scale, Geom gf, Geom g, int first_jet,
                    int n_jets, sf_mt_params_t *params, bool backward_one_direction, const color_image_t *channel_w,
                    const JetOutputs &out) {
    cudaStream_t st = c->stream;
    const int steps = params->S - 1, F = 2 * steps + 1, R = 3 * steps + 1; // R: frames of one jet
    const bool scaled = scale != 1.0f;
    const size_t P = g.plane(), Pf = gf.plane();
    const int nblk = norm_blocks(g);
    size_t raw_slot = 0;
    for (int f = 0; f < n_frames; f++) raw_slot = std::max(raw_slot, frames[f].step * (size_t)frames[f].height);
    // io area, in floats, every region a multiple of 64 floats (256 bytes):
    //   raw ring (R slots of packed frames) | frame ring (R normalised frames) | download planes of two jets (fwd x, y, occ,
    //   back x, y) | channel weights | pre-scaling scratch (unpacked, blur tmp, blurred: 3 x 3 planes of gf) | pass-1 partials
    auto up64 = [](size_t n) { return (n + 63) & ~(size_t)63; };
    const size_t raw_floats = up64((raw_slot + 3) / 4);
    const size_t n_raw = R * raw_floats, n_ring = up64(R * 3 * P), n_out = up64(2 * 5 * P), n_chw = channel_w ? up64(3 * P) : 0,
                 n_scratch = scaled ? up64(9 * Pf) : 0, n_sums = up64((size_t)n_frames * nblk * 6 * 2);
    int rc = c->ensure_io(n_raw + n_ring + n_out + n_chw + n_scratch + n_sums);
    if (rc != SFGPU_OK) return rc;
    unsigned char *raw = reinterpret_cast<unsigned char *>(c->io);
    float *ring = c->io + n_raw, *outp = ring + n_ring, *chw = outp + n_out, *scratch = chw + n_chw;
    double *sums = reinterpret_cast<double *>(scratch + n_scratch);
    auto raw_of = [&](int f) { return raw + (size_t)(f % R) * raw_floats * 4; };
    auto ring_of = [&](int f) { return ring + (size_t)(f % R) * 3 * P; };
    auto raw_copy = [&](int f) { return HostCopy{raw_of(f), const_cast<void *>(frames[f].data), frames[f].step * (size_t)frames[f].height}; };
    // frame f as a window frame of g: normalised (nc != null, in the ring) or only pre-scaled (nc == null, into dst)
    auto convert = [&](int f, const NormCoef *nc, float *dst) {
        const sf_frame_int_t &q = frames[f];
        if (!scaled) { // only with nc: pass 1 reads the packed samples directly
            const dim3 grid((g.S + 31) / 32, (g.H + 7) / 8);
            if (bits == 8)
                k_unpack_normalize<unsigned char><<<grid, dim3(32, 8), 0, st>>>(g, raw_of(f), q.step, q.channels, *nc, dst);
            else
                k_unpack_normalize<unsigned short><<<grid, dim3(32, 8), 0, st>>>(g, raw_of(f), q.step, q.channels, *nc, dst);
            c->prof_acc.kernel_launches++;
            return;
        }
        launch_unpack_frame(st, gf, raw_of(f), q.step, q.channels, bits, scratch);
        launch_prescale(st, gf, scratch, scratch + 3 * Pf, scratch + 6 * Pf, g, dst, scale);
        c->prof_acc.kernel_launches += 4;
        if (nc) {
            launch_norm_apply(st, g, dst, nc->avg, nc->sd);
            c->prof_acc.kernel_launches++;
        }
    };

    // ---- pass 1: block partials of every frame; stage f = frame f in raw slot f % R, last read by frame f - R (R >= 4)
    const double t_call = now_ms();
    std::vector<const void *> buffers;
    for (int f = 0; f < n_frames; f++) buffers.push_back(frames[f].data);
    CopyPipeline pipe(c);
    int status = pipe.start(buffers);
    if (status == SFGPU_OK) status = pipe.upload(0, {raw_copy(0)});
    for (int f = 0; f < n_frames && status == SFGPU_OK; f++) {
        if ((status = pipe.wait(f)) != SFGPU_OK) break;
        double *part = sums + (size_t)f * nblk * 6;
        if (scaled) {
            convert(f, nullptr, ring);
            launch_norm_sums(st, g, ring, part);
        } else {
            launch_norm_sums_packed(st, g, raw_of(f), frames[f].step, frames[f].channels, bits, part);
        }
        c->prof_acc.kernel_launches++;
        if ((status = pipe.pass(f)) != SFGPU_OK) break;
        if (f + 1 < n_frames) status = pipe.upload(f + 1, {raw_copy(f + 1)}, f - 3);
    }
    status = pipe.finish(status);
    if (status != SFGPU_OK) return status;
    SF_CUDA(cudaGetLastError());
    std::vector<double> hs((size_t)n_frames * nblk * 6);
    SF_CUDA(cudaMemcpyAsync(hs.data(), sums, hs.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    SF_CUDA(cudaStreamSynchronize(st));
    NormCoef nc;
    norm_statistics(hs.data(), n_frames, g, nc.avg, nc.sd);
    norm_publish(nc.avg, nc.sd, params); // the windows read the published values (dpsis weight)
    c->mt_stats.setup_ms = now_ms() - t_call;

    // ---- pass 2: stage k = jet first_jet + k.  Stage 0 uploads its 3*steps + 1 frames (and the channel weights), stage
    // k > 0 the steps frames jet k - 1 did not read; their raw slots were last read by stage k - 1's conversions.
    const int f0 = first_jet * steps;
    auto first_new = [&](int k) { return k == 0 ? f0 : f0 + k * steps + 2 * steps + 1; };
    auto upload = [&](int k) {
        std::vector<HostCopy> up;
        for (int f = first_new(k); f <= f0 + k * steps + 3 * steps; f++) up.push_back(raw_copy(f));
        if (k == 0 && channel_w) up.push_back({chw, channel_w->c1, 3 * P * sizeof(float)});
        return pipe.upload(k, up, k - 1);
    };
    buffers.clear();
    for (int f = f0; f <= f0 + (n_jets - 1) * steps + 3 * steps; f++) buffers.push_back(frames[f].data);
    for (int k = 0; k < n_jets; k++) {
        for (image_t *const *a : {out.fwd_x, out.fwd_y, out.back_x, out.back_y}) buffers.push_back(a[k]->data);
        if (out.occ) buffers.push_back(out.occ[k]->data);
    }
    if (channel_w) buffers.push_back(channel_w->c1);
    // one window on ring frames fr[0 .. F-1]; the outputs of level 0 go to ox, oy (x steps) and oocc (nullable)
    auto window = [&](const float *const *fr, const sf_mt_params_t *p, bool one_direction, const float *wchw, float *ox, float *oy,
                      float *oocc) -> int {
        MtWindow w;
        int r = mt_window_layout(c, p, g, false, false, w);
        if (r != SFGPU_OK) return r;
        if (w.levels == 0) { // the reference computes nothing: the zero initial flow stays, no labels are made
            launch_fill(st, ox, P, 0.0f);
            launch_fill(st, oy, P, 0.0f);
            if (oocc) launch_fill(st, oocc, P, 0.0f);
            return SFGPU_OK;
        }
        for (int f = 0; f < F; f++) w.frames[0][f] = const_cast<float *>(fr[f]);
        w.chw = wchw;
        SF_CUDA(cudaMemsetAsync(w.wx, 0, P * sizeof(float), st));
        SF_CUDA(cudaMemsetAsync(w.wy, 0, P * sizeof(float), st));
        if ((r = mt_window_build(c, w)) != SFGPU_OK) return r;
        float avg_change[2];
        if ((r = mt_window_solve(c, p, one_direction, w, avg_change)) != SFGPU_OK) return r;
        k_jet_out<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(P, w.wx, w.wy, oocc ? w.occ : nullptr, (float)steps, ox, oy, oocc);
        c->prof_acc.kernel_launches++;
        SF_CUDA(cudaGetLastError());
        return SFGPU_OK;
    };

    status = pipe.start(buffers);
    if (status == SFGPU_OK) status = upload(0);
    for (int k = 0; k < n_jets && status == SFGPU_OK; k++) {
        const int j0 = f0 + k * steps; // first frame of the jet
        // the download planes of this parity were last drained by stage k - 2
        if ((status = pipe.wait(k, k - 2)) != SFGPU_OK) break;
        for (int f = first_new(k); f <= j0 + 3 * steps; f++) convert(f, &nc, ring_of(f));
        if ((status = pipe.pass(k)) != SFGPU_OK) break;
        if (k + 1 < n_jets && (status = upload(k + 1)) != SFGPU_OK) break;
        float *o = outp + (size_t)(k & 1) * 5 * P;
        const float *fwd[2 * SF_MT_MAX_REF + 1], *bwd[2 * SF_MT_MAX_REF + 1];
        for (int f = 0; f < F; f++) {
            fwd[f] = ring_of(j0 + f);
            bwd[f] = ring_of(j0 + 3 * steps - f);
        }
        if ((status = window(fwd, params, params->one_direction != 0, channel_w ? chw : nullptr, o, o + P, out.occ ? o + 2 * P : nullptr)) != SFGPU_OK)
            break;
        if ((status = pipe.pass(k)) != SFGPU_OK) break;
        std::vector<HostCopy> down = {{o, out.fwd_x[k]->data, P * sizeof(float)}, {o + P, out.fwd_y[k]->data, P * sizeof(float)}};
        if (out.occ) down.push_back({o + 2 * P, out.occ[k]->data, P * sizeof(float)});
        if ((status = pipe.download(k, down)) != SFGPU_OK) break;
        // the backward window: no channel weights (Q10), one direction if asked
        if ((status = window(bwd, params, params->one_direction != 0 || backward_one_direction, nullptr, o + 3 * P, o + 4 * P, nullptr)) != SFGPU_OK)
            break;
        if ((status = pipe.pass(k)) != SFGPU_OK) break;
        status = pipe.download(k, {{o + 3 * P, out.back_x[k]->data, P * sizeof(float)}, {o + 4 * P, out.back_y[k]->data, P * sizeof(float)}});
    }
    status = pipe.finish(status);
    c->mt_stats.total_ms = now_ms() - t_call;
    return status;
}

} // namespace sf

using namespace sf;

extern "C" {

int sfgpu_slow_flow_jets(sfgpu_ctx *c, int n_frames, const sf_frame_int_t *frames, int bits, float scale, int first_jet, int n_jets,
                         sf_mt_params_t *params, int backward_one_direction, const color_image_t *channel_w, image_t *const *fwd_x,
                         image_t *const *fwd_y, image_t *const *back_x, image_t *const *back_y, image_t *const *occlusions) {
    const std::string at = "sfgpu_slow_flow_jets: ";
    if (!c || !frames || !params || !fwd_x || !fwd_y || !back_x || !back_y || (bits != 8 && bits != 16) || first_jet < 0 || n_jets < 1 ||
        !(scale > 0.0f) || !std::isfinite(scale)) {
        set_error(at + "bad argument (non-null context, frames, params and output arrays; bits 8 or 16; first_jet >= 0; n_jets >= 1; "
                       "scale > 0)");
        return SFGPU_ERR_ARG;
    }
    const int steps = params->S - 1;
    if (steps < 1 || steps > SF_MT_MAX_REF) {
        set_error(at + "slow_flow_S out of range");
        return SFGPU_ERR_ARG;
    }
    if (params->smoothing < 0 || params->smoothing > 1) {
        set_error(at + "slow_flow_smoothing >= 2 is not supported (reference bug, SURVEY Q6)");
        return SFGPU_ERR_UNSUPPORTED;
    }
    if (params->layers < 1 || (params->layers > 1 && !(params->p_scale > 0.f && params->p_scale < 1.f))) {
        set_error(at + "bad pyramid parameters");
        return SFGPU_ERR_ARG;
    }
    const long long need = 1 + ((long long)first_jet + n_jets + 2) * steps;
    if (n_frames < need) {
        set_error(at + "n_frames = " + std::to_string(n_frames) + ", jets " + std::to_string(first_jet) + " .. " +
                  std::to_string((long long)first_jet + n_jets - 1) + " read frames up to " + std::to_string(need - 1));
        return SFGPU_ERR_ARG;
    }
    if (frames[0].width < 1 || frames[0].height < 1) {
        set_error(at + "frames[0]: width and height must be >= 1");
        return SFGPU_ERR_ARG;
    }
    const Geom gf = make_geom(frames[0].width, frames[0].height);
    for (int f = 0; f < n_frames; f++)
        if (!arg_frame_int(at, "frames[" + std::to_string(f) + "]", frames[f], gf, bits)) return SFGPU_ERR_ARG;
    Geom g = gf;
    if (scale != 1.0f) {
        int w = 0, h = 0;
        if (sfgpu_prescale_size(gf.W, gf.H, scale, &w, &h) != SFGPU_OK) {
            set_error(at + "the frames scaled by " + std::to_string(scale) + " are empty");
            return SFGPU_ERR_ARG;
        }
        g = make_geom(w, h);
    }
    if (channel_w && !arg_is(at, "channel_w", channel_w, g)) return SFGPU_ERR_ARG;
    const Caller who{"sfgpu_slow_flow_jets", "jet", first_jet};
    for (int k = 0; k < n_jets; k++)
        if (!arg_is(who.at(k), "fwd_x", fwd_x[k], g) || !arg_is(who.at(k), "fwd_y", fwd_y[k], g) || !arg_is(who.at(k), "back_x", back_x[k], g) ||
            !arg_is(who.at(k), "back_y", back_y[k], g) || (occlusions && !arg_is(who.at(k), "occlusions", occlusions[k], g)))
            return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    memset(&c->mt_stats, 0, sizeof(c->mt_stats));
    return run_jets(c, n_frames, frames, bits, scale, gf, g, first_jet, n_jets, params, backward_one_direction != 0, channel_w,
                    JetOutputs{fwd_x, fwd_y, back_x, back_y, occlusions});
}

} // extern "C"
