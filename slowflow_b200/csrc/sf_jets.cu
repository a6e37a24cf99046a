// sf_jets.cu -- the jet loop of Slow Flow (slow_flow.cpp:706-1030) over one sequence of integer frames on the device:
// sfgpu_slow_flow_jets (deep_matching = 0: every window starts from a zero flow) and sfgpu_slow_flow_jets_epic (every
// window starts from an EPIC interpolation of the caller's matches, slow_flow.cpp:801-843, 979).
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
// With EPIC, pass 2 runs in chunks of JET_CHUNK jets.  Per chunk, on the one compute stream: the conversions of its new
// frames, the Lab planes of its reference frames (saliency filter on), one EPIC batch over its 2 x JET_CHUNK windows into
// a flow buffer of the chunk, then every jet's two windows from that flow x 1 / steps.  EPIC never runs beside a window.
//
// Copies go through CopyPipeline (sf_hostcopy.cu).  Pass 2's stage k = jet first_jet + k, and a chunk's uploads are those
// of its first jet's stage: its new frames (and edge maps) go up right after the chunk before it has converted its own
// (and made its EPIC batch), so they cross PCIe while that chunk's windows solve.
#include <string.h>

#include <cmath>

#include <algorithm>
#include <chrono>
#include <set>
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

// One pointwise pass over whole planes: ox, oy = wx, wy * factor in fp32, occlusion labels copied (occ may be null).  It
// scales a window's flow by steps into its outputs (slow_flow.cpp:907-911, 1026-1030) and an EPIC flow by 1 / steps into
// a window's initial flow (SURVEY §3.2).  ox, oy may be wx, wy (no __restrict__): each thread reads its element first.
__global__ void __launch_bounds__(256) k_jet_out(size_t P, const float *wx, const float *wy, const float *occ, float factor, float *ox,
                                                 float *oy, float *oocc) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    ox[i] = wx[i] * factor;
    oy[i] = wy[i] * factor;
    if (occ) oocc[i] = occ[i];
}

static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct JetOutputs {
    image_t *const *fwd_x, *const *fwd_y, *const *back_x, *const *back_y, *const *occ;
};

// The initial flows of sfgpu_slow_flow_jets_epic: per jet the matches of its two windows, the edge maps of reference
// frames 0 .. n_jets (euc not yet added), EPIC's parameters, and 2 stats per jet (nullable).
struct JetEpic {
    const float_image *const *fwd_matches, *const *back_matches;
    float_image *const *edges;
    const epic_params_t *params;
    sfgpu_epic_stats_t *stats;
};

// Jets per chunk of pass 2 with EPIC initial flows: 2 x 4 = 8 EPIC items, the N at which the batch was measured
// (profiles/r3_epic_batch.md).  Without EPIC a chunk is one jet.
constexpr int JET_CHUNK = 4;

// The arguments have been checked.  gf: the frames' geometry, g: the (pre-scaled) geometry of the windows and outputs.
// epic == null: every window starts from a zero flow.
static int run_jets(sfgpu_ctx *c, int n_frames, const sf_frame_int_t *frames, int bits, float scale, Geom gf, Geom g, int first_jet,
                    int n_jets, sf_mt_params_t *params, bool backward_one_direction, const color_image_t *channel_w,
                    const JetOutputs &out, const JetEpic *epic) {
    cudaStream_t st = c->stream;
    const int C = epic ? JET_CHUNK : 1;
    const int steps = params->S - 1, F = 2 * steps + 1, R = C * steps + 2 * steps + 1; // R: frames of one chunk
    const bool scaled = scale != 1.0f, sal = epic && epic->params->saliency_th != 0;
    const size_t P = g.plane(), Pf = gf.plane(), N = (size_t)g.W * g.H;
    const int nblk = norm_blocks(g);
    size_t raw_slot = 0;
    for (int f = 0; f < n_frames; f++) raw_slot = std::max(raw_slot, frames[f].step * (size_t)frames[f].height);
    // io area, in floats, every region a multiple of 64 floats (256 bytes):
    //   raw ring (R slots of packed frames) | frame ring (R normalised frames) | download planes of two jets (fwd x, y, occ,
    //   back x, y) | channel weights | pre-scaling scratch (unpacked, blur tmp, blurred: 3 x 3 planes of gf) | pass-1 partials
    //   | with EPIC: edge maps of C + 1 reference frames | per EPIC item (2 C of them): edge costs, Lab planes (saliency
    //   filter on), flow x and y
    auto up64 = [](size_t n) { return (n + 63) & ~(size_t)63; };
    const size_t raw_floats = up64((raw_slot + 3) / 4);
    const size_t n_raw = R * raw_floats, n_ring = up64(R * 3 * P), n_out = up64(2 * 5 * P), n_chw = channel_w ? up64(3 * P) : 0,
                 n_scratch = scaled ? up64(9 * Pf) : 0, n_sums = up64((size_t)n_frames * nblk * 6 * 2);
    const size_t n_edge = epic ? up64((C + 1) * N) : 0, n_cost = epic ? up64(2 * C * N) : 0, n_lab = sal ? up64(2 * C * 3 * P) : 0,
                 n_flow = epic ? up64(2 * C * 2 * P) : 0;
    int rc = c->ensure_io(n_raw + n_ring + n_out + n_chw + n_scratch + n_sums + n_edge + n_cost + n_lab + n_flow);
    if (rc != SFGPU_OK) return rc;
    unsigned char *raw = reinterpret_cast<unsigned char *>(c->io);
    float *ring = c->io + n_raw, *outp = ring + n_ring, *chw = outp + n_out, *scratch = chw + n_chw;
    double *sums = reinterpret_cast<double *>(scratch + n_scratch);
    float *edge0 = scratch + n_scratch + n_sums, *costs = edge0 + n_edge, *lab = costs + n_cost, *flows = lab + n_lab;
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

    // ---- pass 2 in chunks of C jets: stage k = jet first_jet + k, and chunk q's uploads are stage q * C's.  Chunk 0 uploads
    // its frames (and the channel weights), a later chunk the frames the chunk before it did not read; their raw slots were
    // last read by that chunk's conversions.  With EPIC, reference frame i = (first_jet + i) * steps + steps (i = 0 ..
    // n_jets) has its edge map in slot i % (C + 1); a chunk uploads those of its reference frames the chunk before it did
    // not have, into slots that chunk last read before its EPIC batch.
    const int f0 = first_jet * steps, n_chunks = (n_jets + C - 1) / C;
    auto count = [&](int q) { return std::min(C, n_jets - q * C); };
    auto last_frame = [&](int q) { return f0 + (q * C + count(q) - 1) * steps + 3 * steps; };
    auto first_new = [&](int q) { return q == 0 ? f0 : last_frame(q - 1) + 1; };
    auto edge_of = [&](int i) { return edge0 + (size_t)(i % (C + 1)) * N; };
    auto upload = [&](int q) {
        const int k0 = q * C, m = count(q);
        std::vector<HostCopy> up;
        for (int f = first_new(q); f <= last_frame(q); f++) up.push_back(raw_copy(f));
        if (q == 0 && channel_w) up.push_back({chw, channel_w->c1, 3 * P * sizeof(float)});
        if (epic) {
            const int i0 = q == 0 ? 0 : k0 + 1;
            epic_add_euc(k0 + m + 1 - i0, epic->edges + i0, epic->params->euc); // epic.cpp:155-163, once per edge map
            for (int i = i0; i <= k0 + m; i++) up.push_back({edge_of(i), epic->edges[i]->pixels, N * sizeof(float)});
        }
        return pipe.upload(k0, up, k0 - C);
    };
    buffers.clear();
    for (int f = f0; f <= f0 + (n_jets - 1) * steps + 3 * steps; f++) buffers.push_back(frames[f].data);
    for (int k = 0; k < n_jets; k++) {
        for (image_t *const *a : {out.fwd_x, out.fwd_y, out.back_x, out.back_y}) buffers.push_back(a[k]->data);
        if (out.occ) buffers.push_back(out.occ[k]->data);
    }
    if (channel_w) buffers.push_back(channel_w->c1);
    if (epic)
        for (int i = 0; i <= n_jets; i++) buffers.push_back(epic->edges[i]->pixels);
    // chunk q's EPIC batch into `flows`: item 2 i is the forward window of jet q C + i, item 2 i + 1 its backward window.
    // Reference frame q C + i feeds items 2 i - 1 and 2 i (those that exist); the items' edge costs and Lab planes are
    // device copies of its edge map and of one Lab conversion of its normalised frame.
    auto chunk_epic = [&](int q) -> int {
        const int k0 = q * C, m = count(q);
        for (int i = 0; i <= m; i++) {
            const int a = i > 0 ? 2 * i - 1 : 0, b = i < m ? 2 * i : 2 * m - 1;
            SF_CUDA(cudaMemcpyAsync(costs + a * N, edge_of(k0 + i), N * sizeof(float), cudaMemcpyDeviceToDevice, st));
            if (b != a) SF_CUDA(cudaMemcpyAsync(costs + b * N, edge_of(k0 + i), N * sizeof(float), cudaMemcpyDeviceToDevice, st));
            if (sal) {
                launch_rgb_to_lab(c, P, ring_of(f0 + (k0 + i) * steps + steps), lab + a * 3 * P);
                if (b != a) SF_CUDA(cudaMemcpyAsync(lab + b * 3 * P, lab + a * 3 * P, 3 * P * sizeof(float), cudaMemcpyDeviceToDevice, st));
            }
        }
        std::vector<const float_image *> matches;
        for (int i = 0; i < m; i++) matches.insert(matches.end(), {epic->fwd_matches[k0 + i], epic->back_matches[k0 + i]});
        std::vector<sfgpu_epic_stats_t> es((size_t)2 * m);
        static const char *const direction[2] = {"forward", "backward"};
        const int r = epic_device(c, 2 * m, g, costs, sal ? lab : nullptr, matches.data(), epic->params, flows, es.data(),
                                  Caller{"sfgpu_slow_flow_jets_epic", "jet", first_jet + k0, 2, direction});
        if (r == SFGPU_OK && epic->stats) std::copy(es.begin(), es.end(), epic->stats + 2 * k0);
        return r;
    };
    // one window on ring frames fr[0 .. F-1] from the initial flow init x 1 / steps (null: zero); the outputs of level 0 go
    // to ox, oy (x steps) and oocc (nullable)
    const unsigned plane_blocks = (unsigned)((P + 255) / 256);
    auto window = [&](const float *const *fr, const sf_mt_params_t *p, bool one_direction, const float *wchw, const float *init, float *ox,
                      float *oy, float *oocc) -> int {
        MtWindow w;
        int r = mt_window_layout(c, p, g, false, false, w);
        if (r != SFGPU_OK) return r;
        if (w.levels == 0) { // the reference computes nothing: the initial flow stays, no labels are made
            if (init) { // (the second pass in place)
                k_jet_out<<<plane_blocks, 256, 0, st>>>(P, init, init + P, nullptr, 1.0f / steps, ox, oy, nullptr);
                k_jet_out<<<plane_blocks, 256, 0, st>>>(P, ox, oy, nullptr, (float)steps, ox, oy, nullptr);
                c->prof_acc.kernel_launches += 2;
            } else {
                launch_fill(st, ox, P, 0.0f);
                launch_fill(st, oy, P, 0.0f);
            }
            if (oocc) launch_fill(st, oocc, P, 0.0f);
            return SFGPU_OK;
        }
        for (int f = 0; f < F; f++) w.frames[0][f] = const_cast<float *>(fr[f]);
        w.chw = wchw;
        if (init) {
            k_jet_out<<<plane_blocks, 256, 0, st>>>(P, init, init + P, nullptr, 1.0f / steps, w.wx, w.wy, nullptr);
            c->prof_acc.kernel_launches++;
        } else {
            SF_CUDA(cudaMemsetAsync(w.wx, 0, P * sizeof(float), st));
            SF_CUDA(cudaMemsetAsync(w.wy, 0, P * sizeof(float), st));
        }
        if ((r = mt_window_build(c, w)) != SFGPU_OK) return r;
        float avg_change[2];
        if ((r = mt_window_solve(c, p, one_direction, w, avg_change)) != SFGPU_OK) return r;
        k_jet_out<<<plane_blocks, 256, 0, st>>>(P, w.wx, w.wy, oocc ? w.occ : nullptr, (float)steps, ox, oy, oocc);
        c->prof_acc.kernel_launches++;
        SF_CUDA(cudaGetLastError());
        return SFGPU_OK;
    };

    status = pipe.start(buffers);
    if (status == SFGPU_OK) status = upload(0);
    for (int q = 0; q < n_chunks && status == SFGPU_OK; q++) {
        const int k0 = q * C;
        // the download planes of jet k's parity were last drained by stage k - 2
        if ((status = pipe.wait(k0, k0 - 2)) != SFGPU_OK) break;
        for (int f = first_new(q); f <= last_frame(q); f++) convert(f, &nc, ring_of(f));
        if (epic && (status = chunk_epic(q)) != SFGPU_OK) break;
        if ((status = pipe.pass(k0)) != SFGPU_OK) break;
        if (q + 1 < n_chunks && (status = upload(q + 1)) != SFGPU_OK) break;
        for (int k = k0; k < k0 + count(q); k++) {
            const int j0 = f0 + k * steps; // first frame of the jet
            if (k > k0 && (status = pipe.wait(-1, k - 2)) != SFGPU_OK) break;
            float *o = outp + (size_t)(k & 1) * 5 * P;
            const float *init = epic ? flows + (size_t)(k - k0) * 4 * P : nullptr; // the jet's forward item, then its backward one
            const float *fwd[2 * SF_MT_MAX_REF + 1], *bwd[2 * SF_MT_MAX_REF + 1];
            for (int f = 0; f < F; f++) {
                fwd[f] = ring_of(j0 + f);
                bwd[f] = ring_of(j0 + 3 * steps - f);
            }
            if ((status = window(fwd, params, params->one_direction != 0, channel_w ? chw : nullptr, init, o, o + P,
                                 out.occ ? o + 2 * P : nullptr)) != SFGPU_OK)
                break;
            if ((status = pipe.pass(k)) != SFGPU_OK) break;
            std::vector<HostCopy> down = {{o, out.fwd_x[k]->data, P * sizeof(float)}, {o + P, out.fwd_y[k]->data, P * sizeof(float)}};
            if (out.occ) down.push_back({o + 2 * P, out.occ[k]->data, P * sizeof(float)});
            if ((status = pipe.download(k, down)) != SFGPU_OK) break;
            // the backward window: no channel weights (Q10), one direction if asked
            if ((status = window(bwd, params, params->one_direction != 0 || backward_one_direction, nullptr, init ? init + 2 * P : nullptr,
                                 o + 3 * P, o + 4 * P, nullptr)) != SFGPU_OK)
                break;
            if ((status = pipe.pass(k)) != SFGPU_OK) break;
            if ((status = pipe.download(k, {{o + 3 * P, out.back_x[k]->data, P * sizeof(float)}, {o + 4 * P, out.back_y[k]->data, P * sizeof(float)}})) != SFGPU_OK)
                break;
        }
    }
    status = pipe.finish(status);
    c->mt_stats.total_ms = now_ms() - t_call;
    return status;
}

// The argument checks of sfgpu_slow_flow_jets, also run by sfgpu_slow_flow_jets_epic (fn: the entry's name).  gf: the
// frames' geometry, g: that of the windows and outputs.
static int check_jets(const char *fn, sfgpu_ctx *c, int n_frames, const sf_frame_int_t *frames, int bits, float scale, int first_jet,
                      int n_jets, const sf_mt_params_t *params, const color_image_t *channel_w, const JetOutputs &out, Geom &gf, Geom &g) {
    const std::string at = std::string(fn) + ": ";
    if (!c || !frames || !params || !out.fwd_x || !out.fwd_y || !out.back_x || !out.back_y || (bits != 8 && bits != 16) || first_jet < 0 ||
        n_jets < 1 || !(scale > 0.0f) || !std::isfinite(scale)) {
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
    gf = make_geom(frames[0].width, frames[0].height);
    for (int f = 0; f < n_frames; f++)
        if (!arg_frame_int(at, "frames[" + std::to_string(f) + "]", frames[f], gf, bits)) return SFGPU_ERR_ARG;
    g = gf;
    if (scale != 1.0f) {
        int w = 0, h = 0;
        if (sfgpu_prescale_size(gf.W, gf.H, scale, &w, &h) != SFGPU_OK) {
            set_error(at + "the frames scaled by " + std::to_string(scale) + " are empty");
            return SFGPU_ERR_ARG;
        }
        g = make_geom(w, h);
    }
    if (channel_w && !arg_is(at, "channel_w", channel_w, g)) return SFGPU_ERR_ARG;
    const Caller who{fn, "jet", first_jet};
    for (int k = 0; k < n_jets; k++)
        if (!arg_is(who.at(k), "fwd_x", out.fwd_x[k], g) || !arg_is(who.at(k), "fwd_y", out.fwd_y[k], g) ||
            !arg_is(who.at(k), "back_x", out.back_x[k], g) || !arg_is(who.at(k), "back_y", out.back_y[k], g) ||
            (out.occ && !arg_is(who.at(k), "occlusions", out.occ[k], g)))
            return SFGPU_ERR_ARG;
    return SFGPU_OK;
}

// The checks epic_check_args makes, on the matches of every window and the n_jets + 1 edge maps (window geometry g), and
// that the edge maps are distinct arrays (euc is added to each once)
static int check_jets_epic(const char *fn, int first_jet, int n_jets, Geom g, const JetEpic &e) {
    const std::string at = std::string(fn) + ": ";
    const Caller who{fn, "jet", first_jet};
    for (int k = 0; k < n_jets; k++)
        for (int back = 0; back < 2; back++) {
            const float_image *m = (back ? e.back_matches : e.fwd_matches)[k];
            const std::string name = back ? "back_matches" : "fwd_matches";
            if (!m || !m->pixels) {
                set_error(who.at(k) + name + ": null argument");
                return SFGPU_ERR_ARG;
            }
            if (m->tx < 4) {
                set_error(who.at(k) + name + ": need >= 4 columns (x1 y1 x2 y2)");
                return SFGPU_ERR_ARG;
            }
        }
    std::set<const float *> seen;
    for (int i = 0; i <= n_jets; i++) {
        const float_image *x = e.edges[i];
        const std::string name = at + "edges[" + std::to_string(i) + "]: ";
        if (!x || !x->pixels) {
            set_error(name + "null argument");
            return SFGPU_ERR_ARG;
        }
        if (x->tx != g.W || x->ty != g.H) {
            set_error(name + "must have the window's width x height (" + std::to_string(g.W) + "x" + std::to_string(g.H) + ")");
            return SFGPU_ERR_ARG;
        }
        if (!seen.insert(x->pixels).second) {
            set_error(name + "shares its array with an earlier edge map (euc is added to each once)");
            return SFGPU_ERR_ARG;
        }
    }
    if (strcmp(e.params->method, "LA") != 0 && strcmp(e.params->method, "NW") != 0) {
        set_error(at + "method " + std::string(e.params->method, strnlen(e.params->method, sizeof(e.params->method))) + " not recognized");
        return SFGPU_ERR_ARG;
    }
    return SFGPU_OK;
}

} // namespace sf

using namespace sf;

extern "C" {

int sfgpu_slow_flow_jets(sfgpu_ctx *c, int n_frames, const sf_frame_int_t *frames, int bits, float scale, int first_jet, int n_jets,
                         sf_mt_params_t *params, int backward_one_direction, const color_image_t *channel_w, image_t *const *fwd_x,
                         image_t *const *fwd_y, image_t *const *back_x, image_t *const *back_y, image_t *const *occlusions) {
    const JetOutputs out{fwd_x, fwd_y, back_x, back_y, occlusions};
    Geom gf, g;
    const int rc = check_jets("sfgpu_slow_flow_jets", c, n_frames, frames, bits, scale, first_jet, n_jets, params, channel_w, out, gf, g);
    if (rc != SFGPU_OK) return rc;
    SF_CUDA(cudaSetDevice(c->device));
    memset(&c->mt_stats, 0, sizeof(c->mt_stats));
    return run_jets(c, n_frames, frames, bits, scale, gf, g, first_jet, n_jets, params, backward_one_direction != 0, channel_w, out, nullptr);
}

int sfgpu_slow_flow_jets_epic(sfgpu_ctx *c, int n_frames, const sf_frame_int_t *frames, int bits, float scale, int first_jet, int n_jets,
                              sf_mt_params_t *params, int backward_one_direction, const color_image_t *channel_w,
                              const float_image *const *fwd_matches, const float_image *const *back_matches, float_image *const *edges,
                              const epic_params_t *epic_params, image_t *const *fwd_x, image_t *const *fwd_y, image_t *const *back_x,
                              image_t *const *back_y, image_t *const *occlusions, sfgpu_epic_stats_t *epic_stats) {
    const char *fn = "sfgpu_slow_flow_jets_epic";
    const JetOutputs out{fwd_x, fwd_y, back_x, back_y, occlusions};
    Geom gf, g;
    int rc = check_jets(fn, c, n_frames, frames, bits, scale, first_jet, n_jets, params, channel_w, out, gf, g);
    if (rc != SFGPU_OK) return rc;
    if (!fwd_matches || !back_matches || !edges || !epic_params) {
        set_error(std::string(fn) + ": bad argument (non-null match arrays, edge array and epic_params)");
        return SFGPU_ERR_ARG;
    }
    const JetEpic epic{fwd_matches, back_matches, edges, epic_params, epic_stats};
    if ((rc = check_jets_epic(fn, first_jet, n_jets, g, epic)) != SFGPU_OK) return rc;
    SF_CUDA(cudaSetDevice(c->device));
    memset(&c->mt_stats, 0, sizeof(c->mt_stats));
    return run_jets(c, n_frames, frames, bits, scale, gf, g, first_jet, n_jets, params, backward_one_direction != 0, channel_w, out, &epic);
}

} // extern "C"
