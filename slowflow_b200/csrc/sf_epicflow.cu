// sf_epicflow.cu -- the EpicFlow two-step on the device: rgb_to_lab (image.c:694), then epic() (epic.cpp:147), then
// variational() (variational.c:101), as epicflow.cpp:124-129 and adaptiveFR.cpp:568-574 run them.
//   sfgpu_rgb_to_lab          operator twin of rgb_to_lab (k_rgb_to_lab)
//   sfgpu_epicflow_sequence   the two-step over consecutive pairs of one geometry: each frame is uploaded once for both
//                             steps, the Lab planes are made and read on the device, and the interpolated flows stay
//                             resident until they are refined.
#include <algorithm>
#include <string>
#include <vector>

#include "sf_context.cuh"

namespace sf {

// rgb_to_lab of EpicFlow's image.c, operation for operation with C's float / double promotions (the reference is built
// with -msse4: no FMA, so every product and sum here is an explicitly rounded intrinsic that nvcc cannot contract).
// Pointwise over the P = stride * height floats of a plane, padding columns included, like the reference's loop.
__global__ void __launch_bounds__(256) k_rgb_to_lab(size_t P, const float *__restrict__ src, float *__restrict__ dst) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const float T = 0.008856f, color_attenuation = 1.5f;
    const double r = __fdiv_rn(src[i], 255.f), g = __fdiv_rn(src[i + P], 255.f), b = __fdiv_rn(src[i + 2 * P], 255.f);
    float X = __double2float_rn(__dadd_rn(__dadd_rn(__dmul_rn(0.412453, r), __dmul_rn(0.357580, g)), __dmul_rn(0.180423, b)));
    const float Y = __double2float_rn(__dadd_rn(__dadd_rn(__dmul_rn(0.212671, r), __dmul_rn(0.715160, g)), __dmul_rn(0.072169, b)));
    float Z = __double2float_rn(__dadd_rn(__dadd_rn(__dmul_rn(0.019334, r), __dmul_rn(0.119193, g)), __dmul_rn(0.950227, b)));
    X = __double2float_rn(__ddiv_rn((double)X, 0.950456));
    Z = __double2float_rn(__ddiv_rn((double)Z, 1.088754));
    const float Y3 = __double2float_rn(pow((double)Y, 1. / 3));
    const float fX = __double2float_rn(X > T ? pow((double)X, 1. / 3) : __dadd_rn(__dmul_rn(7.787, (double)X), 16 / 116.));
    const float fY = Y > T ? Y3 : __double2float_rn(__dadd_rn(__dmul_rn(7.787, (double)Y), 16 / 116.));
    const float fZ = __double2float_rn(Z > T ? pow((double)Z, 1. / 3) : __dadd_rn(__dmul_rn(7.787, (double)Z), 16 / 116.));
    const float L = __double2float_rn(Y > T ? __dsub_rn((double)__fmul_rn(116.f, Y3), 16.0) : __dmul_rn(903.3, (double)Y));
    const float A = __fmul_rn(500.f, __fsub_rn(fX, fY)), B = __fmul_rn(200.f, __fsub_rn(fY, fZ));
    // correct_lab = exp(-color_attenuation * pow2(pow2(L/100) - 0.6)): the inner square in float, the outer in double
    const float l = __fdiv_rn(L, 100.f);
    const double q = __dsub_rn((double)__fmul_rn(l, l), 0.6);
    const float corr = __double2float_rn(exp(__dmul_rn((double)-color_attenuation, __dmul_rn(q, q))));
    dst[i] = L;
    dst[i + P] = __fmul_rn(A, corr);
    dst[i + 2 * P] = __fmul_rn(B, corr);
}

void launch_rgb_to_lab(sfgpu_ctx *c, size_t P, const float *src, float *dst) {
    k_rgb_to_lab<<<(unsigned)((P + 255) / 256), 256, 0, c->stream>>>(P, src, dst);
    c->prof_acc.kernel_launches++;
}

// Pairs per EPIC batch: the N at which the batch was measured (profiles/r3_epic_batch.md); EPIC's workspace takes about
// 100 B per pixel per item, so a chunk of 2560x1440 pairs needs about 3 GB whatever n_pairs is.
constexpr int EF_CHUNK = 8;

// The argument checks have passed.  Pair j of chunk q = j / EF_CHUNK.  Per chunk, on the one compute stream: the Lab planes
// of its first frames, the EPIC batch into the chunk's flow buffer, then run_two_frame on each pair in place.  The copies
// go through CopyPipeline (sf_hostcopy.cu), one stage per chunk: with page-locked caller memory the next chunk's frames
// and edge costs go up while this chunk's pairs are refined, and each refined pair goes down while the next one computes.
// Device layout (the context's io area):
//   frame ring: 2 * EF_CHUNK + 2 frames, frame f in slot f % R, so the frames of two consecutive chunks never share a slot
//   Lab planes of one chunk | flows of two chunks (by chunk parity) | edge costs of two chunks (by chunk parity)
static int run_epicflow(sfgpu_ctx *c, int n_pairs, Geom g, const color_image_t *const *frames, const float_image *const *matches,
                        float_image *const *edges, const epic_params_t *ep, const variational_params_t *vp, image_t *const *wx,
                        image_t *const *wy, sfgpu_epic_stats_t *stats) {
    const size_t P = g.plane(), N = (size_t)g.W * g.H;
    const int CH = EF_CHUNK, R = 2 * CH + 2, n_chunks = (n_pairs + CH - 1) / CH;
    const bool sal = ep->saliency_th != 0;
    int rc = c->ensure_io((size_t)R * 3 * P + (size_t)CH * 3 * P + 2 * (size_t)CH * 2 * P + 2 * (size_t)CH * N); // (also ends a _u8/_u16 sequence)
    if (rc != SFGPU_OK) return rc;
    float *ring = c->io, *lab = ring + (size_t)R * 3 * P, *flow0 = lab + (size_t)CH * 3 * P, *cost0 = flow0 + 2 * (size_t)CH * 2 * P;
    auto frame = [&](int f) { return ring + (size_t)(f % R) * 3 * P; };
    auto flows = [&](int q) { return flow0 + (size_t)(q & 1) * CH * 2 * P; };
    auto costs = [&](int q) { return cost0 + (size_t)(q & 1) * CH * N; };
    auto count = [&](int q) { return std::min(CH, n_pairs - q * CH); };

    CopyPipeline pipe(c); // stage q = chunk q
    // chunk q's inputs: its frames (frame q * CH is already resident for q > 0) and its edge costs after += euc.  The frame
    // slots and the cost parity it fills were last read by chunk q - 2.
    auto upload = [&](int q) -> int {
        const int j0 = q * CH, m = count(q);
        epic_add_euc(m, edges + j0, ep->euc);
        std::vector<HostCopy> up;
        for (int f = q == 0 ? 0 : j0 + 1; f <= j0 + m; f++) up.push_back({frame(f), frames[f]->c1, 3 * P * sizeof(float)});
        for (int k = 0; k < m; k++) up.push_back({costs(q) + k * N, edges[j0 + k]->pixels, N * sizeof(float)});
        return pipe.upload(q, up, q - 2);
    };

    std::vector<const void *> buffers;
    for (int f = 0; f <= n_pairs; f++) buffers.push_back(frames[f]->c1);
    for (int j = 0; j < n_pairs; j++) buffers.insert(buffers.end(), {wx[j]->data, wy[j]->data, edges[j]->pixels});
    int status = pipe.start(buffers);
    if (status == SFGPU_OK) status = upload(0);
    std::vector<sfgpu_epic_stats_t> st((size_t)CH);
    for (int q = 0; q < n_chunks && status == SFGPU_OK; q++) {
        const int j0 = q * CH, m = count(q);
        // the flow buffer of this parity was last drained by chunk q - 2's downloads
        if ((status = pipe.wait(q, q - 2)) != SFGPU_OK) break;
        if (sal)
            for (int k = 0; k < m; k++) launch_rgb_to_lab(c, P, frame(j0 + k), lab + (size_t)k * 3 * P);
        status = epic_device(c, m, g, costs(q), sal ? lab : nullptr, matches + j0, ep, flows(q), st.data(), Caller{"sfgpu_epicflow_sequence", "pair", j0});
        if (status != SFGPU_OK) break;
        if (stats)
            for (int k = 0; k < m; k++) stats[j0 + k] = st[k];
        if (q + 1 < n_chunks && (status = upload(q + 1)) != SFGPU_OK) break;
        for (int k = 0; k < m && status == SFGPU_OK; k++) {
            float *fx = flows(q) + (size_t)k * 2 * P;
            status = run_two_frame(c, g, fx, fx + P, frame(j0 + k), frame(j0 + k + 1), vp);
            if (status == SFGPU_OK) status = pipe.pass(q); // re-marked per pair: the last mark ends chunk q
            if (status == SFGPU_OK) status = pipe.download(q, {{fx, wx[j0 + k]->data, P * sizeof(float)}, {fx + P, wy[j0 + k]->data, P * sizeof(float)}});
        }
    }
    return pipe.finish(status);
}

} // namespace sf

using namespace sf;

extern "C" {

int sfgpu_rgb_to_lab(sfgpu_ctx *c, color_image_t *dst, const color_image_t *src) {
    Geom g;
    if (!c) {
        set_error("sfgpu_rgb_to_lab: null argument");
        return SFGPU_ERR_ARG;
    }
    if (!arg_geom("sfgpu_rgb_to_lab: ", "src", src, g) || !arg_is("sfgpu_rgb_to_lab: ", "dst", dst, g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    int rc = c->ensure_io(6 * P);
    if (rc != SFGPU_OK) return rc;
    rc = host_copies(c, {{c->io, src->c1, 3 * P * sizeof(float)}}, true);
    if (rc != SFGPU_OK) return rc;
    launch_rgb_to_lab(c, P, c->io, c->io + 3 * P);
    SF_CUDA(cudaGetLastError());
    rc = host_copies(c, {{c->io + 3 * P, dst->c1, 3 * P * sizeof(float)}}, false);
    if (rc != SFGPU_OK) return rc;
    SF_CUDA(cudaStreamSynchronize(c->stream));
    return SFGPU_OK;
}

int sfgpu_epicflow_sequence(sfgpu_ctx *c, int n_pairs, const color_image_t *const *frames, const float_image *const *matches,
                            float_image *const *edges, const epic_params_t *epic_params, const variational_params_t *flow_params,
                            image_t *const *wx, image_t *const *wy, sfgpu_epic_stats_t *stats) {
    const Caller who{"sfgpu_epicflow_sequence", "pair", 0};
    if (!c || n_pairs < 1 || !frames || !matches || !edges || !epic_params || !wx || !wy) {
        set_error("sfgpu_epicflow_sequence: bad argument (n_pairs >= 1, non-null context, arrays and epic_params)");
        return SFGPU_ERR_ARG;
    }
    const char *const names[3] = {"wx", "wy", "frames[0]"};
    Geom g;
    int rc = epic_check_args(c, n_pairs, wx, wy, frames, matches, edges, epic_params, who, names, g);
    if (rc != SFGPU_OK) return rc;
    for (int j = 0; j < n_pairs; j++) // frames[1..n_pairs], each under the first pair that reads it
        if (!arg_is(who.at(j), "frames[" + std::to_string(j + 1) + "]", frames[j + 1], g)) return SFGPU_ERR_ARG;
    SF_CUDA(cudaSetDevice(c->device));
    return run_epicflow(c, n_pairs, g, frames, matches, edges, epic_params, flow_params, wx, wy, stats);
}

} // extern "C"
