// sf_sequence.cu -- pipelined refinement of consecutive frame pairs through host buffers (BASELINE config 5; the shard
// loop of adaptiveFR.cpp:496-574 / slow_flow.cpp:706): sfgpu_variational_sequence (fp32 planar frames) and
// sfgpu_variational_sequence_u8 / _u16 (the integer images the reference holds before its float conversion,
// adaptiveFR.cpp:450-464 colorMat2colorImg<Vec3b> / mat2colorImg<uchar>, slow_flow.cpp:470-477 convertTo(CV_32F)).
//
// The copies go through CopyPipeline (sf_hostcopy.cu), one stage per pair: with page-locked caller memory the upload of
// pair j+1 and the download of pair j-1 overlap the solve of pair j; pageable memory takes the staged copies.  A frame
// shared by two pairs is uploaded once (3-slot device ring); with `continue_from_previous` the first frame of a call is
// the last frame of the previous call and is not uploaded at all.  Integer frames cross PCIe as they are (1 or 2 bytes
// per sample, interleaved) and are converted to the planar fp32 layout of image.c:71-89 on the device -- exact, since
// every 8-/16-bit integer is a float -- which takes the upload per 2560x1440 field from 73.7 MB to 40.6 MB.
#include <algorithm>

#include "sf_context.cuh"

namespace sf {

// interleaved (or single-channel) integer frame -> planar fp32; the stride padding is zeroed.  One thread = 4 pixels.
template <typename T>
__global__ void __launch_bounds__(256) k_unpack_frame(Geom g, const unsigned char *__restrict__ raw, size_t step, int channels,
                                                      float *__restrict__ dst) {
    pdl_enter();
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x4 >= g.S) return;
    const T *row = reinterpret_cast<const T *>(raw + (size_t)y * step);
    const size_t P = g.plane();
    float4 o[3];
    float *f = reinterpret_cast<float *>(o);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int x = x4 + k;
        if (x < g.W) {
            if (channels == 1) { // mat2colorImg<T>: the grey value goes to all three channels (utils/utils.h:122-130)
                const float v = (float)row[x];
                f[k] = v; f[4 + k] = v; f[8 + k] = v;
            } else { // colorMat2colorImg<Vec3>: channel c of the Mat -> plane c
                f[k] = (float)row[3 * x]; f[4 + k] = (float)row[3 * x + 1]; f[8 + k] = (float)row[3 * x + 2];
            }
        } else {
            f[k] = 0.f; f[4 + k] = 0.f; f[8 + k] = 0.f;
        }
    }
    const size_t off = (size_t)y * g.S + x4;
#pragma unroll
    for (int c = 0; c < 3; c++) *reinterpret_cast<float4 *>(dst + c * P + off) = o[c];
}

struct SeqFrames { // where the frames of a call come from
    const color_image_t *const *f32 = nullptr; // planar fp32 (3*P floats at c1)
    const sf_frame_int_t *ints = nullptr;      // packed integer frames
    int depth = 0;                             // 8 or 16 for ints
    size_t raw_bytes(int f) const { return ints ? (size_t)ints[f].step * ints[f].height : 0; }
    const void *host(int f) const { return ints ? ints[f].data : (const void *)f32[f]->c1; }
};

void launch_unpack_frame(cudaStream_t st, Geom g, const unsigned char *raw, size_t step, int channels, int bits, float *dst) {
    const dim3 grid((g.S / 4 + 255) / 256, g.H);
    if (bits == 8)
        launch_pdl(k_unpack_frame<unsigned char>, grid, dim3(256), 0, st, g, raw, step, channels, dst);
    else
        launch_pdl(k_unpack_frame<unsigned short>, grid, dim3(256), 0, st, g, raw, step, channels, dst);
}

static void launch_unpack(sfgpu_ctx *c, Geom g, const SeqFrames &src, int f, const unsigned char *raw, float *dst) {
    launch_unpack_frame(c->stream, g, raw, (size_t)src.ints[f].step, src.ints[f].channels, src.depth, dst);
    c->prof_acc.kernel_launches++;
}

// the arguments have been checked; g: their geometry
static int run_sequence(sfgpu_ctx *c, int n_pairs, const SeqFrames &src, Geom g, image_t *const *wx, image_t *const *wy,
                        const variational_params_t *params, bool continue_from_previous) {
    SF_CUDA(cudaSetDevice(c->device));
    const size_t P = g.plane();
    const bool keep = continue_from_previous && c->seq_last_slot >= 0 && c->seq_geom.W == g.W && c->seq_geom.H == g.H;
    if (continue_from_previous && !keep) {
        set_error("sequence: continue_from_previous needs a previous sequence call of the same geometry on this context");
        return SFGPU_ERR_ARG;
    }
    const int base = keep ? c->seq_last_slot : 0; // ring slot of frame 0
    c->seq_last_slot = -1;
    // device ring: 3 frame slots, 3 flow slots (pair j -> slot j%3)
    const float *io_before = c->io;
    int rc = c->ensure_io((3 * 3 + 3 * 2) * P);
    if (rc != SFGPU_OK) return rc;
    if (keep && c->io != io_before) {
        set_error("sequence: the frame ring was re-allocated since the previous call");
        return SFGPU_ERR_ARG;
    }
    rc = c->ensure_workspace(g);
    if (rc != SFGPU_OK) return rc;
    size_t raw_slot = 0;
    if (src.ints) {
        for (int f = 0; f <= n_pairs; f++) raw_slot = std::max(raw_slot, src.raw_bytes(f));
        raw_slot = (raw_slot + 255) & ~(size_t)255;
        if (raw_slot > c->seq_raw_bytes) {
            SF_CUDA(cudaStreamSynchronize(c->stream));
            if (c->seq_raw) cudaFree(c->seq_raw);
            c->seq_raw = nullptr;
            c->seq_raw_bytes = 0;
            SF_CUDA(cudaMalloc(&c->seq_raw, 3 * raw_slot));
            c->seq_raw_bytes = raw_slot;
        }
        raw_slot = c->seq_raw_bytes;
    }
    auto frame_slot = [&](int f) { return c->io + (size_t)((f + base) % 3) * 3 * P; };
    auto raw_of = [&](int f) { return c->seq_raw + (size_t)((f + base) % 3) * raw_slot; };
    auto flow_slot = [&](int j) { return c->io + 9 * P + (size_t)(j % 3) * 2 * P; };
    auto frame_copy = [&](int f) -> HostCopy {
        if (src.ints) return HostCopy{raw_of(f), const_cast<void *>(src.host(f)), src.raw_bytes(f)};
        return HostCopy{frame_slot(f), const_cast<void *>(src.host(f)), 3 * P * sizeof(float)};
    };
    auto flow_copies = [&](int j) -> std::vector<HostCopy> {
        return {{flow_slot(j), wx[j]->data, P * sizeof(float)}, {flow_slot(j) + P, wy[j]->data, P * sizeof(float)}};
    };
    CopyPipeline pipe(c); // stage j = pair j
    // inputs of pair j: frame j+1 (and frame 0 for j == 0) + initial flow j.  Frame slot (j+1)%3 was last read by pair
    // j-2, flow slot j%3 last drained for pair j-3.
    auto upload = [&](int j) {
        std::vector<HostCopy> up = flow_copies(j);
        up.insert(up.begin(), frame_copy(j + 1));
        if (j == 0 && !keep) up.insert(up.begin(), frame_copy(0));
        return pipe.upload(j, up, j - 2, j - 3);
    };
    std::vector<const void *> buffers;
    for (int f = 0; f <= n_pairs; f++) buffers.push_back(src.host(f));
    for (int j = 0; j < n_pairs; j++) buffers.insert(buffers.end(), {wx[j]->data, wy[j]->data});
    int status = pipe.start(buffers);
    if (status == SFGPU_OK) status = upload(0);
    for (int j = 0; j < n_pairs && status == SFGPU_OK; j++) {
        if ((status = pipe.wait(j)) != SFGPU_OK) break;
        if (src.ints) {
            if (j == 0 && !keep) launch_unpack(c, g, src, 0, raw_of(0), frame_slot(0));
            launch_unpack(c, g, src, j + 1, raw_of(j + 1), frame_slot(j + 1));
        }
        if ((status = run_two_frame(c, g, flow_slot(j), flow_slot(j) + P, frame_slot(j), frame_slot(j + 1), params)) != SFGPU_OK) break;
        if ((status = pipe.pass(j)) != SFGPU_OK) break;
        if (j + 1 < n_pairs && (status = upload(j + 1)) != SFGPU_OK) break;
        status = pipe.download(j, flow_copies(j));
    }
    status = pipe.finish(status);
    if (status == SFGPU_OK) {
        c->seq_geom = g;
        c->seq_last_slot = (n_pairs + base) % 3;
    }
    return status;
}

// The argument checks of the three entries, all before anything is touched: the flows' geometry from wx[0], every flow
// plane, then frame f under the first pair that reads it.
static int sequence(sfgpu_ctx *c, const char *fn, int n_pairs, const SeqFrames &src, image_t *const *wx, image_t *const *wy,
                    const variational_params_t *params, int continue_from_previous) {
    if (!c || n_pairs < 0 || !(src.f32 || src.ints) || !wx || !wy) {
        set_error(std::string(fn) + ": bad argument");
        return SFGPU_ERR_ARG;
    }
    if (n_pairs == 0) return SFGPU_OK;
    const Caller who{fn, "pair", 0};
    Geom g;
    if (!arg_geom(who.at(0), "wx", wx[0], g)) return SFGPU_ERR_ARG;
    for (int j = 0; j < n_pairs; j++)
        if (!arg_is(who.at(j), "wx", wx[j], g) || !arg_is(who.at(j), "wy", wy[j], g)) return SFGPU_ERR_ARG;
    for (int f = 0; f <= n_pairs; f++) {
        const std::string at = who.at(std::max(f - 1, 0)), name = "frames[" + std::to_string(f) + "]";
        if (src.f32 ? !arg_is(at, name, src.f32[f], g) : !arg_frame_int(at, name, src.ints[f], g, src.depth)) return SFGPU_ERR_ARG;
    }
    return run_sequence(c, n_pairs, src, g, wx, wy, params, continue_from_previous != 0);
}

} // namespace sf

using namespace sf;

extern "C" {

int sfgpu_variational_sequence(sfgpu_ctx *c, int n_pairs, const color_image_t *const *frames, image_t *const *wx,
                               image_t *const *wy, const variational_params_t *params) {
    return sequence(c, "sfgpu_variational_sequence", n_pairs, SeqFrames{frames}, wx, wy, params, 0);
}

int sfgpu_variational_sequence_u8(sfgpu_ctx *c, int n_pairs, const sf_frame_int_t *frames, image_t *const *wx, image_t *const *wy,
                                  const variational_params_t *params, int continue_from_previous) {
    return sequence(c, "sfgpu_variational_sequence_u8", n_pairs, SeqFrames{nullptr, frames, 8}, wx, wy, params, continue_from_previous);
}

int sfgpu_variational_sequence_u16(sfgpu_ctx *c, int n_pairs, const sf_frame_int_t *frames, image_t *const *wx, image_t *const *wy,
                                   const variational_params_t *params, int continue_from_previous) {
    return sequence(c, "sfgpu_variational_sequence_u16", n_pairs, SeqFrames{nullptr, frames, 16}, wx, wy, params, continue_from_previous);
}

} // extern "C"
