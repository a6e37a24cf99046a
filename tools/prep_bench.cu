// Stand-alone timing harness for the two-frame data pass (debug aid, not part of the library): includes the kernel
// sources, fills a frame pair / flow / increment / smoothness weight with a smooth synthetic pattern and times, in one
// process and alternating,
//   chain: k_flow_smooth (launch_smoothness / launch_update_smoothness) + k_prep_two_frame (launch_prep_two_frame)
//   fused: k_prep_fused (launch_prep_fused)
// for both outer-iteration forms (first: no flow update; later: w += du).  Prints the average time per launch (per pair
// of launches for the chain) and whether the two produce identical outputs: the five system planes, psi_h, psi_v and the
// updated flow.  Build variants with -D flags (tools/build_tools.sh).
#include "../slowflow_b200/csrc/sf_prep.cu"
#include "../slowflow_b200/csrc/sf_kernels.cu"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
namespace sf {
void set_error(const std::string &m) { fprintf(stderr, "error: %s\n", m.c_str()); }
bool cuda_ok(cudaError_t e, const char *what) { if (e != cudaSuccess) { fprintf(stderr, "%s: %s\n", what, cudaGetErrorString(e)); return false; } return true; }
}
int main(int argc, char **argv) {
    const int W = argc > 1 ? atoi(argv[1]) : 2560, H = argc > 2 ? atoi(argv[2]) : 1440, reps = argc > 3 ? atoi(argv[3]) : 20;
    const float hd = argc > 4 ? (float)atof(argv[4]) : 0.0f;
    const float hg = 0.71f * 0.5f / 3.f, ha = 0.5f;
    sf::Geom g = sf::make_geom(W, H);
    const size_t P = g.plane();
    enum { IM1 = 0, IM2 = 3, WX = 6, WY = 7, DU = 8, DV = 9, DPS = 10, NIN = 11 };
    std::vector<float> h(NIN * P, 0.f);
    for (int y = 0; y < H; y++)
        for (int x = 0; x < g.S; x++) { // padding columns too: the flow update stores w + du there
            const size_t o = (size_t)y * g.S + x;
            for (int c = 0; c < 3; c++) {
                h[(IM1 + c) * P + o] = 127.f + 60.f * sinf(0.11f * x + 0.07f * y + c) + 30.f * sinf(0.53f * x - 0.31f * y + 2 * c);
                h[(IM2 + c) * P + o] = 127.f + 60.f * sinf(0.11f * (x - 1.3f) + 0.07f * (y - 0.6f) + c) + 30.f * sinf(0.53f * (x - 1.3f) - 0.31f * (y - 0.6f) + 2 * c);
            }
            h[WX * P + o] = 1.3f + 0.4f * sinf(0.013f * y) + ((x * 7 + y * 13) % 17) * 0.02f;
            h[WY * P + o] = 0.6f + 0.3f * cosf(0.017f * x) + ((x * 5 + y * 11) % 13) * 0.02f;
            h[DU * P + o] = 0.05f * sinf(0.031f * x + 0.02f * y) + ((x * 3 + y * 7) % 11) * 0.003f;
            h[DV * P + o] = 0.04f * cosf(0.027f * x - 0.015f * y) + ((x * 11 + y * 5) % 7) * 0.004f;
            h[DPS * P + o] = 0.5f * expf(-0.2f * fabsf(sinf(0.05f * x) + cosf(0.07f * y)));
        }
    enum { A11 = 0, B2 = 4, PH = 5, PV = 6, OX = 7, OY = 8, NOUT = 9 };
    float *in, *out[2];
    cudaMalloc(&in, h.size() * 4);
    cudaMemcpy(in, h.data(), h.size() * 4, cudaMemcpyHostToDevice);
    for (int k = 0; k < 2; k++) { cudaMalloc(&out[k], NOUT * P * 4); cudaMemset(out[k], 0, NOUT * P * 4); }
    int sms = 0; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    sf::Penalty two_frame_reg{-1, 0.f, 0.0, 0.f};
    auto chain = [&](bool update, float *o) {
        const float *fx = in + WX * P, *fy = in + WY * P;
        if (update) {
            sf::launch_update_smoothness(0, g, fx, fy, in + DU * P, in + DV * P, in + DPS * P, ha, two_frame_reg, 1, o + OX * P,
                                         o + OY * P, o + PH * P, o + PV * P);
            fx = o + OX * P; fy = o + OY * P;
        } else {
            sf::launch_smoothness(0, g, fx, fy, in + DPS * P, ha, two_frame_reg, 1, o + PH * P, o + PV * P);
        }
        sf::launch_prep_two_frame(0, g, sms, in + IM1 * P, in + IM2 * P, fx, fy, nullptr, nullptr, o + PH * P, o + PV * P, hd, hg,
                                  o, o + P, o + 2 * P, o + 3 * P, o + 4 * P);
    };
    auto fused = [&](bool update, float *o) {
        sf::launch_prep_fused(0, g, sms, in + IM1 * P, in + IM2 * P, in + WX * P, in + WY * P, update ? in + DU * P : nullptr,
                              update ? in + DV * P : nullptr, in + DPS * P, ha, hd, hg, o + OX * P, o + OY * P, o + PH * P, o + PV * P,
                              o, o + P, o + 2 * P, o + 3 * P, o + 4 * P);
    };
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    auto time = [&](auto fn, bool update, float *o) {
        for (int k = 0; k < 3; k++) fn(update, o);
        cudaEventRecord(e0);
        for (int k = 0; k < reps; k++) fn(update, o);
        cudaEventRecord(e1); cudaEventSynchronize(e1);
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        return ms * 1e3f / reps;
    };
    const char *names[NOUT] = {"a11", "a12", "a22", "b1", "b2", "psi_h", "psi_v", "flow_x", "flow_y"};
    bool all_same = true;
    for (int update = 0; update < 2; update++) {
        float tc[3], tf[3]; // alternating rounds
        for (int k = 0; k < 3; k++) { tc[k] = time(chain, update, out[0]); tf[k] = time(fused, update, out[1]); }
        cudaDeviceSynchronize();
        std::vector<float> a(NOUT * P), b(NOUT * P);
        for (int k = 0; k < 2; k++) cudaMemset(out[k], 0, NOUT * P * 4);
        chain(update, out[0]);
        fused(update, out[1]);
        cudaMemcpy(a.data(), out[0], NOUT * P * 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(b.data(), out[1], NOUT * P * 4, cudaMemcpyDeviceToHost);
        const int nplanes = update ? NOUT : OX;
        size_t diff[NOUT] = {}, nonfinite = 0;
        for (int q = 0; q < nplanes; q++)
            for (size_t i = 0; i < P; i++) {
                if (memcmp(&a[q * P + i], &b[q * P + i], 4)) diff[q]++;
                if (!isfinite(a[q * P + i])) nonfinite++;
            }
        size_t total = 0;
        for (int q = 0; q < nplanes; q++) total += diff[q];
        all_same &= total == 0;
        printf("%dx%d hd=%.3f %s: chain %.2f %.2f %.2f us, fused %.2f %.2f %.2f us per outer iteration (%d launches each, alternating); "
               "fused bytes model %d B/px -> %.0f GB/s; outputs %s",
               W, H, hd, update ? "update" : "first", tc[0], tc[1], tc[2], tf[0], tf[1], tf[2], reps, update ? 80 : 64,
               (update ? 80.0 : 64.0) * W * H / (tf[2] * 1e-6) / 1e9, total ? "DIFFER" : "identical");
        for (int q = 0; q < nplanes; q++)
            if (diff[q]) printf(" %s:%zu", names[q], diff[q]);
        printf(" (nonfinite %zu) err=%s\n", nonfinite, cudaGetErrorString(cudaGetLastError()));
    }
    return all_same ? 0 : 1;
}
