// Host-emulated build of csrc/augment.cu (see cuda_host_emul.h): host pointers instead of device pointers.
// Test tooling only; built by tests/test_augment_host_emul.py with g++.
#include "../../fewshot_detection_b200/csrc/augment.cu"

namespace emul {
Block g_block;
unsigned char* g_dyn_smem = nullptr;
}  // namespace emul
namespace fsdet {
void set_error(const char*, ...) {}
}  // namespace fsdet

using namespace fsdet;

extern "C" int emul_augment_batch_pitched(const uint8_t* const* src, const int32_t* geom, const double* color, int n, int W,
                                          int H, int kmax, int filter, int32_t* tables, uint8_t* luts, float* out,
                                          long long out_pitch, uint8_t* out_u8, int32_t* status) {
    const int L = W > H ? W : H;
    *status = 0;
    const int setup_threads = 2 * L > 768 ? 2 * L : 768;
    emul::launch_serial(dim3(ceil_div(setup_threads, 256), n), dim3(256),
                        [&]() { augment_setup_kernel(geom, color, n, W, H, L, kmax, filter, tables, luts, status); });
    AugArgs p;
    p.src = src; p.geom = geom; p.tables = tables; p.luts = luts; p.out = out; p.out_u8 = out_u8;
    p.n = n; p.W = W; p.H = H; p.L = L; p.kmax = kmax; p.filter = filter; p.out_pitch = out_pitch;
    emul::launch_serial(dim3(ceil_div((long long)W * H, kAugThreads), n), dim3(kAugThreads), [&]() { augment_kernel(p); });
    return 0;
}

extern "C" int emul_augment_batch(const uint8_t* const* src, const int32_t* geom, const double* color, int n, int W, int H,
                                  int kmax, int filter, int32_t* tables, uint8_t* luts, float* out, uint8_t* out_u8,
                                  int32_t* status) {
    return emul_augment_batch_pitched(src, geom, color, n, W, H, kmax, filter, tables, luts, out, 3LL * W * H, out_u8, status);
}

// all 2^24 (a, b, c) byte triples through the two colour conversions: out[(a*65536 + b*256 + c)*3 ..]
extern "C" void emul_rgb2hsv_all(uint8_t* out) {
    for (int r = 0; r < 256; ++r)
        for (int g = 0; g < 256; ++g)
            for (int b = 0; b < 256; ++b) {
                int h, s, v;
                rgb2hsv(r, g, b, h, s, v);
                uint8_t* o = out + ((size_t)r * 65536 + g * 256 + b) * 3;
                o[0] = (uint8_t)h; o[1] = (uint8_t)s; o[2] = (uint8_t)v;
            }
}

extern "C" void emul_hsv2rgb_all(uint8_t* out) {
    for (int h = 0; h < 256; ++h)
        for (int s = 0; s < 256; ++s)
            for (int v = 0; v < 256; ++v) {
                int r, g, b;
                hsv2rgb(h, s, v, r, g, b);
                uint8_t* o = out + ((size_t)h * 65536 + s * 256 + v) * 3;
                o[0] = (uint8_t)r; o[1] = (uint8_t)g; o[2] = (uint8_t)b;
            }
}

extern "C" int emul_box_masks(const int32_t* rects, int n, int H, int W, float* out) {
    emul::launch_serial(dim3(ceil_div((long long)n * H * W, 256)), dim3(256), [&]() { box_masks_kernel(rects, n, H, W, out); });
    return 0;
}
