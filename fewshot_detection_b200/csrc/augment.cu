// Training-input augmentation on the device (SURVEY.md §8f row 3): the pixel work of image.data_augmentation
// (image.py:52-87) + transforms.ToTensor for a whole batch in one launch, from decoded uint8 RGB images.
//
//   crop (zero fill outside the source, image.py:72)  ->  resize to the network input (image.py:77; PIL's separable
//   two-pass resampler with 22-bit fixed-point coefficients and a uint8 rounding after EACH pass)  ->  horizontal
//   flip (:79-80)  ->  RGB->HSV, S *= dsat, V *= dexp, H += dhue*255 with wrap (image.py:19-37; PIL `point` tables:
//   round-half-even, clipped to 0..255)  ->  HSV->RGB  ->  float32 / 255 in NCHW (ToTensor, train_meta.py:176-178).
//
// The reference calls `cropped.resize(shape)` without a filter argument, so the filter is whatever the installed
// Pillow defaults to: BICUBIC since Pillow 7 (the container's 12.2), NEAREST before.  Both are implemented
// (`filter` = 3 / 0, PIL's enum values).  Results are bit-identical to Pillow's uint8 pipeline: integer arithmetic
// for the resampling, IEEE float/double operations in Pillow's order (explicit round-to-nearest intrinsics, no FMA
// contraction) for the coefficient tables and the colour conversions (Convert.c rgb2hsv_row / hsv2rgb follow
// colorsys.py).  tests/test_augment_host_emul.py checks the kernel source against Pillow itself on the CPU
// (exhaustively over all 2^24 colours for the two conversions).
#include "common.cuh"

namespace fsdet {

constexpr int kPrecisionBits = 32 - 8 - 2;  // Pillow Resample.c PRECISION_BITS
constexpr int kGeomInts = 8;                // per image: ow, oh, pleft, ptop, cw, ch, flip, distort
constexpr int kAugThreads = 256;

// PIL.Image.BICUBIC kernel (Resample.c bicubic_filter, a = -0.5), double arithmetic in Pillow's order
__device__ __forceinline__ double bicubic_filter(double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) {
        const double t = __dsub_rn(__dmul_rn(a + 2.0, x), a + 3.0);
        return __dadd_rn(__dmul_rn(__dmul_rn(t, x), x), 1.0);
    }
    if (x < 2.0) {
        const double t = __dadd_rn(__dmul_rn(__dsub_rn(x, 5.0), x), 8.0);
        return __dmul_rn(__dsub_rn(__dmul_rn(t, x), 4.0), a);
    }
    return 0.0;
}

// Resample.c precompute_coeffs + normalize_coeffs_8bpc for ONE output coordinate.
// row = {xmin, n, k[0..kmax)}; returns false when the taps do not fit kmax.
__device__ __forceinline__ bool resample_row(int insize, int outsize, int xx, int kmax, int32_t* row) {
    const double scale = __ddiv_rn((double)insize, (double)outsize);
    const double filterscale = scale < 1.0 ? 1.0 : scale;
    const double support = __dmul_rn(2.0, filterscale);
    const double ss = __ddiv_rn(1.0, filterscale);
    const double center = __dmul_rn((double)xx + 0.5, scale);
    int xmin = (int)__dadd_rn(__dsub_rn(center, support), 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)__dadd_rn(__dadd_rn(center, support), 0.5);
    if (xmax > insize) xmax = insize;
    const int n = xmax - xmin;
    row[0] = xmin;
    row[1] = n;
    if (n > kmax) return false;
    double ww = 0.0;
    for (int x = 0; x < n; ++x) {
        const double w = bicubic_filter(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
        ww = __dadd_rn(ww, w);
    }
    for (int x = 0; x < n; ++x) {
        double w = bicubic_filter(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
        if (ww != 0.0) w = __ddiv_rn(w, ww);
        const double scaled = __dmul_rn(w, (double)(1 << kPrecisionBits));
        row[2 + x] = w < 0.0 ? (int)__dadd_rn(-0.5, scaled) : (int)__dadd_rn(0.5, scaled);
    }
    for (int x = n; x < kmax; ++x) row[2 + x] = 0;
    return true;
}

// PIL `point(lambda i: f(i))` table entry: round-half-even, clip to a byte
__device__ __forceinline__ uint8_t lut_byte(double v) {
    const double r = rint(v);
    return (uint8_t)(r < 0.0 ? 0.0 : (r > 255.0 ? 255.0 : r));
}

// Setup: one thread per (image, axis, output coordinate) fills the coefficient tables; the first 768 threads of
// each image also fill its three colour tables (image.py:19-33).
//   tables [n][2][L][2 + kmax] int32 (L = max(W, H); axis 0 = horizontal), luts [n][3][256] uint8, status int32[1]
// filter == 0 (PIL NEAREST = Geometry.c ImagingScaleAffine): the source coordinate of output x is (int)xo with
// xo = a*0.5 + a + a + ... (x sequential double additions of a = in/out), so one thread per axis runs the serial
// recurrence and stores the index (-1 = outside: PIL leaves the zero fill) in row[0].
__global__ void augment_setup_kernel(const int32_t* __restrict__ geom, const double* __restrict__ color, int n, int W, int H,
                                     int L, int kmax, int filter, int32_t* __restrict__ tables, uint8_t* __restrict__ luts,
                                     int32_t* __restrict__ status) {
    const int img = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int32_t* g = geom + (size_t)img * kGeomInts;
    if (t < 2 * L) {
        const int axis = t / L, xx = t - axis * L;
        const int outsize = axis == 0 ? W : H;
        const int insize = axis == 0 ? g[4] : g[5];
        int32_t* row = tables + (((size_t)img * 2 + axis) * L + xx) * (2 + kmax);
        if (insize <= 0) {
            if (xx == 0) atomicExch(status, 1 + img);
        } else if (filter == 0) {
            if (xx == 0) {
                const double a = __ddiv_rn((double)insize, (double)outsize);
                double xo = __dmul_rn(a, 0.5);
                for (int x = 0; x < outsize; ++x) {
                    const int xin = (int)xo;
                    row[(size_t)x * (2 + kmax)] = (xin >= 0 && xin < insize) ? xin : -1;
                    row[(size_t)x * (2 + kmax) + 1] = 1;
                    xo = __dadd_rn(xo, a);
                }
            }
        } else if (xx < outsize) {
            if (!resample_row(insize, outsize, xx, kmax, row)) atomicExch(status, 1 + img);
        }
    }
    if (t < 768) {
        const int ch = t >> 8, i = t & 255;
        const double* c = color + (size_t)img * 3;
        double v;
        if (ch == 0) {  // change_hue, image.py:25-31
            v = __dadd_rn((double)i, __dmul_rn(c[0], 255.0));
            if (v > 255.0) v = __dsub_rn(v, 255.0);
            if (v < 0.0) v = __dadd_rn(v, 255.0);
        } else {
            v = __dmul_rn((double)i, c[ch]);  // i * sat, i * val
        }
        luts[((size_t)img * 3 + ch) * 256 + i] = lut_byte(v);
    }
}

// Convert.c rgb2hsv_row
__device__ __forceinline__ void rgb2hsv(int r, int g, int b, int& uh, int& us, int& uv) {
    const int maxc = max(r, max(g, b)), minc = min(r, min(g, b));
    uv = maxc;
    if (minc == maxc) {
        uh = 0;
        us = 0;
        return;
    }
    const float cr = (float)(maxc - minc);
    const float s = __fdiv_rn(cr, (float)maxc);
    const float rc = __fdiv_rn((float)(maxc - r), cr);
    const float gc = __fdiv_rn((float)(maxc - g), cr);
    const float bc = __fdiv_rn((float)(maxc - b), cr);
    float h;
    if (r == maxc) h = __fsub_rn(bc, gc);
    else if (g == maxc) h = (float)__dsub_rn(__dadd_rn(2.0, (double)rc), (double)bc);
    else h = (float)__dsub_rn(__dadd_rn(4.0, (double)gc), (double)rc);
    h = (float)fmod(__dadd_rn(__ddiv_rn((double)h, 6.0), 1.0), 1.0);
    int ih = (int)__dmul_rn((double)h, 255.0), is = (int)__dmul_rn((double)s, 255.0);
    uh = ih < 0 ? 0 : (ih > 255 ? 255 : ih);
    us = is < 0 ? 0 : (is > 255 ? 255 : is);
}

__device__ __forceinline__ int round_clip8(double v) {  // C round(): half away from zero, then CLIP8
    const double r = round(v);
    return r < 0.0 ? 0 : (r > 255.0 ? 255 : (int)r);
}

// Convert.c hsv2rgb
__device__ __forceinline__ void hsv2rgb(int h, int s, int v, int& r, int& g, int& b) {
    if (s == 0) {
        r = g = b = v;
        return;
    }
    const double h6 = __ddiv_rn(__dmul_rn((double)(float)h, 6.0), 255.0);
    const int i = (int)floor(h6);
    const float f = (float)__dsub_rn(h6, (double)(float)i);
    const double sd = __ddiv_rn((double)(float)s, 255.0);
    const float fs = (float)__dmul_rn(sd, (double)f);
    const double vd = (double)(float)v;
    const int p = round_clip8(__dmul_rn(vd, __dsub_rn(1.0, sd)));
    const int q = round_clip8(__dmul_rn(vd, __dsub_rn(1.0, (double)fs)));
    const int t = round_clip8(__dmul_rn(vd, __dadd_rn(__dsub_rn(1.0, sd), (double)fs)));
    switch (i % 6) {
        case 0: r = v; g = t; b = p; break;
        case 1: r = q; g = v; b = p; break;
        case 2: r = p; g = v; b = t; break;
        case 3: r = p; g = q; b = v; break;
        case 4: r = t; g = p; b = v; break;
        default: r = v; g = p; b = q; break;
    }
}

__device__ __forceinline__ int clip8_fixed(int acc) {  // Resample.c clip8
    const int v = acc >> kPrecisionBits;
    return v < 0 ? 0 : (v > 255 ? 255 : v);
}

struct AugArgs {
    const uint8_t* const* src;  // [n] device pointers to HWC uint8 RGB images
    const int32_t* geom;        // [n][8]
    const int32_t* tables;      // [n][2][L][2 + kmax]
    const uint8_t* luts;        // [n][3][256]
    float* out;                 // [n][3][H][W], image i at out + i * out_pitch
    uint8_t* out_u8;            // optional [n][H][W][3]: the uint8 image before ToTensor (what PIL would hold)
    int n, W, H, L, kmax, filter;
    long long out_pitch;        // floats from one image's output to the next (>= 3*H*W)
};

// cropped pixel (x, y) of image.py:72: zero outside the source
__device__ __forceinline__ void crop_px(const uint8_t* __restrict__ s, int ow, int oh, int pleft, int ptop, int x, int y,
                                        int& r, int& g, int& b) {
    const int sx = x + pleft, sy = y + ptop;
    if (sx < 0 || sy < 0 || sx >= ow || sy >= oh) {
        r = g = b = 0;
        return;
    }
    const uint8_t* p = s + ((size_t)sy * ow + sx) * 3;
    r = __ldg(p);
    g = __ldg(p + 1);
    b = __ldg(p + 2);
}

// One thread per output pixel (all three channels).  The horizontal pass is recomputed for each of the pixel's
// vertical taps (n_y * n_x * 3 integer MACs, ~150 at VOC sizes) instead of staging an intermediate image: the source
// rows stay in L1/L2 and the only HBM traffic is the source bytes once and the float32 output once.
__global__ void __launch_bounds__(kAugThreads) augment_kernel(AugArgs p) {
    const int img = blockIdx.y;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.W * p.H) return;
    const int yy = idx / p.W, xx = idx - yy * p.W;
    const int32_t* g = p.geom + (size_t)img * kGeomInts;
    const int ow = g[0], oh = g[1], pleft = g[2], ptop = g[3], cw = g[4], ch = g[5], flip = g[6], distort = g[7];
    (void)cw; (void)ch;
    const uint8_t* s = p.src[img];
    int r, gg, b;
    if (p.filter == 0) {
        const int stride = 2 + p.kmax;
        const int sx = p.tables[(((size_t)img * 2 + 0) * p.L + xx) * stride];
        const int sy = p.tables[(((size_t)img * 2 + 1) * p.L + yy) * stride];
        if (sx < 0 || sy < 0) r = gg = b = 0;
        else crop_px(s, ow, oh, pleft, ptop, sx, sy, r, gg, b);
    } else {
        const int stride = 2 + p.kmax;
        const int32_t* kx = p.tables + (((size_t)img * 2 + 0) * p.L + xx) * stride;
        const int32_t* ky = p.tables + (((size_t)img * 2 + 1) * p.L + yy) * stride;
        const int xmin = kx[0], nx = kx[1], ymin = ky[0], ny = ky[1];
        const bool hpass = cw != p.W, vpass = ch != p.H;  // Resample.c skips a pass whose size does not change
        int ar = 1 << (kPrecisionBits - 1), ag = ar, ab = ar;
        const int y0 = vpass ? ymin : yy, y1 = vpass ? ymin + ny : yy + 1;
        for (int y = y0; y < y1; ++y) {
            int tr, tg, tb;
            if (hpass) {
                int hr = 1 << (kPrecisionBits - 1), hg = hr, hb = hr;
                for (int x = 0; x < nx; ++x) {
                    int cr, cg, cb;
                    crop_px(s, ow, oh, pleft, ptop, xmin + x, y, cr, cg, cb);
                    const int k = kx[2 + x];
                    hr += cr * k;
                    hg += cg * k;
                    hb += cb * k;
                }
                tr = clip8_fixed(hr);
                tg = clip8_fixed(hg);
                tb = clip8_fixed(hb);
            } else {
                crop_px(s, ow, oh, pleft, ptop, xx, y, tr, tg, tb);
            }
            if (vpass) {
                const int k = ky[2 + (y - ymin)];
                ar += tr * k;
                ag += tg * k;
                ab += tb * k;
            } else {
                ar = tr; ag = tg; ab = tb;
            }
        }
        if (vpass) {
            r = clip8_fixed(ar);
            gg = clip8_fixed(ag);
            b = clip8_fixed(ab);
        } else {
            r = ar; gg = ag; b = ab;
        }
    }
    if (distort) {
        int h, sat, v;
        rgb2hsv(r, gg, b, h, sat, v);
        const uint8_t* lut = p.luts + (size_t)img * 768;
        h = __ldg(lut + h);
        sat = __ldg(lut + 256 + sat);
        v = __ldg(lut + 512 + v);
        hsv2rgb(h, sat, v, r, gg, b);
    }
    const int ox = flip ? p.W - 1 - xx : xx;  // Image.FLIP_LEFT_RIGHT (colour ops are per pixel: order is irrelevant)
    const size_t plane = (size_t)p.W * p.H;
    float* o = p.out + (size_t)img * p.out_pitch + (size_t)yy * p.W + ox;
    o[0] = __fdiv_rn((float)r, 255.f);
    o[plane] = __fdiv_rn((float)gg, 255.f);
    o[2 * plane] = __fdiv_rn((float)b, 255.f);
    if (p.out_u8) {
        uint8_t* u = p.out_u8 + ((size_t)img * plane + (size_t)yy * p.W + ox) * 3;
        u[0] = (uint8_t)r;
        u[1] = (uint8_t)gg;
        u[2] = (uint8_t)b;
    }
}

// dataset.MetaDataset.get_img_mask (dataset.py:378-398): mask[:, y1:y2, x1:x2] = 1 for n support images at once;
// rects [n][4] = x1, y1, x2, y2 already rounded / clamped on the host as the reference does (Python round()).
__global__ void box_masks_kernel(const int32_t* __restrict__ rects, int n, int H, int W, float* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)n * H * W;
    if (i >= total) return;
    const int img = (int)(i / ((size_t)H * W));
    const int rem = (int)(i - (size_t)img * H * W);
    const int y = rem / W, x = rem - y * W;
    const int32_t* r = rects + (size_t)img * 4;
    out[i] = (x >= r[0] && x < r[2] && y >= r[1] && y < r[3]) ? 1.f : 0.f;
}

}  // namespace fsdet

#ifndef FSDET_HOST_EMULATION
using namespace fsdet;

extern "C" size_t fsdet_augment_workspace_bytes(int n, int W, int H, int kmax) {
    if (n <= 0 || W <= 0 || H <= 0 || kmax <= 0) return 0;
    const size_t L = (size_t)(W > H ? W : H);
    return (size_t)n * 2 * L * (2 + (size_t)kmax) * sizeof(int32_t) + (size_t)n * 768;
}

extern "C" int fsdet_augment_batch(const uint8_t* const* src, const int32_t* geom, const double* color, int n, int W,
                                   int H, int kmax, int filter, void* workspace, size_t workspace_bytes, float* out,
                                   uint8_t* out_u8, int32_t* status, void* stream) {
    FSDET_CHECK_ARG(W > 0 && H > 0, "augment_batch: bad shape");
    return fsdet_augment_batch_pitched(src, geom, color, n, W, H, kmax, filter, workspace, workspace_bytes, out,
                                       (size_t)3 * W * H, out_u8, status, stream);
}

extern "C" int fsdet_augment_batch_pitched(const uint8_t* const* src, const int32_t* geom, const double* color, int n, int W,
                                           int H, int kmax, int filter, void* workspace, size_t workspace_bytes, float* out,
                                           size_t out_pitch, uint8_t* out_u8, int32_t* status, void* stream) {
    FSDET_CHECK_ARG(src && geom && color && workspace && out && status, "augment_batch: null pointer");
    FSDET_CHECK_ARG(n >= 0 && W > 0 && H > 0, "augment_batch: bad shape");
    FSDET_CHECK_ARG(out_pitch >= (size_t)3 * W * H, "augment_batch: output pitch %zu < 3*H*W", out_pitch);
    FSDET_CHECK_ARG(filter == 0 || filter == 3, "augment_batch: filter %d (0 = NEAREST, 3 = BICUBIC)", filter);
    FSDET_CHECK_ARG(kmax >= 1 && kmax <= 254, "augment_batch: kmax %d (1..254)", kmax);
    FSDET_CHECK_ARG(workspace_bytes >= fsdet_augment_workspace_bytes(n, W, H, kmax) && aligned16(workspace),
                    "augment_batch: workspace too small or misaligned");
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(status, 0, sizeof(int32_t), s);
    if (e != cudaSuccess) { set_error("augment_batch: memset: %s", cudaGetErrorString(e)); return (int)e; }
    if (n == 0) return 0;
    const int L = W > H ? W : H;
    int32_t* tables = reinterpret_cast<int32_t*>(workspace);
    uint8_t* luts = reinterpret_cast<uint8_t*>(workspace) + (size_t)n * 2 * L * (2 + (size_t)kmax) * sizeof(int32_t);
    const int setup_threads = 2 * L > 768 ? 2 * L : 768;
    augment_setup_kernel<<<dim3(ceil_div(setup_threads, 256), n), 256, 0, s>>>(geom, color, n, W, H, L, kmax, filter, tables,
                                                                               luts, status);
    int st = launch_status("augment_setup");
    if (st) return st;
    AugArgs p;
    p.src = src; p.geom = geom; p.tables = tables; p.luts = luts; p.out = out; p.out_u8 = out_u8;
    p.n = n; p.W = W; p.H = H; p.L = L; p.kmax = kmax; p.filter = filter; p.out_pitch = (long long)out_pitch;
    augment_kernel<<<dim3(ceil_div((long long)W * H, kAugThreads), n), kAugThreads, 0, s>>>(p);
    return launch_status("augment");
}

extern "C" int fsdet_box_masks(const int32_t* rects, int n, int H, int W, float* out, void* stream) {
    FSDET_CHECK_ARG(rects && out && n >= 0 && H > 0 && W > 0, "box_masks: bad args");
    const size_t total = (size_t)n * H * W;
    if (total == 0) return 0;
    box_masks_kernel<<<ceil_div((long long)total, 256), 256, 0, (cudaStream_t)stream>>>(rects, n, H, W, out);
    return launch_status("box_masks");
}
#endif  // FSDET_HOST_EMULATION
