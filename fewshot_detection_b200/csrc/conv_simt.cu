// fp32 SIMT implicit-GEMM convolution (stride 1, "same" padding, k in {1,3}).
//
// Replaces the cuDNN calls behind nn.Conv2d in the reference
// (darknet_meta.py:236-252) for every layer / precision where the tensor-core
// path (conv_tc.cu) is not used, and is the exact-fp32 parity baseline.
//
//   forward / dgrad : z[p][n]  = sum_k A[p][k] * w[n][k],   A = im2col(x) gathered on the fly
//   wgrad           : dw[n][k] = sum_p dz[p][n] * A[p][k]
//
// Tiles: 128 pixels x BN channels x 16 k, 256 threads, 8 x TN register tile,
// double-buffered shared memory with register prefetch.
#include "common.cuh"

namespace fsdet {

struct ConvArgs {
    const float* x;
    const float* w;
    const float* bias;
    float* z;
    float* stat;
    int ldx, ldz;
    int B, H, W, Cin, Cout, ks, pad;
    int K;        // ks*ks*Cin
    long long M;  // B*H*W
    int accumulate;
};

constexpr int BM = 128;
constexpr int BK = 16;
constexpr int APAD = 4;

template <int TN>
__global__ void __launch_bounds__(256) conv_igemm_kernel(const ConvArgs p) {
    constexpr int BN = 16 * TN;
    __shared__ __align__(16) float As[2][BK][BM + APAD];
    __shared__ __align__(16) float Bs[2][BK][BN + APAD];

    const int tid = threadIdx.x;
    const int tx = tid & 15;   // n direction
    const int ty = tid >> 4;   // m direction
    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int HW = p.H * p.W;

    // ---- A (im2col) load bookkeeping: 2 rows per thread, one float4 of k each
    const int kv = tid & 3;
    const int rowA = tid >> 2;  // 0..63, second row = +64
    int a_h[2], a_w[2];
    bool a_ok[2];
    const float* a_ptr[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        long long m = m0 + rowA + r * 64;
        a_ok[r] = m < p.M;
        long long mm = a_ok[r] ? m : 0;
        int rem = (int)(mm % HW);
        a_h[r] = rem / p.W;
        a_w[r] = rem - a_h[r] * p.W;
        a_ptr[r] = p.x + mm * p.ldx;
    }
    // running decomposition of this thread's k index into (tap, ci)
    int a_ci = kv * 4, a_tap = 0;
    while (a_ci >= p.Cin) { a_ci -= p.Cin; ++a_tap; }

    // ---- B (weights) load bookkeeping
    constexpr int B_ROWS_PER_PASS = 64;
    constexpr int B_PASSES = (BN + B_ROWS_PER_PASS - 1) / B_ROWS_PER_PASS;
    const int rowB = tid >> 2;

    float4 ra[2], rb[B_PASSES];
    const int nk = (p.K + BK - 1) / BK;

    auto load_global = [&](int kc) {
        const int k = kc * BK + kv * 4;
        const bool kok = k < p.K;
        int dy = 0, dx = 0;
        if (p.ks == 3) { dy = a_tap / 3 - 1; dx = a_tap - (a_tap / 3) * 3 - 1; }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            int hh = a_h[r] + dy, ww = a_w[r] + dx;
            if (kok && a_ok[r] && hh >= 0 && hh < p.H && ww >= 0 && ww < p.W)
                v = ldg4(a_ptr[r] + (long long)(dy * p.W + dx) * p.ldx + a_ci);
            ra[r] = v;
        }
#pragma unroll
        for (int q = 0; q < B_PASSES; ++q) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            int rr = rowB + q * B_ROWS_PER_PASS;
            int n = n0 + rr;
            if (rr < BN && kok && n < p.Cout) v = ldg4(p.w + (long long)n * p.K + k);
            rb[q] = v;
        }
        // advance (tap, ci) by BK for the next chunk
        a_ci += BK;
        while (a_ci >= p.Cin) { a_ci -= p.Cin; ++a_tap; }
    };
    auto store_smem = [&](int buf) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            int row = rowA + r * 64;
            As[buf][kv * 4 + 0][row] = ra[r].x;
            As[buf][kv * 4 + 1][row] = ra[r].y;
            As[buf][kv * 4 + 2][row] = ra[r].z;
            As[buf][kv * 4 + 3][row] = ra[r].w;
        }
#pragma unroll
        for (int q = 0; q < B_PASSES; ++q) {
            int rr = rowB + q * B_ROWS_PER_PASS;
            if (rr < BN) {
                Bs[buf][kv * 4 + 0][rr] = rb[q].x;
                Bs[buf][kv * 4 + 1][rr] = rb[q].y;
                Bs[buf][kv * 4 + 2][rr] = rb[q].z;
                Bs[buf][kv * 4 + 3][rr] = rb[q].w;
            }
        }
    };

    float acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    load_global(0);
    store_smem(0);
    __syncthreads();
    int buf = 0;
    for (int kc = 0; kc < nk; ++kc) {
        if (kc + 1 < nk) load_global(kc + 1);
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[8], b[TN];
            float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
            float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
            a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
            a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
            if constexpr (TN == 8) {
                float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
                float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
                b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
                b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
            } else if constexpr (TN == 4) {
                float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
                b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
            } else {
                float2 b0 = *reinterpret_cast<const float2*>(&Bs[buf][kk][tx * 2]);
                b[0] = b0.x; b[1] = b0.y;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (kc + 1 < nk) store_smem(buf ^ 1);
        __syncthreads();
        buf ^= 1;
    }

    // ---- epilogue ------------------------------------------------------
    // column index of register column j
    auto col_of = [&](int j) -> int {
        if constexpr (TN == 8) return (j < 4) ? (tx * 4 + j) : (64 + tx * 4 + (j - 4));
        else if constexpr (TN == 4) return tx * 4 + j;
        else return tx * 2 + j;
    };
    const bool vec_ok = ((p.ldz & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.z) & 15u) == 0) && (TN >= 4);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        long long m = m0 + ((i < 4) ? (ty * 4 + i) : (64 + ty * 4 + (i - 4)));
        if (m >= p.M) continue;
        float* zr = p.z + m * p.ldz;
#pragma unroll
        for (int j0 = 0; j0 < TN; j0 += (TN >= 4 ? 4 : 2)) {
            int n = n0 + col_of(j0);
            if constexpr (TN >= 4) {
                if (vec_ok && n + 3 < p.Cout) {
                    float4 v = make_float4(acc[i][j0], acc[i][j0 + 1], acc[i][j0 + 2], acc[i][j0 + 3]);
                    if (p.bias) { v.x += p.bias[n]; v.y += p.bias[n + 1]; v.z += p.bias[n + 2]; v.w += p.bias[n + 3]; }
                    if (p.accumulate) {
                        float4 o = *reinterpret_cast<const float4*>(zr + n);
                        v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                    }
                    *reinterpret_cast<float4*>(zr + n) = v;
                    continue;
                }
            }
#pragma unroll
            for (int j = j0; j < j0 + (TN >= 4 ? 4 : 2); ++j) {
                int nn = n0 + col_of(j);
                if (nn < p.Cout) {
                    float v = acc[i][j];
                    if (p.bias) v += p.bias[nn];
                    if (p.accumulate) v += zr[nn];
                    zr[nn] = v;
                }
            }
        }
    }

    if (p.stat) {
        // per-CTA column statistics over the valid rows: sum, sum of squares, min, max (BatchNorm partials +
        // the activation range).  Reduce the 16 ty-threads through shared memory (re-using the operand buffers).
        float* red_s = &As[0][0][0];       // [16][BN]
        float* red_mn = red_s + 16 * BN;   // [16][BN]   (As holds 2*16*(128+4) floats)
        float* red_q = &Bs[0][0][0];       // [16][BN]
        float* red_mx = red_q + 16 * BN;   // [16][BN]   (Bs holds 2*16*(BN+4) floats)
        __syncthreads();
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            float s = 0.f, q = 0.f, mn = INFINITY, mx = -INFINITY;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const long long m = m0 + ((i < 4) ? (ty * 4 + i) : (64 + ty * 4 + (i - 4)));
                if (m < p.M) {
                    const float v = acc[i][j];
                    s += v; q += v * v; mn = fminf(mn, v); mx = fmaxf(mx, v);
                }
            }
            red_s[ty * BN + col_of(j)] = s;
            red_q[ty * BN + col_of(j)] = q;
            red_mn[ty * BN + col_of(j)] = mn;
            red_mx[ty * BN + col_of(j)] = mx;
        }
        __syncthreads();
        if (tid < BN) {
            int n = n0 + tid;
            if (n < p.Cout) {
                float s = 0.f, q = 0.f, mn = INFINITY, mx = -INFINITY;
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    s += red_s[t * BN + tid]; q += red_q[t * BN + tid];
                    mn = fminf(mn, red_mn[t * BN + tid]); mx = fmaxf(mx, red_mx[t * BN + tid]);
                }
                float* dst = p.stat + (long long)blockIdx.x * 4 * p.Cout;
                dst[n] = s;
                dst[p.Cout + n] = q;
                dst[2 * p.Cout + n] = mn;
                dst[3 * p.Cout + n] = mx;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// wgrad: dw[co][kidx] = sum_p dz[p][co] * A[p][kidx]
struct WgradArgs {
    const float* x;
    const float* dz;
    float* out;  // dw (splits == 1) or workspace [splits][Cout][K]
    int ldx, lddz;
    int B, H, W, Cin, Cout, ks, pad, K;
    long long M;
    long long pix_per_split;
};

template <int BMC>  // co tile: 64 or 128
__global__ void __launch_bounds__(256) conv_wgrad_kernel(const WgradArgs p) {
    constexpr int BNK = 128;
    constexpr int TM = BMC / 16;  // 4 or 8
    __shared__ __align__(16) float As[2][BK][BMC];
    __shared__ __align__(16) float Bs[2][BK][BNK];

    const int tid = threadIdx.x;
    const int tx = tid & 15;  // kidx direction
    const int ty = tid >> 4;  // co direction
    const int k0 = blockIdx.x * BNK;
    const int co0 = blockIdx.y * BMC;
    const long long pbeg = (long long)blockIdx.z * p.pix_per_split;
    long long pend = pbeg + p.pix_per_split;
    if (pend > p.M) pend = p.M;
    const int HW = p.H * p.W;

    // dz loads: BK x BMC floats
    constexpr int A_VECS_PER_ROW = BMC / 4;             // 16 or 32
    constexpr int A_ROWS_PER_PASS = 256 / A_VECS_PER_ROW;  // 16 or 8
    constexpr int A_PASSES = BK / A_ROWS_PER_PASS;      // 1 or 2
    const int a_vec = tid % A_VECS_PER_ROW;
    const int a_row = tid / A_VECS_PER_ROW;
    const int a_co = co0 + a_vec * 4;
    const bool a_cok = a_co < p.Cout;  // Cout % 4 == 0 is required

    // im2col loads: BK x 128 floats, 2 passes of 8 rows
    const int b_vec = tid & 31;
    const int b_row = tid >> 5;
    const int b_k = k0 + b_vec * 4;
    const bool b_kok = b_k < p.K;
    int b_tap = 0, b_ci = 0, b_dy = 0, b_dx = 0;
    if (b_kok) {
        b_tap = b_k / p.Cin;
        b_ci = b_k - b_tap * p.Cin;
        if (p.ks == 3) { b_dy = b_tap / 3 - 1; b_dx = b_tap - (b_tap / 3) * 3 - 1; }
    }

    float4 ra[A_PASSES], rb[2];
    const long long npix = pend > pbeg ? (pend - pbeg) : 0;
    const int nk = (int)((npix + BK - 1) / BK);

    auto load_global = [&](int kc) {
        const long long pb = pbeg + (long long)kc * BK;
#pragma unroll
        for (int q = 0; q < A_PASSES; ++q) {
            long long pp = pb + a_row + q * A_ROWS_PER_PASS;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (a_cok && pp < pend) v = ldg4(p.dz + pp * p.lddz + a_co);
            ra[q] = v;
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            long long pp = pb + b_row + q * 8;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (b_kok && pp < pend) {
                int rem = (int)(pp % HW);
                int h = rem / p.W;
                int w = rem - h * p.W;
                int hh = h + b_dy, ww = w + b_dx;
                if (hh >= 0 && hh < p.H && ww >= 0 && ww < p.W)
                    v = ldg4(p.x + (pp + b_dy * p.W + b_dx) * p.ldx + b_ci);
            }
            rb[q] = v;
        }
    };
    auto store_smem = [&](int buf) {
#pragma unroll
        for (int q = 0; q < A_PASSES; ++q)
            *reinterpret_cast<float4*>(&As[buf][a_row + q * A_ROWS_PER_PASS][a_vec * 4]) = ra[q];
#pragma unroll
        for (int q = 0; q < 2; ++q) *reinterpret_cast<float4*>(&Bs[buf][b_row + q * 8][b_vec * 4]) = rb[q];
    };

    float acc[TM][8];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    if (nk > 0) {
        load_global(0);
        store_smem(0);
    }
    __syncthreads();
    int buf = 0;
    for (int kc = 0; kc < nk; ++kc) {
        if (kc + 1 < nk) load_global(kc + 1);
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[TM], b[8];
            if constexpr (TM == 8) {
                float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
                float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
                a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
                a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
            } else {
                float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
                a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
            }
            float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
            float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
            b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
            b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (kc + 1 < nk) store_smem(buf ^ 1);
        __syncthreads();
        buf ^= 1;
    }

    float* out = p.out + (long long)blockIdx.z * p.Cout * p.K;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        int co = co0 + ((i < 4) ? (ty * 4 + i) : (64 + ty * 4 + (i - 4)));
        if (co >= p.Cout) continue;
        float* orow = out + (long long)co * p.K;
#pragma unroll
        for (int j0 = 0; j0 < 8; j0 += 4) {
            int k = k0 + ((j0 == 0) ? tx * 4 : 64 + tx * 4);
            if (k < p.K)  // K % 4 == 0
                *reinterpret_cast<float4*>(orow + k) = make_float4(acc[i][j0], acc[i][j0 + 1], acc[i][j0 + 2], acc[i][j0 + 3]);
        }
    }
}

__global__ void splitk_reduce_kernel(const float4* __restrict__ ws, float4* __restrict__ out, long long n4, int splits) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float4 s = ws[i];
    for (int k = 1; k < splits; ++k) {
        float4 v = ws[(long long)k * n4 + i];
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    out[i] = s;
}

__global__ void weight_flip_transpose_kernel(const float* __restrict__ w, float* __restrict__ wt, int Cout, int kk, int Cin) {
    // wt[ci][kk-1-tap][co] = w[co][tap][ci]; 32x32 smem transpose per tap
    __shared__ float tile[32][33];
    int tap = blockIdx.z;
    int ci0 = blockIdx.x * 32, co0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int co = co0 + r, ci = ci0 + threadIdx.x;
        tile[r][threadIdx.x] = (co < Cout && ci < Cin) ? w[((long long)co * kk + tap) * Cin + ci] : 0.f;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int ci = ci0 + r, co = co0 + threadIdx.x;
        if (ci < Cin && co < Cout) wt[((long long)ci * kk + (kk - 1 - tap)) * Cout + co] = tile[threadIdx.x][r];
    }
}

__global__ void pad_channels_kernel(const float* __restrict__ in, int cin, float* __restrict__ out, int cout, size_t rows) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t n = rows * (size_t)cout;
    if (i >= n) return;
    size_t r = i / cout;
    int c = (int)(i - r * cout);
    out[i] = c < cin ? in[r * cin + c] : 0.f;
}

// ---------------------------------------------------------------------------
// First layer (3 or 3+1 input channels read straight from the reference-facing NCHW tensors, Cout <= 32, 3x3).
// HBM-bound: forward writes 128 B per pixel, the weight gradient reads them once.

// channel c of the (virtually concatenated) NCHW input pair, zero outside the image / beyond C0+C1
__device__ __forceinline__ float in_px(const float* __restrict__ in0, int C0, const float* __restrict__ in1, int C1, int b, int c,
                                       int h, int w, int H, int W) {
    if (h < 0 || h >= H || w < 0 || w >= W) return 0.f;
    if (c < C0) return __ldg(in0 + (((long long)b * C0 + c) * H + h) * W + w);
    if (c < C0 + C1) return __ldg(in1 + (((long long)b * C1 + (c - C0)) * H + h) * W + w);
    return 0.f;
}

// packed fp32 pairs: FFMA2 (fma.rn.f32x2) issues two IEEE fp32 FMAs per lane from one instruction slot, each half
// rounding exactly like fmaf()
typedef unsigned long long f32x2;
__device__ __forceinline__ void fma2(f32x2& acc, f32x2 a, f32x2 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b)); }
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float2 unpack2(f32x2 v) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
// pair arithmetic in two flavours (same rounding): packed FFMA2 or two scalar FFMAs
template <bool PACKED> struct Pair;
template <> struct Pair<true> {
    f32x2 v;
    __device__ __forceinline__ static Pair make(float lo, float hi) { Pair p; p.v = pack2(lo, hi); return p; }
    __device__ __forceinline__ static Pair raw(f32x2 bits) { Pair p; p.v = bits; return p; }
    __device__ __forceinline__ void fma(const Pair& a, const Pair& b) { fma2(v, a.v, b.v); }
    __device__ __forceinline__ float2 get() const { return unpack2(v); }
};
template <> struct Pair<false> {
    float2 v;
    __device__ __forceinline__ static Pair make(float lo, float hi) { Pair p; p.v = make_float2(lo, hi); return p; }
    __device__ __forceinline__ static Pair raw(f32x2 bits) { Pair p; p.v = unpack2(bits); return p; }
    __device__ __forceinline__ void fma(const Pair& a, const Pair& b) { v.x = fmaf(a.v.x, b.v.x, v.x); v.y = fmaf(a.v.y, b.v.y, v.y); }
    __device__ __forceinline__ float2 get() const { return v; }
};

__device__ __forceinline__ void cp_async4_zfill(void* smem_dst, const float* src, bool valid) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(src), "r"(valid ? 4 : 0) : "memory");
}
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const float* src, bool valid) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// forward: lane = output channel (its 9x(4*NQ) filter lives in registers as pairs), one warp walks along an image row
// keeping the 3x3 input window in registers (3*NQ broadcast shared-memory loads + 36*NQ FMAs per pixel, one coalesced
// 128-byte store).  The walk is unrolled by three so the window rotates by renaming, not by moves.  Persistent CTAs
// (two per SM) loop over tiles of FT_H rows (one per warp) x FT_W columns; the next tile's input is fetched with
// asynchronous copies into the other half of a double buffer while the current one is being computed.
// NQ = channel quads per pixel: 1 for <= 4 input channels (image + mask), 2 for 5..8 (image + cropped object [+ mask]).
constexpr int FT_H = 8, FT_W = 104, FT_NPX = (FT_H + 2) * (FT_W + 2);
template <bool PK> struct Px4 { Pair<PK> lo, hi; };   // one pixel: channels (0,1) and (2,3)
template <bool PK> __device__ __forceinline__ Px4<PK> lds_px(const float4* p) {
    const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p);
    Px4<PK> r; r.lo = Pair<PK>::raw(v.x); r.hi = Pair<PK>::raw(v.y);
    return r;
}
template <bool PK, int NQ> struct PxN { Px4<PK> q[NQ]; };   // one pixel: NQ channel quads
template <bool PK, int NQ> __device__ __forceinline__ PxN<PK, NQ> lds_pxn(const float4* p) {
    PxN<PK, NQ> r;
#pragma unroll
    for (int q = 0; q < NQ; ++q) r.q[q] = lds_px<PK>(p + q);
    return r;
}
// input tile bytes of the 8-channel forward (double buffered): above the 48 KB static limit, so dynamic shared memory
constexpr int first_fwd_smem_bytes(int nq) { return 2 * FT_NPX * nq * (int)sizeof(float4); }
// STATS: the BatchNorm partial row of this CTA (sum | sum of squares | min | max per channel, the layout
// fsdet_bn_finalize reads) is taken from the values while they are in registers - a thread owns ONE output channel, so
// there is nothing to transpose - instead of a separate pass over the 1.4 GB tensor (fsdet_colstats).
// (NQ = 1: two CTAs per SM at 122 registers; three at 80 registers measured slower: 1.12 vs 1.02 ms per step,
// tools/r2b_callE.sh.  NQ = 2 holds twice the weights and window: one CTA per SM, no spills.)
template <bool PK, bool STATS, int NQ>
__global__ void __launch_bounds__(256, NQ == 1 ? 2 : 1) conv_first_fwd_kernel(const float* __restrict__ in0, int C0,
                                                                const float* __restrict__ in1,
                                                                int C1, const float* __restrict__ w /* [Cout][9][4*NQ] */,
                                                                float* __restrict__ z, int ldz, int B, int H, int W, int Cout,
                                                                float* __restrict__ stats) {
    typedef float4 Tile[FT_NPX * NQ];                   // one buffer: [FT_NPX pixels][NQ quads]
    __shared__ float4 xs_static[NQ == 1 ? 2 : 1][NQ == 1 ? FT_NPX : 1];
    extern __shared__ __align__(16) float4 xs_dyn[];
    Tile* const xs = NQ == 1 ? reinterpret_cast<Tile*>(xs_static) : reinterpret_cast<Tile*>(xs_dyn);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tiles_w = (W + FT_W - 1) / FT_W, tiles_h = (H + FT_H - 1) / FT_H;
    const int tiles = B * tiles_h * tiles_w;
    const int HW = H * W;
    // input tile (+halo) of tile t, channel plane by channel plane, 4-byte async copies (zero fill outside the image)
    auto stage = [&](int t, int buf) {
        const int tw = t % tiles_w; t /= tiles_w;
        const int th = t % tiles_h;
        const int b = t / tiles_h;
        const int h0 = th * FT_H, w0 = tw * FT_W;
        // warp = tile row (two passes cover the FT_H + 2 rows), lane + 32 j = tile column
        bool cok_[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = lane + 32 * j, ww = w0 + c - 1;
            cok_[j] = c < FT_W + 2 && ww >= 0 && ww < W;
        }
        for (int r = warp; r < FT_H + 2; r += 8) {
            const int h = h0 + r - 1;
            const bool rok = h >= 0 && h < H;
            const unsigned dst = (unsigned)__cvta_generic_to_shared(&xs[buf][(r * (FT_W + 2) + lane) * NQ]);
            const long long off = (long long)(rok ? h : 0) * W + (w0 - 1 + lane);
#pragma unroll
            for (int ch = 0; ch < 4 * NQ; ++ch) {
                const float* plane = ch < C0 ? in0 + ((long long)b * C0 + ch) * HW
                                             : (ch < C0 + C1 ? in1 + ((long long)b * C1 + (ch - C0)) * HW : nullptr);
                const bool pok = rok && plane != nullptr;
                const float* src = pok ? plane + off : in0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (lane + 32 * j < FT_W + 2) {
                        const bool ok = pok && cok_[j];
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst + (32 * j * 4 * NQ + ch) * 4),
                                     "l"(ok ? src + 32 * j : in0), "r"(ok ? 4 : 0) : "memory");
                    }
                }
            }
        }
    };
    static_assert(NQ == 1 || NQ == 2, "up to 8 input channels");
    PxN<PK, NQ> wr[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const float4 v = lane < Cout ? ldg4(w + (lane * 9 + k) * 4 * NQ) : make_float4(0.f, 0.f, 0.f, 0.f);
        wr[k].q[0].lo = Pair<PK>::make(v.x, v.y); wr[k].q[0].hi = Pair<PK>::make(v.z, v.w);
        if (NQ == 2) {
            const float4 u = lane < Cout ? ldg4(w + (lane * 9 + k) * 4 * NQ + 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            wr[k].q[NQ - 1].lo = Pair<PK>::make(u.x, u.y); wr[k].q[NQ - 1].hi = Pair<PK>::make(u.z, u.w);
        }
    }
    const bool cok = lane < Cout;
    float tsum = 0.f, esum = 0.f, tsq = 0.f, esq = 0.f, tmn = INFINITY, tmx = -INFINITY;   // this thread's channel, all its pixels
    int buf = 0;
    if ((int)blockIdx.x < tiles) stage(blockIdx.x, 0);
    for (int t = blockIdx.x; t < tiles; t += gridDim.x, buf ^= 1) {
        cp_async_wait_all();
        __syncthreads();            // tile t has landed; everyone is done with the other buffer
        if (t + (int)gridDim.x < tiles) stage(t + gridDim.x, buf ^ 1);
        int tt = t;
        const int tw = tt % tiles_w; tt /= tiles_w;
        const int th = tt % tiles_h;
        const int b = tt / tiles_h;
        const int h = th * FT_H + warp, w0 = tw * FT_W;
        if (h >= H) continue;
        const int wn = min(FT_W, W - w0);
        const float4* r0 = &xs[buf][warp * (FT_W + 2) * NQ];
        const float4* r1 = r0 + (FT_W + 2) * NQ;
        const float4* r2 = r1 + (FT_W + 2) * NQ;
        float* zr = z + (((long long)b * H + h) * W + w0) * ldz + lane;
        // window columns: P = c, Q = c + 1, R = c + 2 (rows 0..2)
        PxN<PK, NQ> p0 = lds_pxn<PK, NQ>(r0), p1 = lds_pxn<PK, NQ>(r1), p2 = lds_pxn<PK, NQ>(r2);
        PxN<PK, NQ> q0 = lds_pxn<PK, NQ>(r0 + NQ), q1 = lds_pxn<PK, NQ>(r1 + NQ), q2 = lds_pxn<PK, NQ>(r2 + NQ);
        PxN<PK, NQ> s0, s1, s2;
#define FSDET_TAP(X, K)                                                                                   \
    alo.fma(X.q[0].lo, wr[K].q[0].lo); ahi.fma(X.q[0].hi, wr[K].q[0].hi);                                 \
    if (NQ == 2) { alo.fma(X.q[NQ - 1].lo, wr[K].q[NQ - 1].lo); ahi.fma(X.q[NQ - 1].hi, wr[K].q[NQ - 1].hi); }
#define FSDET_PIXEL(A0, A1, A2, B0, B1, B2, C0_, C1_, C2_, COL)                                           \
    {                                                                                                     \
        C0_ = lds_pxn<PK, NQ>(r0 + (COL) * NQ + 2 * NQ); C1_ = lds_pxn<PK, NQ>(r1 + (COL) * NQ + 2 * NQ);  \
        C2_ = lds_pxn<PK, NQ>(r2 + (COL) * NQ + 2 * NQ);                                                  \
        Pair<PK> alo = Pair<PK>::make(0.f, 0.f), ahi = alo;   /* one accumulator per channel of a quad */  \
        FSDET_TAP(A0, 0) FSDET_TAP(B0, 1) FSDET_TAP(C0_, 2)                                                \
        FSDET_TAP(A1, 3) FSDET_TAP(B1, 4) FSDET_TAP(C1_, 5)                                                \
        FSDET_TAP(A2, 6) FSDET_TAP(B2, 7) FSDET_TAP(C2_, 8)                                                \
        const float2 l = alo.get(), u = ahi.get();                                                        \
        const float v = (l.x + l.y) + (u.x + u.y);                                                        \
        if (cok) *zr = v;                                                                                 \
        if (STATS) { rs += v; rq = fmaf(v, v, rq); tmn = fminf(tmn, v); tmx = fmaxf(tmx, v); }            \
        zr += ldz;                                                                                        \
    }
        float rs = 0.f, rq = 0.f;     // this row run (<= FT_W pixels), folded into the compensated totals below
        int c = 0;
#pragma unroll 1
        for (; c + 3 <= wn; c += 3) {
            FSDET_PIXEL(p0, p1, p2, q0, q1, q2, s0, s1, s2, c)
            FSDET_PIXEL(q0, q1, q2, s0, s1, s2, p0, p1, p2, c + 1)
            FSDET_PIXEL(s0, s1, s2, p0, p1, p2, q0, q1, q2, c + 2)
        }
        if (c < wn) {
            FSDET_PIXEL(p0, p1, p2, q0, q1, q2, s0, s1, s2, c)
            if (c + 1 < wn) FSDET_PIXEL(q0, q1, q2, s0, s1, s2, p0, p1, p2, c + 1)
        }
#undef FSDET_PIXEL
#undef FSDET_TAP
        if (STATS) {
            float y = rs - esum, t2 = tsum + y;
            esum = (t2 - tsum) - y; tsum = t2;
            y = rq - esq; t2 = tsq + y;
            esq = (t2 - tsq) - y; tsq = t2;
        }
    }
    if (STATS) {
        __shared__ float4 red[8][32];
        __syncthreads();
        red[warp][lane] = make_float4(tsum - esum, tsq - esq, tmn, tmx);
        __syncthreads();
        if (warp == 0 && cok) {
            float4 tt = red[0][lane];
#pragma unroll
            for (int q = 1; q < 8; ++q) {
                const float4 o = red[q][lane];
                tt.x += o.x; tt.y += o.y; tt.z = fminf(tt.z, o.z); tt.w = fmaxf(tt.w, o.w);
            }
            float* dst = stats + (long long)blockIdx.x * 4 * Cout + lane;
            dst[0] = tt.x; dst[Cout] = tt.y; dst[2 * Cout] = tt.z; dst[3 * Cout] = tt.w;
        }
    }
}

// weight gradient: dw[co][tap][ci] = sum_p dz[p][co] * x[p+tap][ci].  One persistent CTA per SM walks a contiguous
// run of image rows.  The dz row is double buffered and the x rows live in a 6-slot ring in shared memory (one new
// x row per step, three at an image boundary); the next row is fetched with asynchronous copies while the current
// one is computed.  Thread (co, filter row ty, column segment) keeps the 3 taps of its filter row x 4 input channels
// in registers and slides a 3-pixel window along its segment of the image row (one new x pixel + one dz value per
// step feed 12 FMAs per channel quad); partials are reduced in a fixed order afterwards.  NQ = channel quads, as in the
// forward.
// column segments per row (thread groups): 6 for one channel quad; 5 for two, whose 15 warps leave each thread the
// 128 registers that its 24 accumulators and 3-pixel window need without spilling (18 warps allow 96)
template <int NQ> struct FirstWgrad {
    static constexpr int SEG = NQ == 1 ? 6 : 5;
    static constexpr int THREADS = 32 * 3 * SEG;
};
constexpr int first_wgrad_seg(int nq) { return nq == 1 ? FirstWgrad<1>::SEG : FirstWgrad<2>::SEG; }
constexpr int FW_SLOTS = 6;
// shared-memory bytes of the weight-gradient kernel: the x ring and the double-buffered dz row
constexpr size_t first_wgrad_smem_bytes(int nq, int W) {
    return ((size_t)FW_SLOTS * (W + 2) * 4 * nq + (size_t)2 * W * 32) * sizeof(float);
}
template <bool PK, int NQ>
__global__ void __launch_bounds__(FirstWgrad<NQ>::THREADS, 1) conv_first_wgrad_kernel(const float* __restrict__ in0, int C0,
                                                                         const float* __restrict__ in1, int C1,
                                                                         const float* __restrict__ dz, int lddz,
                                                                         float* __restrict__ part, int B, int H, int W, int Cout) {
    extern __shared__ __align__(16) float sm[];
    float4* xs = reinterpret_cast<float4*>(sm);              // [FW_SLOTS][W + 2] pixels of 4*NQ channels (zero halo)
    float* ds = sm + FW_SLOTS * (W + 2) * 4 * NQ;            // [2][W][32]
    const int tid = threadIdx.x;
    const int co = tid & 31;
    const int ty = (tid >> 5) % 3;                           // filter row
    constexpr int FW_SEG = FirstWgrad<NQ>::SEG, FW_THREADS = FirstWgrad<NQ>::THREADS;
    const int seg = (tid >> 5) / 3;                          // column segment 0..FW_SEG-1
    const int wseg = (W + FW_SEG - 1) / FW_SEG;
    const int wbeg = seg * wseg, wend = min(W, wbeg + wseg);
    const int HW = H * W;
    Pair<PK> acc[3][2 * NQ];                                 // taps (ty, 0..2) x channel pairs
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int q = 0; q < 2 * NQ; ++q) acc[i][q] = Pair<PK>::make(0.f, 0.f);
    const long long rows = (long long)B * H;
    const long long per = (rows + gridDim.x - 1) / gridDim.x;
    const long long rbeg = (long long)blockIdx.x * per, rend = min(rows, rbeg + per);
    // ring state of the most recently staged row: x rows have_h-1 .. have_h+1 of image have_b sit in slots win..win+2
    int have_b = -1, have_h = -2, win = 0;
    auto stage = [&](long long row, int buf) {
        const int b = (int)(row / H), h = (int)(row - (long long)b * H);
        const bool step = (b == have_b && h == have_h + 1);
        const int nnew = step ? 1 : 3;
        win = (win + nnew) % FW_SLOTS;                       // step: window slides by one; else a fresh window
        for (int c = tid; c < W + 2; c += FW_THREADS) {      // x rows: thread = column (one pass unless W + 2 > FW_THREADS)
            const bool cok_ = c >= 1 && c <= W;
            for (int k = 3 - nnew; k < 3; ++k) {
                const int q = h - 1 + k;
                const unsigned dst = (unsigned)__cvta_generic_to_shared(xs + ((win + k) % FW_SLOTS) * (W + 2) * NQ + c * NQ);
                const bool ok = cok_ && q >= 0 && q < H;
                const long long off = (long long)(ok ? q : 0) * W + (c - 1);
#pragma unroll
                for (int ch = 0; ch < 4 * NQ; ++ch) {
                    const float* plane = ch < C0 ? in0 + ((long long)b * C0 + ch) * HW
                                                 : (ch < C0 + C1 ? in1 + ((long long)b * C1 + (ch - C0)) * HW : nullptr);
                    const bool okc = ok && plane != nullptr;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst + ch * 4), "l"(okc ? plane + off : in0),
                                 "r"(okc ? 4 : 0) : "memory");
                }
            }
        }
        have_b = b; have_h = h;
        // dz row: FW_THREADS is a multiple of 8, so a thread keeps its channel quad and strides over pixels
        {
            const int c4 = (tid & 7) * 4, pstep = FW_THREADS / 8;
            const bool ok = c4 < Cout;
            const float* src = dz + (row * W + (tid >> 3)) * lddz + c4;
            unsigned dst = (unsigned)__cvta_generic_to_shared(ds + buf * W * 32 + tid * 4);
            const long long sstep = (long long)pstep * lddz;
            for (int pw = tid >> 3; pw < W; pw += pstep, src += sstep, dst += FW_THREADS * 16)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(ok ? src : dz), "r"(ok ? 16 : 0) : "memory");
        }
    };
    if (rbeg < rend) stage(rbeg, 0);
    int buf = 0;
    for (long long row = rbeg; row < rend; ++row, buf ^= 1) {
        cp_async_wait_all();
        __syncthreads();            // this row has landed; everyone is done with the previous one
        const int wcur = win;
        if (row + 1 < rend) stage(row + 1, buf ^ 1);
        const float4* xr = xs + ((wcur + ty) % FW_SLOTS) * (W + 2) * NQ;   // image row h + ty - 1;  xr[(w + tx) NQ] = x[.][w + tx - 1]
        const float* dcur = ds + buf * W * 32 + co;
        if (wbeg < wend) {
            PxN<PK, NQ> x0 = lds_pxn<PK, NQ>(xr + wbeg * NQ), x1 = lds_pxn<PK, NQ>(xr + wbeg * NQ + NQ), x2;
#define FSDET_MAC(I, X)                                                                          \
    acc[I][0].fma(dd, X.q[0].lo); acc[I][1].fma(dd, X.q[0].hi);                                  \
    if (NQ == 2) { acc[I][2 * NQ - 2].fma(dd, X.q[NQ - 1].lo); acc[I][2 * NQ - 1].fma(dd, X.q[NQ - 1].hi); }
#define FSDET_STEP(X0, X1, X2, WW)                                                               \
    {                                                                                            \
        X2 = lds_pxn<PK, NQ>(xr + (WW) * NQ + 2 * NQ);                                           \
        const float d = dcur[(WW) * 32];                                                         \
        const Pair<PK> dd = Pair<PK>::make(d, d);                                                \
        FSDET_MAC(0, X0) FSDET_MAC(1, X1) FSDET_MAC(2, X2)                                       \
    }
            int w = wbeg;
#pragma unroll 1
            for (; w + 3 <= wend; w += 3) {
                FSDET_STEP(x0, x1, x2, w)
                FSDET_STEP(x1, x2, x0, w + 1)
                FSDET_STEP(x2, x0, x1, w + 2)
            }
            if (w < wend) {
                FSDET_STEP(x0, x1, x2, w)
                if (w + 1 < wend) FSDET_STEP(x1, x2, x0, w + 1)
            }
#undef FSDET_STEP
#undef FSDET_MAC
        }
    }
    if (co < Cout) {
        float* dst = part + (((long long)blockIdx.x * FW_SEG + seg) * Cout + co) * 36 * NQ + ty * 12 * NQ;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                const float2 l = acc[i][2 * q].get(), u = acc[i][2 * q + 1].get();
                *reinterpret_cast<float4*>(dst + 4 * (i * NQ + q)) = make_float4(l.x, l.y, u.x, u.y);
            }
    }
}

// fixed-order reduction of the first-layer partials: one CTA per float4 of dw, threads stride over the partials,
// then a shared-memory tree
__global__ void __launch_bounds__(128) first_wgrad_reduce_kernel(const float4* __restrict__ ws, float4* __restrict__ out, int n4,
                                                                 int parts) {
    __shared__ float4 red[128];
    const int i = blockIdx.x;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = threadIdx.x; k < parts; k += 128) {
        const float4 v = ws[(long long)k * n4 + i];
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            const float4 a = red[threadIdx.x], b = red[threadIdx.x + o];
            red[threadIdx.x] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[i] = red[0];
}

static int wgrad_splits(long long M, int Cin, int Cout, int ks, int bmc) {
    int K = ks * ks * Cin;
    long long tiles = (long long)ceil_div(K, 128) * ceil_div(Cout, bmc);
    long long want = (2LL * kNumSMs + tiles - 1) / tiles;
    long long maxs = (M + 255) / 256;  // at least 256 pixels per split
    if (want > maxs) want = maxs;
    if (want < 1) want = 1;
    if (want > 1024) want = 1024;
    return (int)want;
}

}  // namespace fsdet

using namespace fsdet;

extern "C" int fsdet_conv_stat_rows(int npix) { return ceil_div(npix, BM); }

extern "C" int fsdet_conv_fwd(const float* x, int ldx, const float* w, const float* bias, float* z, int ldz,
                              float* stat_partial, int B, int H, int W, int Cin, int Cout, int ksize, int accumulate,
                              void* stream) {
    FSDET_CHECK_ARG(x && w && z, "conv_fwd: null pointer");
    FSDET_CHECK_ARG(ksize == 1 || ksize == 3, "conv_fwd: ksize %d unsupported (1 or 3)", ksize);
    FSDET_CHECK_ARG(Cin > 0 && Cin % 4 == 0 && ldx % 4 == 0 && ldx >= Cin, "conv_fwd: Cin=%d ldx=%d must be multiples of 4", Cin, ldx);
    FSDET_CHECK_ARG(Cout > 0 && ldz >= Cout, "conv_fwd: Cout=%d ldz=%d", Cout, ldz);
    FSDET_CHECK_ARG(aligned16(x) && aligned16(w), "conv_fwd: x/w must be 16-byte aligned");
    FSDET_CHECK_ARG(!(stat_partial && (bias || accumulate)), "conv_fwd: stats are only defined for the plain product");
    ConvArgs a;
    a.x = x; a.w = w; a.bias = bias; a.z = z; a.stat = stat_partial;
    a.ldx = ldx; a.ldz = ldz; a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.ks = ksize; a.pad = (ksize - 1) / 2;
    a.K = ksize * ksize * Cin; a.M = (long long)B * H * W; a.accumulate = accumulate;
    if (a.M == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    dim3 block(256);
    if (Cout > 64) {
        dim3 grid(ceil_div(a.M, BM), ceil_div(Cout, 128));
        conv_igemm_kernel<8><<<grid, block, 0, s>>>(a);
    } else if (Cout > 32) {
        dim3 grid(ceil_div(a.M, BM), 1);
        conv_igemm_kernel<4><<<grid, block, 0, s>>>(a);
    } else {
        dim3 grid(ceil_div(a.M, BM), 1);
        conv_igemm_kernel<2><<<grid, block, 0, s>>>(a);
    }
    return launch_status("conv_fwd");
}

extern "C" size_t fsdet_conv_wgrad_workspace_floats(int B, int H, int W, int Cin, int Cout, int ksize) {
    long long M = (long long)B * H * W;
    int bmc = Cout > 64 ? 128 : 64;
    int splits = wgrad_splits(M, Cin, Cout, ksize, bmc);
    if (splits <= 1) return 0;
    return (size_t)splits * (size_t)Cout * (size_t)(ksize * ksize * Cin);
}

extern "C" int fsdet_conv_wgrad(const float* x, int ldx, const float* dz, int lddz, float* dw, float* workspace,
                                size_t workspace_floats, int B, int H, int W, int Cin, int Cout, int ksize, void* stream) {
    FSDET_CHECK_ARG(x && dz && dw, "conv_wgrad: null pointer");
    FSDET_CHECK_ARG(ksize == 1 || ksize == 3, "conv_wgrad: ksize %d unsupported", ksize);
    FSDET_CHECK_ARG(Cin % 4 == 0 && Cout % 4 == 0 && ldx % 4 == 0 && lddz % 4 == 0,
                    "conv_wgrad: Cin=%d Cout=%d ldx=%d lddz=%d must be multiples of 4", Cin, Cout, ldx, lddz);
    FSDET_CHECK_ARG(aligned16(x) && aligned16(dz) && aligned16(dw), "conv_wgrad: pointers must be 16-byte aligned");
    WgradArgs a;
    a.x = x; a.dz = dz; a.ldx = ldx; a.lddz = lddz; a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout;
    a.ks = ksize; a.pad = (ksize - 1) / 2; a.K = ksize * ksize * Cin; a.M = (long long)B * H * W;
    int bmc = Cout > 64 ? 128 : 64;
    int splits = wgrad_splits(a.M, Cin, Cout, ksize, bmc);
    size_t need = splits > 1 ? (size_t)splits * Cout * a.K : 0;
    FSDET_CHECK_ARG(workspace_floats >= need && (need == 0 || (workspace && aligned16(workspace))),
                    "conv_wgrad: workspace too small (%zu < %zu floats)", workspace_floats, need);
    long long pps = (a.M + splits - 1) / splits;
    pps = (pps + BK - 1) / BK * BK;
    a.pix_per_split = pps;
    a.out = splits > 1 ? workspace : dw;
    cudaStream_t s = (cudaStream_t)stream;
    dim3 grid(ceil_div(a.K, 128), ceil_div(Cout, bmc), splits);
    if (bmc == 128) conv_wgrad_kernel<128><<<grid, 256, 0, s>>>(a);
    else conv_wgrad_kernel<64><<<grid, 256, 0, s>>>(a);
    int st = launch_status("conv_wgrad");
    if (st) return st;
    if (splits > 1) {
        long long n4 = (long long)Cout * a.K / 4;
        splitk_reduce_kernel<<<ceil_div(n4, 256), 256, 0, s>>>(reinterpret_cast<const float4*>(workspace),
                                                              reinterpret_cast<float4*>(dw), n4, splits);
        st = launch_status("conv_wgrad_reduce");
    }
    return st;
}

extern "C" int fsdet_weight_flip_transpose(const float* w, float* wt, int Cout, int kk, int Cin, void* stream) {
    FSDET_CHECK_ARG(w && wt && Cout > 0 && Cin > 0 && kk > 0, "weight_flip_transpose: bad args");
    dim3 grid(ceil_div(Cin, 32), ceil_div(Cout, 32), kk), block(32, 8);
    weight_flip_transpose_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(w, wt, Cout, kk, Cin);
    return launch_status("weight_flip_transpose");
}

extern "C" int fsdet_pad_channels(const float* in, int cin, float* out, int cout, size_t rows, void* stream) {
    FSDET_CHECK_ARG(in && out && cin > 0 && cout > 0, "pad_channels: bad args");
    size_t n = rows * (size_t)cout;
    if (n == 0) return 0;
    pad_channels_kernel<<<ceil_div((long long)n, 256), 256, 0, (cudaStream_t)stream>>>(in, cin, out, cout, rows);
    return launch_status("pad_channels");
}

static int first_wgrad_ctas(int B, int H) {
    long long rows = (long long)B * H;
    long long n = kNumSMs;
    return (int)(rows < n ? rows : n);
}

static int first_quads(int C) { return C <= 4 ? 1 : 2; }   // weight / dw channel pitch 4 * quads

extern "C" size_t fsdet_conv_first_wgrad_workspace_floats(int B, int H, int W, int Cout) {
    return fsdet_conv_first_wgrad_workspace_floats_cin(B, H, W, 4, Cout);
}

extern "C" size_t fsdet_conv_first_wgrad_workspace_floats_cin(int B, int H, int W, int Cin, int Cout) {
    (void)W;
    const int nq = first_quads(Cin);
    return (size_t)first_wgrad_ctas(B, H) * first_wgrad_seg(nq) * Cout * 36 * nq;
}

extern "C" int fsdet_conv_first_wgrad_supported(int Cin, int W) {
    return Cin >= 1 && Cin <= 8 && W > 0 && first_wgrad_smem_bytes(first_quads(Cin), W) <= 227 * 1024;
}

template <bool STATS, int NQ>
static int launch_first_fwd(const float* in0, int C0, const float* in1, int C1, const float* w, float* z, int ldz, int B, int H,
                            int W, int Cout, float* stats, unsigned ctas, cudaStream_t s) {
    // packed FFMA2 flavour: fewer issue slots per pixel (measured 705 us vs 750 us at B=64, 416x416, 4 channels)
    auto kern = conv_first_fwd_kernel<true, STATS, NQ>;
    const int smem = NQ == 1 ? 0 : first_fwd_smem_bytes(NQ);
    if (NQ > 1) {   // dynamic shared-memory opt-in per launch, as conv_first_wgrad
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) { set_error("conv_first_fwd: %s", cudaGetErrorString(e)); return (int)e; }
    }
    kern<<<ctas, 256, smem, s>>>(in0, C0, in1, C1, w, z, ldz, B, H, W, Cout, stats);
    return 0;
}

extern "C" int fsdet_conv_first_fwd(const float* in0, int C0, const float* in1, int C1, const float* w_pad, float* z, int ldz,
                                    int B, int H, int W, int Cout, void* stream) {
    FSDET_CHECK_ARG(in0 && w_pad && z && C0 > 0 && C1 >= 0 && (C1 == 0 || in1) && C0 + C1 <= 8, "conv_first_fwd: bad inputs");
    FSDET_CHECK_ARG(Cout > 0 && Cout <= 32 && Cout % 4 == 0 && ldz % 4 == 0 && aligned16(z) && aligned16(w_pad),
                    "conv_first_fwd: Cout=%d ldz=%d", Cout, ldz);
    long long tiles = (long long)B * ceil_div(H, FT_H) * ceil_div(W, FT_W);
    if (tiles == 0) return 0;
    FSDET_CHECK_ARG(tiles < (1ll << 31), "conv_first_fwd: too many tiles");
    const unsigned ctas = (unsigned)(tiles < 2LL * kNumSMs ? tiles : 2LL * kNumSMs);
    const int e = first_quads(C0 + C1) == 1
        ? launch_first_fwd<false, 1>(in0, C0, in1, C1, w_pad, z, ldz, B, H, W, Cout, nullptr, ctas, (cudaStream_t)stream)
        : launch_first_fwd<false, 2>(in0, C0, in1, C1, w_pad, z, ldz, B, H, W, Cout, nullptr, ctas, (cudaStream_t)stream);
    if (e) return e;
    return launch_status("conv_first_fwd");
}

extern "C" int fsdet_conv_first_stat_rows(int B, int H, int W) {
    long long tiles = (long long)B * ceil_div(H, FT_H) * ceil_div(W, FT_W);
    return (int)(tiles < 2LL * kNumSMs ? tiles : 2LL * kNumSMs);
}

extern "C" int fsdet_conv_first_fwd_stats(const float* in0, int C0, const float* in1, int C1, const float* w_pad, float* z, int ldz,
                                          int B, int H, int W, int Cout, float* stat_partial, void* stream) {
    FSDET_CHECK_ARG(in0 && w_pad && z && stat_partial && C0 > 0 && C1 >= 0 && (C1 == 0 || in1) && C0 + C1 <= 8,
                    "conv_first_fwd_stats: bad inputs");
    FSDET_CHECK_ARG(Cout > 0 && Cout <= 32 && Cout % 4 == 0 && ldz % 4 == 0 && aligned16(z) && aligned16(w_pad),
                    "conv_first_fwd_stats: Cout=%d ldz=%d", Cout, ldz);
    long long tiles = (long long)B * ceil_div(H, FT_H) * ceil_div(W, FT_W);
    if (tiles == 0) return 0;
    FSDET_CHECK_ARG(tiles < (1ll << 31), "conv_first_fwd_stats: too many tiles");
    const unsigned ctas = (unsigned)fsdet_conv_first_stat_rows(B, H, W);
    const int e = first_quads(C0 + C1) == 1
        ? launch_first_fwd<true, 1>(in0, C0, in1, C1, w_pad, z, ldz, B, H, W, Cout, stat_partial, ctas, (cudaStream_t)stream)
        : launch_first_fwd<true, 2>(in0, C0, in1, C1, w_pad, z, ldz, B, H, W, Cout, stat_partial, ctas, (cudaStream_t)stream);
    if (e) return e;
    return launch_status("conv_first_fwd_stats");
}

template <int NQ>
static int launch_first_wgrad(const float* in0, int C0, const float* in1, int C1, const float* dz, int lddz, float* ws, int B,
                              int H, int W, int Cout, int ctas, cudaStream_t s) {
    auto kern = conv_first_wgrad_kernel<false, NQ>;
    {   // the opt-in ceiling (227 KB), per launch like every other kernel of the library: no cached state, and never lowered under
        // a graph that was captured at a wider image
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) { set_error("conv_first_wgrad: %s", cudaGetErrorString(e)); return (int)e; }
    }
    // scalar FFMA flavour (the packed one is register-bandwidth bound here: 900 us vs 873 us)
    kern<<<ctas, FirstWgrad<NQ>::THREADS, first_wgrad_smem_bytes(NQ, W), s>>>(in0, C0, in1, C1, dz, lddz, ws, B, H, W, Cout);
    return 0;
}

extern "C" int fsdet_conv_first_wgrad(const float* in0, int C0, const float* in1, int C1, const float* dz, int lddz, float* dw,
                                      float* workspace, size_t workspace_floats, int B, int H, int W, int Cout, void* stream) {
    FSDET_CHECK_ARG(in0 && dz && dw && workspace && C0 > 0 && C1 >= 0 && (C1 == 0 || in1) && C0 + C1 <= 8,
                    "conv_first_wgrad: bad inputs");
    FSDET_CHECK_ARG(Cout > 0 && Cout <= 32 && Cout % 4 == 0 && lddz % 4 == 0, "conv_first_wgrad: Cout=%d lddz=%d", Cout, lddz);
    FSDET_CHECK_ARG(aligned16(dz) && aligned16(dw) && aligned16(workspace), "conv_first_wgrad: alignment");
    const int nq = first_quads(C0 + C1);
    const int ctas = first_wgrad_ctas(B, H);
    FSDET_CHECK_ARG(workspace_floats >= fsdet_conv_first_wgrad_workspace_floats_cin(B, H, W, C0 + C1, Cout),
                    "conv_first_wgrad: workspace too small");
    if (ctas == 0) return 0;
    FSDET_CHECK_ARG(fsdet_conv_first_wgrad_supported(C0 + C1, W), "conv_first_wgrad: image width %d too large for %d channels", W,
                    C0 + C1);
    cudaStream_t s = (cudaStream_t)stream;
    int st = nq == 1 ? launch_first_wgrad<1>(in0, C0, in1, C1, dz, lddz, workspace, B, H, W, Cout, ctas, s)
                     : launch_first_wgrad<2>(in0, C0, in1, C1, dz, lddz, workspace, B, H, W, Cout, ctas, s);
    if (st) return st;
    st = launch_status("conv_first_wgrad");
    if (st) return st;
    long long n4 = (long long)Cout * 9 * nq;
    first_wgrad_reduce_kernel<<<(unsigned)n4, 128, 0, s>>>(reinterpret_cast<const float4*>(workspace), reinterpret_cast<float4*>(dw),
                                                           (int)n4, ctas * first_wgrad_seg(nq));
    return launch_status("conv_first_wgrad_reduce");
}
