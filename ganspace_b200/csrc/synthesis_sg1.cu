// StyleGAN (v1) synthesis network: G_synthesis up to a stop point, or the whole image.
//
// Replaces models/stylegan/model.py:51-104 (MyConv2d, incl. the fused 4x4 transposed conv of :82-91), :106-122 (NoiseLayer),
// :124-136 (StyleMod), :145-169 (BlurLayer), :171-188 (Upscale2d), :230-303 (LayerEpilogue, InputBlock, GSynthesisBlock) and
// :305-363 (G_synthesis), as driven by models/wrappers.py:368-417.
//
// The chain is a list of layers; layer j reads latent j (block i = layers 2i, 2i+1).  Per layer, on NHWC activations:
//   conv     Y[b,p,tap,co] = sum_ci x[b,p,ci] Wt[tap,co,ci]      the tap GEMM (tc_gemm_plain: tcgen05, fp16 hi/lo split
//                                                                operands, 3 MMAs per product = fp32 grade), weights shared
//                                                                by all samples and pre-scaled by w_mul
//            same      out[y,x] = sum_{ky,kx} Y[(y+ky-1, x+kx-1), (ky,kx)]                                 (3x3, pad 1)
//            nearest   out[y,x] = sum_{ky,kx} Y[(floor((y+ky-1)/2), floor((x+kx-1)/2)), (ky,kx)]          (x2 upscale, 3x3;
//                      the upscaled image is never formed: the GEMM runs on the low-resolution rows)
//            fused     out[u,v] = sum_{ky,kx: u+1-ky, v+1-kx even} Y[((u+1-ky)/2, (v+1-kx)/2), (ky,kx)]    (4x4 taps of the
//                      reference's 4-way summed kernel, stride 2, pad 1; blocks >= 128^2)
//   epilogue [1,2,1]x[1,2,1]/16 blur, pad 1 (up-sampling layers) + bias  (= the conv module's output, a stop point)
//            + noise_w[c] * noise[y,x]; leaky_relu 0.2 (no gain)  -> pre-norm activation P (fp32)
//   stats    per (sample, channel) mean and biased variance of P, two passes in fp64 with a fixed reduction order (no atomics:
//            partial_forward and forward give bit-identical activations)
//   norm     (P - mean) * rsqrt(var + 1e-5) * (s0 + 1) + s1,  s = style_mod.lin(w)   -> the next GEMM's fp16 hi/lo operand, or
//            fp32 NHWC rows with a caller-given row stride at the stop point (straight into the large-d IPCA matrix)
// The 4x4 block's first layer starts from const + bias.  torgb (1x1 conv, gain 1, + bias) follows the last layer.
// The per-tap form has a float64 host restatement that tests pin to the reference's form.
#include "common.cuh"
#include <cuda_fp16.h>
#include <math.h>

namespace gsb {

int tc_gemm_plain(const __half *a_hi, const __half *a_lo, int64_t M, int K, const __half *w_hi, const __half *w_lo, int N,
                  const float *inv_wscale, float *out, unsigned *overflow, int leave_free_sms, cudaStream_t st);

namespace sg1 {

constexpr int MAX_LAYERS = 18;
constexpr int CHUNK_ROWS = 4096;      // GEMM rows per launch (whole samples): 4096 x 9*512 fp32 tap planes = 75 MB, L2-resident
enum Kind { CONST = 0, SAME = 1, NEAREST = 2, FUSED = 3 };
enum Stop { STOP_EPI = 0, STOP_CONV = 1, STOP_STYLE = 2, STOP_IMAGE = 3 };

static int taps_of(int kind) { return kind == FUSED ? 16 : 9; }
static int npad_of(const gsb_sg1_layer &l) { return (taps_of(l.kind) * l.cout + 31) / 32 * 32; }
static int res_in_of(const gsb_sg1_layer &l) { return (l.kind == NEAREST || l.kind == FUSED) ? l.res_out / 2 : l.res_out; }

struct LayerView {
    __half *w_hi, *w_lo;      // [npad, cin]  row = tap * cout + co (rows past taps*cout are zero)
    float *scal;              // inv_wscale, wscale, absmax
    float *cst;               // CONST: [16, c] NHWC
    float *bias, *noise_w;    // [cout]
    float *noise;             // [res_out^2]
    float *style_w;           // [2 cout, dlatent] times 1/sqrt(dlatent)
    float *style_b;           // [2 cout]
};
struct View {
    LayerView L[MAX_LAYERS];
    float *rgb_w;             // [3, c_last] times 1/sqrt(c_last)
    float *rgb_b;             // [3]
    unsigned *overflow;
    size_t bytes;
};

static View view(void *base, const gsb_sg1_layer *layers, int n_layers, int dlatent) {
    View v;
    char *p = reinterpret_cast<char *>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { char *q = p + off; off += align_up(bytes, 256); return q; };
    v.overflow = (unsigned *)take(256);
    for (int l = 0; l < n_layers; ++l) {
        const gsb_sg1_layer &c = layers[l];
        LayerView &L = v.L[l];
        L.w_hi = L.w_lo = nullptr; L.cst = nullptr; L.scal = nullptr;
        if (c.kind == CONST) {
            L.cst = (float *)take((size_t)16 * c.cout * 4);
        } else {
            L.w_hi = (__half *)take((size_t)npad_of(c) * c.cin * 2);
            L.w_lo = (__half *)take((size_t)npad_of(c) * c.cin * 2);
            L.scal = (float *)take(16);
        }
        L.bias = (float *)take((size_t)c.cout * 4);
        L.noise_w = (float *)take((size_t)c.cout * 4);
        L.noise = (float *)take((size_t)c.res_out * c.res_out * 4);
        L.style_w = (float *)take((size_t)2 * c.cout * dlatent * 4);
        L.style_b = (float *)take((size_t)2 * c.cout * 4);
    }
    v.rgb_w = (float *)take((size_t)3 * (n_layers ? layers[n_layers - 1].cout : 0) * 4);
    v.rgb_b = (float *)take(16);
    v.bytes = off;
    return v;
}

static int check(const gsb_sg1_layer *layers, int n_layers, int dlatent) {
    GSB_CHECK_ARG(layers && n_layers >= 2 && n_layers <= MAX_LAYERS && n_layers % 2 == 0, "sg1: need 2..%d layers (pairs)", MAX_LAYERS);
    GSB_CHECK_ARG(dlatent > 0 && dlatent % 4 == 0, "sg1: dlatent %% 4");
    for (int l = 0; l < n_layers; ++l) {
        const gsb_sg1_layer &c = layers[l];
        GSB_CHECK_ARG(c.kind >= CONST && c.kind <= FUSED, "sg1: layer %d bad kind", l);
        GSB_CHECK_ARG(c.cout >= 16 && c.cout % 16 == 0 && c.cin >= 16 && c.cin % 16 == 0, "sg1: layer %d needs cin, cout %% 16 (cin=%d cout=%d)",
                      l, c.cin, c.cout);
        GSB_CHECK_ARG(c.res_out >= 4 && c.res_out <= 1024, "sg1: layer %d bad res_out", l);
        if (l == 0) GSB_CHECK_ARG(c.kind == CONST && c.res_out == 4 && c.cin == c.cout, "sg1: layer 0 is the 4x4 constant");
        else {
            GSB_CHECK_ARG(c.kind != CONST, "sg1: only layer 0 starts from the constant");
            GSB_CHECK_ARG(c.cin == layers[l - 1].cout && res_in_of(c) == layers[l - 1].res_out, "sg1: layer %d does not chain", l);
            GSB_CHECK_ARG((l % 2 == 1) == (c.kind == SAME), "sg1: layer %d: the second layer of a block is the 3x3 conv", l);
        }
    }
    return GSB_OK;
}

// ---- pack ------------------------------------------------------------------------------------------------
// tap value (times w_mul) of the conv: 3x3 taps (ky*3+kx) or, for FUSED, the 4x4 taps of model.py:85-89 in its summation order
__device__ __forceinline__ float tap_value(const float *__restrict__ W, int kind, int co, int ci, int cin, int tap, float wmul) {
    const float *w = W + ((int64_t)co * cin + ci) * 9;
    if (kind != FUSED) return w[tap] * wmul;
    const int ky = tap >> 2, kx = tap & 3;
    // wp = pad(w, 1) (5x5); w4[ky][kx] = wp[ky+1][kx+1] + wp[ky][kx+1] + wp[ky+1][kx] + wp[ky][kx]
    auto wp = [&](int a, int b) { return (a >= 1 && a <= 3 && b >= 1 && b <= 3) ? w[(a - 1) * 3 + (b - 1)] * wmul : 0.f; };
    return ((wp(ky + 1, kx + 1) + wp(ky, kx + 1)) + wp(ky + 1, kx)) + wp(ky, kx);
}

__global__ void absmax_kernel(const float *__restrict__ W, int kind, int cout, int cin, float wmul, float *__restrict__ out) {
    const int taps = kind == FUSED ? 16 : 9;
    const int64_t total = (int64_t)taps * cout * cin;
    float m = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int ci = (int)(i % cin);
        const int64_t r = i / cin;
        m = fmaxf(m, fabsf(tap_value(W, kind, (int)(r % cout), ci, cin, (int)(r / cout), wmul)));
    }
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int *>(out), __float_as_int(m));     // max of non-negatives: exact
}
// scal[2] = absmax -> scal[1] = 2^s, scal[0] = 2^-s with the largest |w 2^s| in [8192, 16384)
__global__ void pick_scale_kernel(float *__restrict__ scal) {
    float m = scal[2];
    if (!(m > 0.f)) m = 1.f;
    int e = 0;
    frexpf(m, &e);
    scal[1] = ldexpf(1.f, 14 - e);
    scal[0] = ldexpf(1.f, e - 14);
}
__global__ void weight_pack_kernel(const float *__restrict__ W, int kind, int cout, int cin, float wmul, const float *__restrict__ scal,
                                   __half *__restrict__ hi, __half *__restrict__ lo) {
    const int taps = kind == FUSED ? 16 : 9;
    const int64_t total = (int64_t)taps * cout * cin;
    const float ws = scal[1];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int ci = (int)(i % cin);
        const int64_t r = i / cin;                                 // r = tap * cout + co
        const float w = tap_value(W, kind, (int)(r % cout), ci, cin, (int)(r / cout), wmul) * ws;
        const __half h = __float2half_rn(w);
        hi[i] = h;
        lo[i] = __float2half_rn(w - __half2float(h));
    }
}
__global__ void scale_copy_kernel(const float *__restrict__ src, int64_t count, float scale, float *__restrict__ dst) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = src[i] * scale;
}
// const[c, 4, 4] -> [16, c]
__global__ void const_nhwc_kernel(const float *__restrict__ src, int c, float *__restrict__ dst) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < 16 * c) { const int p = idx / c, ch = idx % c; dst[idx] = src[ch * 16 + p]; }
}

// ---- forward kernels ------------------------------------------------------------------------------------
// y[r, j] = sum_k x[r, k] w[j, k] + b[j]   (StyleMod.lin, torgb-sized products: one thread per output, fixed order)
__global__ void small_linear_kernel(const float *__restrict__ x, int64_t ldx, const float *__restrict__ w, const float *__restrict__ b,
                                    float *__restrict__ y, int64_t ldy, int64_t n, int N, int K) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= n * N) return;
    const int j = (int)(idx % N);
    const int64_t r = idx / N;
    const float *xr = x + r * ldx, *wr = w + (int64_t)j * K;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int k = 0; k < K; k += 4) {
        const float4 xv = *reinterpret_cast<const float4 *>(xr + k), wv = *reinterpret_cast<const float4 *>(wr + k);
        a0 = fmaf(xv.x, wv.x, a0); a1 = fmaf(xv.y, wv.y, a1); a2 = fmaf(xv.z, wv.z, a2); a3 = fmaf(xv.w, wv.w, a3);
    }
    y[r * ldy + j] = (a0 + a1) + (a2 + a3) + b[j];
}

// conv output (no bias) of nb samples from the tap planes Y [nb * Hin^2, npad]; out [nb, R, R, cout]
template <int KIND>
__global__ void __launch_bounds__(256)
gather_kernel(const float *__restrict__ Y, int64_t nb, int Hin, int R, int cout, int npad, float *__restrict__ out) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= nb * R * R * cout) return;
    const int co = (int)(idx % cout);
    const int64_t pg = idx / cout;
    const int x = (int)(pg % R), y = (int)((pg / R) % R);
    const int64_t b = pg / ((int64_t)R * R);
    const float *Yb = Y + b * Hin * Hin * (int64_t)npad + co;
    float acc = 0.f;
    if (KIND == FUSED) {
#pragma unroll
        for (int ky = 0; ky < 4; ++ky) {
            const int t = y + 1 - ky;
            if (t < 0 || (t & 1) || (t >> 1) >= Hin) continue;
#pragma unroll
            for (int kx = 0; kx < 4; ++kx) {
                const int s = x + 1 - kx;
                if (s < 0 || (s & 1) || (s >> 1) >= Hin) continue;
                acc += Yb[((int64_t)(t >> 1) * Hin + (s >> 1)) * npad + (ky * 4 + kx) * cout];
            }
        }
    } else {
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const int t = y + ky - 1;
            if (t < 0 || t >= R) continue;
            const int yy = KIND == NEAREST ? (t >> 1) : t;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int s = x + kx - 1;
                if (s < 0 || s >= R) continue;
                const int xx = KIND == NEAREST ? (s >> 1) : s;
                acc += Yb[((int64_t)yy * Hin + xx) * npad + (ky * 3 + kx) * cout];
            }
        }
    }
    out[idx] = acc;
}

// (blur) + bias -> [conv module output] -> + noise_w[c] noise[p] -> leaky_relu 0.2 -> P.  src [nb, R, R, c] (CONST: [R, R, c] for
// every sample).  conv_out: row b at conv_out + b * ld (or nullptr)
template <bool BLUR>
__global__ void __launch_bounds__(256)
epilogue_kernel(const float *__restrict__ src, int64_t src_bstride, int64_t nb, int R, int c, const float *__restrict__ bias,
                const float *__restrict__ noise_w, const float *__restrict__ noise, float *__restrict__ conv_out, int64_t ld,
                float *__restrict__ P) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= nb * R * R * c) return;
    const int ch = (int)(idx % c);
    const int64_t pg = idx / c;
    const int pix = (int)(pg % ((int64_t)R * R));
    const int64_t b = pg / ((int64_t)R * R);
    const float *s = src + b * src_bstride + ch;
    float v;
    if (BLUR) {
        const int x = pix % R, y = pix / R;
        const float k1[3] = {1.f, 2.f, 1.f};
        v = 0.f;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const int yy = y + i - 1;
            if (yy < 0 || yy >= R) continue;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int xx = x + j - 1;
                if (xx < 0 || xx >= R) continue;
                v = fmaf(k1[i] * k1[j] * 0.0625f, s[((int64_t)yy * R + xx) * c], v);
            }
        }
    } else {
        v = s[(int64_t)pix * c];
    }
    v += bias[ch];
    if (conv_out) conv_out[b * ld + (int64_t)pix * c + ch] = v;
    v = fmaf(noise_w[ch], noise[pix], v);
    P[idx] = v >= 0.f ? v : v * 0.2f;
}

// per (sample, channel) mean and 1/sqrt(biased var + 1e-5) of P [nb, hw, c]: grid (nb, ceil(c/32)), 256 threads; lane = channel,
// warp w sums pixels w, w+8, ... in fp64; the 8 warp partials are added in warp order (fixed order, no atomics)
__global__ void __launch_bounds__(256)
stats_kernel(const float *__restrict__ P, int hw, int c, float *__restrict__ mean_out, float *__restrict__ rstd_out) {
    __shared__ double red[8][32];
    __shared__ double mean_s[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ch = blockIdx.y * 32 + lane;
    const int64_t b = blockIdx.x;
    const float *Pb = P + b * (int64_t)hw * c;
    double s = 0.0;
    if (ch < c)
        for (int p = warp; p < hw; p += 8) s += (double)Pb[(int64_t)p * c + ch];
    red[warp][lane] = s;
    __syncthreads();
    if (warp == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w][lane];
        mean_s[lane] = t / (double)hw;
    }
    __syncthreads();
    const double mu = mean_s[lane];
    double q = 0.0;
    if (ch < c)
        for (int p = warp; p < hw; p += 8) { const double d = (double)Pb[(int64_t)p * c + ch] - mu; q += d * d; }
    __syncthreads();
    red[warp][lane] = q;
    __syncthreads();
    if (warp == 0 && ch < c) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w][lane];
        mean_out[b * c + ch] = (float)mu;
        rstd_out[b * c + ch] = (float)(1.0 / sqrt(t / (double)hw + 1e-5));
    }
}

// instance norm + StyleMod: y = (P - mean) * rstd * (s0 + 1) + s1;  style [nb, 2c] (chunk-local rows)
__global__ void __launch_bounds__(256)
norm_style_kernel(const float *__restrict__ P, int64_t nb, int hw, int c, const float *__restrict__ mean, const float *__restrict__ rstd,
                  const float *__restrict__ style, __half *__restrict__ out_hi, __half *__restrict__ out_lo, float *__restrict__ out_f32,
                  int64_t ld, unsigned *overflow) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= nb * hw * c) return;
    const int ch = (int)(idx % c);
    const int64_t pg = idx / c;
    const int pix = (int)(pg % hw);
    const int64_t b = pg / hw;
    const float xn = (P[idx] - mean[b * c + ch]) * rstd[b * c + ch];
    const float y = fmaf(xn, style[b * 2 * c + ch] + 1.f, style[b * 2 * c + c + ch]);
    if (out_hi) {
        const __half h = __float2half_rn(y);
        out_hi[idx] = h;
        out_lo[idx] = __float2half_rn(y - __half2float(h));
        if (fabsf(y) > 60000.f) atomicOr(overflow, 1u);
    }
    if (out_f32) out_f32[b * ld + (int64_t)pix * c + ch] = y;
}

// torgb: img[b, o, p] = sum_c w[o, c] x[b, p, c] + bias[o]  (NCHW output, row b at img + b * ld)
__global__ void rgb_kernel(const float *__restrict__ x, int64_t n, int hw, int c, const float *__restrict__ w, const float *__restrict__ bias,
                           float *__restrict__ img, int64_t ld) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= n * hw) return;
    const int p = (int)(idx % hw);
    const int64_t b = idx / hw;
    const float *xr = x + idx * c;
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;
    for (int k = 0; k < c; ++k) { const float v = xr[k]; r0 = fmaf(w[k], v, r0); r1 = fmaf(w[c + k], v, r1); r2 = fmaf(w[2 * c + k], v, r2); }
    float *o = img + b * ld;
    o[p] = r0 + bias[0];
    o[(int64_t)hw + p] = r1 + bias[1];
    o[2 * (int64_t)hw + p] = r2 + bias[2];
}

// ---- workspace ------------------------------------------------------------------------------------------
struct Ws {
    float *S[MAX_LAYERS];     // [n, 2 cout] styles
    __half *act[2][2];        // [ping-pong][hi/lo] NHWC operands
    float *Y, *C, *P, *mean, *rstd, *last;
    size_t bytes;
};
static int chunk_samples(const gsb_sg1_layer &c) {
    const int hw = res_in_of(c) * res_in_of(c);
    return hw >= CHUNK_ROWS ? 1 : CHUNK_ROWS / hw;
}
static Ws workspace(void *base, const gsb_sg1_layer *layers, int n_run, int64_t n, bool image) {
    Ws w;
    char *p = reinterpret_cast<char *>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { char *q = p + off; off += align_up(bytes, 256); return q; };
    size_t act = 16, y = 16, cp = 16, cmax = 16;
    for (int l = 0; l < n_run; ++l) {
        const gsb_sg1_layer &c = layers[l];
        w.S[l] = (float *)take((size_t)n * 2 * c.cout * 4);
        const size_t spc = (size_t)chunk_samples(c), hw_in = (size_t)res_in_of(c) * res_in_of(c), hw = (size_t)c.res_out * c.res_out;
        act = act > (size_t)n * hw * c.cout ? act : (size_t)n * hw * c.cout;
        if (c.kind != CONST) y = y > spc * hw_in * npad_of(c) ? y : spc * hw_in * npad_of(c);
        cp = cp > spc * hw * c.cout ? cp : spc * hw * c.cout;
        cmax = cmax > (size_t)c.cout ? cmax : (size_t)c.cout;
    }
    for (int a = 0; a < 2; ++a)
        for (int h = 0; h < 2; ++h) w.act[a][h] = (__half *)take(act * 2);
    w.Y = (float *)take(y * 4);
    w.C = (float *)take(cp * 4);
    w.P = (float *)take(cp * 4);
    size_t spc_max = 1;
    for (int l = 0; l < n_run; ++l) spc_max = spc_max > (size_t)chunk_samples(layers[l]) ? spc_max : (size_t)chunk_samples(layers[l]);
    w.mean = (float *)take(spc_max * cmax * 4);
    w.rstd = (float *)take(spc_max * cmax * 4);
    const gsb_sg1_layer &last = layers[n_run - 1];
    w.last = image ? (float *)take((size_t)n * last.res_out * last.res_out * last.cout * 4) : nullptr;
    w.bytes = off;
    return w;
}

static unsigned blocks_for(int64_t total) { return (unsigned)((total + 255) / 256); }

}  // namespace sg1
}  // namespace gsb

using namespace gsb::sg1;

extern "C" size_t gsb_sg1_packed_bytes(const gsb_sg1_layer *layers, int n_layers, int dlatent) {
    if (check(layers, n_layers, dlatent)) return 0;
    return view(nullptr, layers, n_layers, dlatent).bytes;
}

extern "C" int gsb_sg1_pack(const gsb_sg1_layer *layers, int n_layers, int dlatent, const float *d_rgb_weight, const float *d_rgb_bias,
                            void *d_packed, size_t packed_bytes, gsb_stream_t stream) {
    if (int r = check(layers, n_layers, dlatent)) return r;
    GSB_CHECK_ARG(d_rgb_weight && d_rgb_bias && d_packed, "sg1_pack: null pointer");
    View v = view(d_packed, layers, n_layers, dlatent);
    if (packed_bytes < v.bytes) { gsb::set_error("sg1_pack: buffer too small (%zu < %zu)", packed_bytes, v.bytes); return GSB_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    GSB_CHECK_CUDA(cudaMemsetAsync(d_packed, 0, v.bytes, st));
    const float smul = (float)(1.0 / sqrt((double)dlatent));             // StyleMod.lin: gain 1, use_wscale (model.py:127-129)
    for (int l = 0; l < n_layers; ++l) {
        const gsb_sg1_layer &c = layers[l];
        const LayerView &L = v.L[l];
        GSB_CHECK_ARG(c.weight && c.bias && c.noise_weight && c.noise && c.style_weight && c.style_bias,
                      "sg1_pack: layer %d has a null parameter pointer", l);
        if (c.kind == CONST) {
            const_nhwc_kernel<<<(16 * c.cout + 255) / 256, 256, 0, st>>>(c.weight, c.cout, L.cst);
            GSB_CHECK_LAUNCH();
        } else {
            // MyConv2d w_mul = sqrt(2) / sqrt(cin * 9) computed in doubles, applied in fp32 (model.py:60-64,85)
            const float wmul = (float)(sqrt(2.0) * pow((double)c.cin * 9.0, -0.5));
            absmax_kernel<<<128, 256, 0, st>>>(c.weight, c.kind, c.cout, c.cin, wmul, L.scal + 2);
            GSB_CHECK_LAUNCH();
            pick_scale_kernel<<<1, 1, 0, st>>>(L.scal);
            GSB_CHECK_LAUNCH();
            weight_pack_kernel<<<256, 256, 0, st>>>(c.weight, c.kind, c.cout, c.cin, wmul, L.scal, L.w_hi, L.w_lo);
            GSB_CHECK_LAUNCH();
        }
        scale_copy_kernel<<<4, 256, 0, st>>>(c.bias, c.cout, 1.f, L.bias);
        GSB_CHECK_LAUNCH();
        scale_copy_kernel<<<4, 256, 0, st>>>(c.noise_weight, c.cout, 1.f, L.noise_w);
        GSB_CHECK_LAUNCH();
        scale_copy_kernel<<<64, 256, 0, st>>>(c.noise, (int64_t)c.res_out * c.res_out, 1.f, L.noise);
        GSB_CHECK_LAUNCH();
        scale_copy_kernel<<<128, 256, 0, st>>>(c.style_weight, (int64_t)2 * c.cout * dlatent, smul, L.style_w);
        GSB_CHECK_LAUNCH();
        scale_copy_kernel<<<4, 256, 0, st>>>(c.style_bias, 2 * c.cout, 1.f, L.style_b);
        GSB_CHECK_LAUNCH();
    }
    const int cl = layers[n_layers - 1].cout;
    scale_copy_kernel<<<4, 256, 0, st>>>(d_rgb_weight, 3 * cl, (float)(1.0 / sqrt((double)cl)), v.rgb_w);      // torgb: gain 1
    GSB_CHECK_LAUNCH();
    scale_copy_kernel<<<1, 32, 0, st>>>(d_rgb_bias, 3, 1.f, v.rgb_b);
    GSB_CHECK_LAUNCH();
    return GSB_OK;
}

extern "C" size_t gsb_sg1_workspace_bytes(const gsb_sg1_layer *layers, int n_layers, int n_run, int stop, int64_t n) {
    if (!layers || n_run < 1 || n_run > n_layers || n_layers > MAX_LAYERS || n < 1) return 0;
    return workspace(nullptr, layers, n_run, n, stop == STOP_IMAGE).bytes;
}

extern "C" int gsb_sg1_forward(const void *d_packed, const gsb_sg1_layer *layers, int n_layers, int dlatent, int n_run, int stop,
                               const float *d_w, int w_layers, int64_t n, float *d_out, int64_t ld_out, void *d_workspace,
                               size_t workspace_bytes, gsb_stream_t stream) {
    if (int r = check(layers, n_layers, dlatent)) return r;
    GSB_CHECK_ARG(d_packed && d_w && d_out && d_workspace, "sg1_forward: null pointer");
    GSB_CHECK_ARG(n_run >= 1 && n_run <= n_layers && w_layers >= 1 && stop >= STOP_EPI && stop <= STOP_IMAGE,
                  "sg1_forward: n_run / w_layers / stop out of range");
    GSB_CHECK_ARG(stop != STOP_IMAGE || n_run == n_layers, "sg1_forward: the image needs every layer");
    if (n == 0) return GSB_OK;
    const gsb_sg1_layer &tgt = layers[n_run - 1];
    const int64_t need = stop == STOP_STYLE ? 2 * tgt.cout : (stop == STOP_IMAGE ? 3 : tgt.cout) * (int64_t)tgt.res_out * tgt.res_out;
    GSB_CHECK_ARG(n > 0 && ld_out >= need, "sg1_forward: ld_out %lld < %lld", (long long)ld_out, (long long)need);
    View v = view(const_cast<void *>(d_packed), layers, n_layers, dlatent);
    cudaStream_t st = (cudaStream_t)stream;
    auto latent = [&](int j) { return d_w + (size_t)(j < w_layers ? j : w_layers - 1) * n * dlatent; };
    if (stop == STOP_STYLE) {                    // the style vector depends on the latent only
        small_linear_kernel<<<blocks_for(n * 2 * tgt.cout), 256, 0, st>>>(latent(n_run - 1), dlatent, v.L[n_run - 1].style_w,
                                                                         v.L[n_run - 1].style_b, d_out, ld_out, n, 2 * tgt.cout, dlatent);
        GSB_CHECK_LAUNCH();
        return GSB_OK;
    }
    Ws w = workspace(d_workspace, layers, n_run, n, stop == STOP_IMAGE);
    if (workspace_bytes < w.bytes) { gsb::set_error("sg1_forward: workspace too small (%zu < %zu)", workspace_bytes, w.bytes); return GSB_ERR_WORKSPACE; }
    for (int l = 0; l < n_run; ++l) {
        const gsb_sg1_layer &c = layers[l];
        small_linear_kernel<<<blocks_for(n * 2 * c.cout), 256, 0, st>>>(latent(l), dlatent, v.L[l].style_w, v.L[l].style_b, w.S[l],
                                                                       2 * c.cout, n, 2 * c.cout, dlatent);
        GSB_CHECK_LAUNCH();
    }
    for (int l = 0; l < n_run; ++l) {
        const gsb_sg1_layer &c = layers[l];
        const LayerView &L = v.L[l];
        const bool target = (l == n_run - 1);
        const int src = l & 1, dst = src ^ 1;
        const int Hin = res_in_of(c), R = c.res_out, hw = R * R, co = c.cout;
        const int64_t hw_in = (int64_t)Hin * Hin;
        const int spc = chunk_samples(c), npad = c.kind == CONST ? 0 : npad_of(c);
        for (int64_t b0 = 0; b0 < n; b0 += spc) {
            const int64_t nb = (b0 + spc <= n) ? spc : (n - b0);
            const int64_t tot = nb * hw * co;
            const float *esrc = L.cst;
            int64_t ebs = 0;
            if (c.kind != CONST) {
                if (int r = gsb::tc_gemm_plain(w.act[src][0] + b0 * hw_in * c.cin, w.act[src][1] + b0 * hw_in * c.cin, nb * hw_in, c.cin,
                                               L.w_hi, L.w_lo, npad, L.scal, w.Y, v.overflow, 0, st)) return r;
                if (c.kind == SAME) gather_kernel<SAME><<<blocks_for(tot), 256, 0, st>>>(w.Y, nb, Hin, R, co, npad, w.C);
                else if (c.kind == NEAREST) gather_kernel<NEAREST><<<blocks_for(tot), 256, 0, st>>>(w.Y, nb, Hin, R, co, npad, w.C);
                else gather_kernel<FUSED><<<blocks_for(tot), 256, 0, st>>>(w.Y, nb, Hin, R, co, npad, w.C);
                GSB_CHECK_LAUNCH();
                esrc = w.C;
                ebs = (int64_t)hw * co;
            }
            float *conv_out = (target && stop == STOP_CONV) ? d_out + b0 * ld_out : nullptr;
            if (c.kind == NEAREST || c.kind == FUSED)
                epilogue_kernel<true><<<blocks_for(tot), 256, 0, st>>>(esrc, ebs, nb, R, co, L.bias, L.noise_w, L.noise, conv_out, ld_out, w.P);
            else
                epilogue_kernel<false><<<blocks_for(tot), 256, 0, st>>>(esrc, ebs, nb, R, co, L.bias, L.noise_w, L.noise, conv_out, ld_out, w.P);
            GSB_CHECK_LAUNCH();
            if (conv_out) continue;
            stats_kernel<<<dim3((unsigned)nb, (unsigned)((co + 31) / 32)), 256, 0, st>>>(w.P, hw, co, w.mean, w.rstd);
            GSB_CHECK_LAUNCH();
            __half *ohi = target ? nullptr : w.act[dst][0] + b0 * hw * co;
            __half *olo = target ? nullptr : w.act[dst][1] + b0 * hw * co;
            float *of = nullptr;
            int64_t ld = 0;
            if (target && stop == STOP_EPI) { of = d_out + b0 * ld_out; ld = ld_out; }
            if (target && stop == STOP_IMAGE) { of = w.last + b0 * hw * co; ld = (int64_t)hw * co; }
            norm_style_kernel<<<blocks_for(tot), 256, 0, st>>>(w.P, nb, hw, co, w.mean, w.rstd, w.S[l] + b0 * 2 * co, ohi, olo, of, ld,
                                                                v.overflow);
            GSB_CHECK_LAUNCH();
        }
    }
    if (stop == STOP_IMAGE) {
        const int R = tgt.res_out;
        rgb_kernel<<<blocks_for(n * R * R), 256, 0, st>>>(w.last, n, R * R, tgt.cout, v.rgb_w, v.rgb_b, d_out, ld_out);
        GSB_CHECK_LAUNCH();
    }
    return GSB_OK;
}

extern "C" int gsb_sg1_status(const void *d_packed, const gsb_sg1_layer *layers, int n_layers, int dlatent, unsigned *h_flags) {
    if (int r = check(layers, n_layers, dlatent)) return r;
    GSB_CHECK_ARG(d_packed && h_flags, "sg1_status: null pointer");
    View v = view(const_cast<void *>(d_packed), layers, n_layers, dlatent);
    GSB_CHECK_CUDA(cudaMemcpy(h_flags, v.overflow, sizeof(unsigned), cudaMemcpyDeviceToHost));
    return GSB_OK;
}
