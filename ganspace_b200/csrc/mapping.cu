// StyleGAN2 mapping network  z[n,dim] -> w[n,dim]   (fp32 FMA path)
//
// Replaces models/stylegan2/stylegan2-pytorch/model.py:400-409 (Generator.style), :14-19 (PixelNorm),
// :151-161 (EqualLinear.forward) and op/fused_act.py:86-92 (fused bias + leaky-ReLU(0.2) * sqrt(2)).
//
// This file holds the reference-grade fp32 path: a PixelNorm kernel and an SGEMM (both operands
// K-major, 128x128x16 tiles, 8x8 register tile per thread, double-buffered smem) with the
// bias + leaky-ReLU + sqrt(2) epilogue fused.  It is the numerics anchor for the tcgen05 path
// (mapping_tc.cu) and the fallback-free default until that path is parity-green.
//
// Packed layout produced by gsb_mapping_pack:  [n_layers][dim*dim] fp32 of (weight*scale) row-major
// (out,in), followed by [n_layers][dim] fp32 of (bias*lr_mul).
#include "common.cuh"

namespace gsb {

// tensor-core path (mapping_tc.cu)
size_t mapping_tc_packed_bytes(int n_layers, int dim);
int mapping_tc_pack(const float *pw, int n_layers, int dim, void *tc_base, cudaStream_t st);
int mapping_forward_tc(const float *pb, void *tc_base, int n_layers, int dim, const float *d_z, float *d_w,
                       int64_t n, bool pixelnorm, void *ws, int leave_free_sms, cudaStream_t st);
size_t mapping_tc_workspace_bytes(int64_t n, int dim);
size_t tc_linear_workspace_bytes(int64_t n, int N, int K);
int tc_linear(const float *x, const float *w, const float *bias, float *y, int64_t n, int N, int K, bool lrelu, void *ws,
              cudaStream_t st);
unsigned *mapping_tc_overflow_flag(void *tc_base, int n_layers, int dim);

static inline size_t simt_packed_bytes(int n_layers, int dim) {
    return align_up(((size_t)n_layers * dim * dim + (size_t)n_layers * dim) * sizeof(float), 256);
}
static inline bool tc_supported(int n_layers, int dim) { return n_layers > 0 && dim % 256 == 0; }

__global__ void mapping_pack_kernel(const float *__restrict__ w, const float *__restrict__ b,
                                    int n_layers, int dim, float scale, float lr_mul,
                                    float *__restrict__ pw, float *__restrict__ pb) {
    int64_t nw = (int64_t)n_layers * dim * dim;
    int64_t nb = (int64_t)n_layers * dim;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nw + nb;
         i += (int64_t)gridDim.x * blockDim.x) {
        if (i < nw) pw[i] = __fmul_rn(w[i], scale);          // model.py:153  self.weight * self.scale
        else pb[i - nw] = __fmul_rn(b[i - nw], lr_mul);      // model.py:154  self.bias * self.lr_mul
    }
}

// One warp per row: x * rsqrt(mean(x^2) + 1e-8)   (model.py:14-19)
__global__ void pixelnorm_kernel(const float *__restrict__ x, float *__restrict__ y, int64_t n, int dim) {
    int64_t row = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const int lane = threadIdx.x & 31;
    const float4 *xr = reinterpret_cast<const float4 *>(x + row * dim);
    float4 *yr = reinterpret_cast<float4 *>(y + row * dim);
    float s = 0.f;
    for (int i = lane; i < dim / 4; i += 32) {
        float4 v = xr[i];
        s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    s = warp_sum(s);
    float r = 1.0f / sqrtf(s / (float)dim + 1e-8f);
    for (int i = lane; i < dim / 4; i += 32) {
        float4 v = xr[i];
        v.x *= r; v.y *= r; v.z *= r; v.w *= r;
        yr[i] = v;
    }
}

constexpr int BM = 128, BN = 128, BK = 16, TM = 8, TN = 8;
constexpr int SGEMM_THREADS = 256;

// C[M,N] = act(A[M,K] * W[N,K]^T + bias[N]);  act = sqrt2 * leaky_relu_0.2 when LRELU.
// Requires K % 16 == 0, N % 128 == 0; M arbitrary.
template <bool LRELU>
__global__ void __launch_bounds__(SGEMM_THREADS, 2)
sgemm_tn_bias_act_kernel(const float *__restrict__ A, const float *__restrict__ W,
                         const float *__restrict__ bias, float *__restrict__ C, int64_t M, int N, int K) {
    __shared__ __align__(16) float As[2][BK][BM + 4];
    __shared__ __align__(16) float Ws[2][BK][BN + 4];
    const int tid = threadIdx.x;
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int tx = tid & 15, ty = tid >> 4;          // 16 x 16 thread grid, 8x8 outputs each
    // global -> smem loader mapping: 128 rows x 16 k = 512 float4; 2 per thread
    const int lr = tid >> 2;        // 0..63
    const int lk = (tid & 3) * 4;   // 0,4,8,12
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    float4 ra[2], rw[2];
    auto gload = [&](int k0) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int r = lr + 64 * h;
            int64_t gm = m0 + r;
            ra[h] = (gm < M) ? *reinterpret_cast<const float4 *>(A + gm * K + k0 + lk)
                             : make_float4(0.f, 0.f, 0.f, 0.f);
            rw[h] = *reinterpret_cast<const float4 *>(W + (int64_t)(n0 + r) * K + k0 + lk);
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int r = lr + 64 * h;
            As[buf][lk + 0][r] = ra[h].x; As[buf][lk + 1][r] = ra[h].y;
            As[buf][lk + 2][r] = ra[h].z; As[buf][lk + 3][r] = ra[h].w;
            Ws[buf][lk + 0][r] = rw[h].x; Ws[buf][lk + 1][r] = rw[h].y;
            Ws[buf][lk + 2][r] = rw[h].z; Ws[buf][lk + 3][r] = rw[h].w;
        }
    };
    gload(0);
    sstore(0);
    __syncthreads();
    const int nk = K / BK;
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) gload((kt + 1) * BK);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[TM], b[TN];
            // rows ty*4..+3 and 64+ty*4..+3 ; cols tx*4..+3 and 64+tx*4..+3 (conflict-free float4 reads)
            float4 a0 = *reinterpret_cast<const float4 *>(&As[buf][k][ty * 4]);
            float4 a1 = *reinterpret_cast<const float4 *>(&As[buf][k][64 + ty * 4]);
            float4 b0 = *reinterpret_cast<const float4 *>(&Ws[buf][k][tx * 4]);
            float4 b1 = *reinterpret_cast<const float4 *>(&Ws[buf][k][64 + tx * 4]);
            a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
            a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
            b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
            b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (kt + 1 < nk) {
            sstore(buf ^ 1);
            __syncthreads();
        }
    }
    // epilogue:  sqrt2 * leaky_relu(acc + bias, 0.2)   (op/fused_act.py:88-90)
    const float sqrt2 = 1.41421356237309515f;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        int64_t gm = m0 + ((i < 4) ? (ty * 4 + i) : (64 + ty * 4 + i - 4));
        if (gm >= M) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int gn = n0 + h * 64 + tx * 4;
            float4 bv = *reinterpret_cast<const float4 *>(bias + gn);
            float v[4] = {acc[i][h * 4 + 0] + bv.x, acc[i][h * 4 + 1] + bv.y,
                          acc[i][h * 4 + 2] + bv.z, acc[i][h * 4 + 3] + bv.w};
            if (LRELU) {
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = __fmul_rn(sqrt2, (v[q] >= 0.f) ? v[q] : __fmul_rn(v[q], 0.2f));
            }
            *reinterpret_cast<float4 *>(C + gm * N + gn) = make_float4(v[0], v[1], v[2], v[3]);
        }
    }
}

int mapping_forward_simt(const float *pw, const float *pb, int n_layers, int dim, const float *d_z,
                         float *d_w, int64_t n, bool pixelnorm, float *tmp0, float *tmp1,
                         cudaStream_t st) {
    const float *cur = d_z;
    if (pixelnorm) {
        int64_t blocks = (n + 7) / 8;
        float *dst = (n_layers == 0) ? d_w : tmp0;
        pixelnorm_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_z, dst, n, dim);
        GSB_CHECK_LAUNCH();
        cur = dst;
    }
    dim3 grid((unsigned)((n + BM - 1) / BM), dim / BN);
    for (int l = 0; l < n_layers; ++l) {
        float *dst = (l == n_layers - 1) ? d_w : ((cur == tmp0) ? tmp1 : tmp0);
        sgemm_tn_bias_act_kernel<true><<<grid, SGEMM_THREADS, 0, st>>>(
            cur, pw + (int64_t)l * dim * dim, pb + (int64_t)l * dim, dst, n, dim, dim);
        GSB_CHECK_LAUNCH();
        cur = dst;
    }
    return GSB_OK;
}

}  // namespace gsb

extern "C" size_t gsb_mapping_packed_bytes(int n_layers, int dim) {
    return gsb::simt_packed_bytes(n_layers, dim) + (gsb::tc_supported(n_layers, dim) ? gsb::mapping_tc_packed_bytes(n_layers, dim) : 0);
}

extern "C" int gsb_mapping_pack(const float *d_weight, const float *d_bias, int n_layers, int dim,
                                float lr_mul, void *d_packed, gsb_stream_t stream) {
    GSB_CHECK_ARG(d_weight && d_bias && d_packed, "mapping_pack: null pointer");
    GSB_CHECK_ARG(n_layers > 0 && dim > 0 && dim % 128 == 0, "mapping_pack: dim must be a multiple of 128");
    float *pw = reinterpret_cast<float *>(d_packed);
    float *pb = pw + (size_t)n_layers * dim * dim;
    // EqualLinear.scale = (1/sqrt(in_dim)) * lr_mul computed in Python doubles, then used as a
    // Python float multiplying a float32 tensor (model.py:148,153) -> rounded to fp32 once.
    float scale = (float)((1.0 / sqrt((double)dim)) * (double)lr_mul);
    gsb::mapping_pack_kernel<<<512, 256, 0, (cudaStream_t)stream>>>(d_weight, d_bias, n_layers, dim, scale,
                                                                   lr_mul, pw, pb);
    GSB_CHECK_LAUNCH();
    if (gsb::tc_supported(n_layers, dim)) {
        void *tc_base = reinterpret_cast<char *>(d_packed) + gsb::simt_packed_bytes(n_layers, dim);
        return gsb::mapping_tc_pack(pw, n_layers, dim, tc_base, (cudaStream_t)stream);
    }
    return GSB_OK;
}

extern "C" size_t gsb_mapping_workspace_bytes(int64_t n, int dim) {
    size_t simt = 2 * gsb::align_up((size_t)n * dim * sizeof(float), 256);
    size_t tc = gsb::mapping_tc_workspace_bytes(n, dim);
    return simt > tc ? simt : tc;
}

extern "C" int gsb_mapping_forward(const void *d_packed, int n_layers, int dim, const float *d_z,
                                   float *d_w, int64_t n, int flags, void *d_workspace,
                                   size_t workspace_bytes, gsb_stream_t stream) {
    GSB_CHECK_ARG(d_z && d_w && (d_packed || n_layers == 0), "mapping_forward: null pointer");
    GSB_CHECK_ARG(n_layers >= 0 && dim % 128 == 0, "mapping_forward: dim must be a multiple of 128");
    GSB_CHECK_ARG(n_layers > 0 || (flags & 1), "mapping_forward: nothing to do (n_layers == 0 without PixelNorm)");
    if (n == 0) return GSB_OK;
    if (workspace_bytes < gsb_mapping_workspace_bytes(n, dim) || !d_workspace) {
        gsb::set_error("mapping_forward: workspace too small (%zu < %zu)", workspace_bytes,
                       gsb_mapping_workspace_bytes(n, dim));
        return GSB_ERR_WORKSPACE;
    }
    const float *pw = reinterpret_cast<const float *>(d_packed);
    const float *pb = pw + (size_t)n_layers * dim * dim;
    if (!(flags & 2) && gsb::tc_supported(n_layers, dim)) {
        void *tc_base = reinterpret_cast<char *>(const_cast<void *>(d_packed)) + gsb::simt_packed_bytes(n_layers, dim);
        return gsb::mapping_forward_tc(pb, tc_base, n_layers, dim, d_z, d_w, n, (flags & 1) != 0, d_workspace,
                                       (flags >> 8) & 0xff, (cudaStream_t)stream);
    }
    float *tmp0 = reinterpret_cast<float *>(d_workspace);
    float *tmp1 = reinterpret_cast<float *>(reinterpret_cast<char *>(d_workspace) +
                                            gsb::align_up((size_t)n * dim * sizeof(float), 256));
    return gsb::mapping_forward_simt(pw, pb, n_layers, dim, d_z, d_w, n, (flags & 1) != 0, tmp0, tmp1,
                                     (cudaStream_t)stream);
}

extern "C" int gsb_mapping_status(const void *d_packed, int n_layers, int dim, unsigned *h_flags) {
    GSB_CHECK_ARG(d_packed && h_flags, "mapping_status: null pointer");
    *h_flags = 0;
    if (!gsb::tc_supported(n_layers, dim)) return GSB_OK;
    void *tc_base = reinterpret_cast<char *>(const_cast<void *>(d_packed)) + gsb::simt_packed_bytes(n_layers, dim);
    GSB_CHECK_CUDA(cudaMemcpy(h_flags, gsb::mapping_tc_overflow_flag(tc_base, n_layers, dim), sizeof(unsigned),
                              cudaMemcpyDeviceToHost));
    return GSB_OK;
}

// Generic affine layer  y[n,N] = x[n,K] * W[N,K]^T + bias[N]  (bias may be NULL), optional sqrt2*lrelu.
//   replaces  nn.Linear / F.linear call sites of the path outside the mapping network, e.g. BigGAN's
//   generator.gen_z (biggan model.py:211-212,232; spectral norm folded into W by the caller).
// bit 1 of flags (the caller vouches that |x| stays inside fp16's range) selects the tcgen05 kernel for shapes it covers
static bool linear_tc_eligible(int64_t n, int N, int K, int flags) {
    return (flags & 2) && n >= 128 && N % 256 == 0 && K % 64 == 0;
}

extern "C" size_t gsb_linear_workspace_bytes(int64_t n, int N, int K, int flags) {
    size_t b = (size_t)N * sizeof(float);
    if (linear_tc_eligible(n, N, K, flags)) {
        size_t t = gsb::tc_linear_workspace_bytes(n, N, K) + gsb::align_up((size_t)N * sizeof(float), 256);
        if (t > b) b = t;
    }
    return b;
}

extern "C" int gsb_linear_forward(const float *d_x, const float *d_w, const float *d_bias, float *d_y, int64_t n,
                                  int N, int K, int flags, void *d_workspace, size_t workspace_bytes,
                                  gsb_stream_t stream) {
    GSB_CHECK_ARG(d_x && d_w && d_y, "linear_forward: null pointer");
    GSB_CHECK_ARG(n >= 0 && N > 0 && K > 0 && N % 128 == 0 && K % 16 == 0, "linear_forward: need N%%128==0, K%%16==0 (N=%d K=%d)", N, K);
    if (n == 0) return GSB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (linear_tc_eligible(n, N, K, flags) && d_workspace && workspace_bytes >= gsb_linear_workspace_bytes(n, N, K, flags)) {
        // tensor cores (tcgen05, fp16 hi/lo split operands = fp32-grade): zero bias first if none was given
        float *zb = reinterpret_cast<float *>(d_workspace);
        char *rest = reinterpret_cast<char *>(d_workspace) + gsb::align_up((size_t)N * sizeof(float), 256);
        if (!d_bias) GSB_CHECK_CUDA(cudaMemsetAsync(zb, 0, (size_t)N * sizeof(float), st));
        return gsb::tc_linear(d_x, d_w, d_bias ? d_bias : zb, d_y, n, N, K, (flags & 1) != 0, rest, st);
    }
    const float *bias = d_bias;
    if (!bias) {
        if (!d_workspace || workspace_bytes < (size_t)N * sizeof(float)) {
            gsb::set_error("linear_forward: workspace of N floats needed when bias is NULL");
            return GSB_ERR_WORKSPACE;
        }
        GSB_CHECK_CUDA(cudaMemsetAsync(d_workspace, 0, (size_t)N * sizeof(float), st));
        bias = reinterpret_cast<const float *>(d_workspace);
    }
    dim3 grid((unsigned)((n + gsb::BM - 1) / gsb::BM), N / gsb::BN);
    if (flags & 1) gsb::sgemm_tn_bias_act_kernel<true><<<grid, gsb::SGEMM_THREADS, 0, st>>>(d_x, d_w, bias, d_y, n, N, K);
    else gsb::sgemm_tn_bias_act_kernel<false><<<grid, gsb::SGEMM_THREADS, 0, st>>>(d_x, d_w, bias, d_y, n, N, K);
    GSB_CHECK_LAUNCH();
    return GSB_OK;
}

// y = leaky_relu(x, slope), elementwise, without the sqrt(2) gain: StyleGAN's G_mapping activation modules
// (models/stylegan/model.py:192-193, nn.LeakyReLU(0.2)), run on their own only when a g_mapping child is hooked
__global__ void leaky_relu_kernel(const float *__restrict__ x, float *__restrict__ y, int64_t n, float slope) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = x[i];
        y[i] = v >= 0.f ? v : __fmul_rn(v, slope);
    }
}

extern "C" int gsb_leaky_relu(const float *d_x, float *d_y, int64_t n, float slope, gsb_stream_t stream) {
    GSB_CHECK_ARG(d_x && d_y && n >= 0, "leaky_relu: null pointer or negative n");
    if (n == 0) return GSB_OK;
    const int64_t blocks = (n + 255) / 256;
    leaky_relu_kernel<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, (cudaStream_t)stream>>>(d_x, d_y, n, slope);
    GSB_CHECK_LAUNCH();
    return GSB_OK;
}
