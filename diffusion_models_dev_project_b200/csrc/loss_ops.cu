// K6  kernels of the SCD adaptation loss (reference src/utils/exp_utils.py:256-257):
//
//     loss(x) = mean((A x - y)^2) + lambda * tv_loss(x)
//     tv_loss(x) = sum(|dh|[..., :-1, :] + |dw|[..., :, :-1])      (src/samplers/adaptation.py:7-11)
//       dh = x[..., :, 1:] - x[..., :, :-1],  dw = x[..., 1:, :] - x[..., :-1, :]
//
// i.e. both difference images are cropped to (H-1) x (W-1).  The reference evaluates this with
// ~10 eager tensor passes forward and as many in autograd's backward; here
//   residual_sq : r = Ax - y and the per-block partial sums of r^2 in one pass; with measurement weights W
//                 (PWLS, loss mean(W (Ax - y)^2)) r = W (Ax - y) and the partial sums of W (Ax - y)^2
//   tv_fwd      : per-block partial sums of the cropped |dh| + |dw|
//   tv_grad     : d tv / dx in one pass (sign(0) = 0 like torch.abs' backward)
// Partial sums are written per block and added by the caller in index order (deterministic).
#include "scd_internal.cuh"

#define LOSS_THREADS 256

__device__ __forceinline__ float loss_block_sum(float v, float *red)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) red[w] = v;
    __syncthreads();
    float t = 0.f;
    if (threadIdx.x < 32) {
        t = (threadIdx.x < (LOSS_THREADS >> 5)) ? red[threadIdx.x] : 0.f;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
    }
    return t;   // valid in thread 0
}

__global__ void __launch_bounds__(LOSS_THREADS)
residual_sq_kernel(const float *__restrict__ ax, const float *__restrict__ y, const float *__restrict__ w,
                   float *__restrict__ r, float *__restrict__ part, int64_t numel)
{
    __shared__ float red[LOSS_THREADS / 32];
    scd_pdl_wait();
    scd_pdl_trigger();
    float acc = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * LOSS_THREADS + threadIdx.x; i < numel; i += (int64_t)gridDim.x * LOSS_THREADS) {
        const float d = ax[i] - y[i];
        const float rw = w ? w[i] * d : d;         // W = 1: the same bits as no weights
        r[i] = rw;
        acc = fmaf(rw, d, acc);
    }
    const float tot = loss_block_sum(acc, red);
    if (threadIdx.x == 0) part[blockIdx.x] = tot;
}

// grid = (blocks over the pixels of one image, images)
__global__ void __launch_bounds__(LOSS_THREADS)
tv_fwd_kernel(const float *__restrict__ x, float *__restrict__ part, int n0, int n1)
{
    __shared__ float red[LOSS_THREADS / 32];
    scd_pdl_wait();
    scd_pdl_trigger();
    const float *im = x + (size_t)blockIdx.y * n0 * n1;
    const int n = (n0 - 1) * (n1 - 1);
    float acc = 0.f;
    for (int i = blockIdx.x * LOSS_THREADS + threadIdx.x; i < n; i += gridDim.x * LOSS_THREADS) {
        const int h = i / (n1 - 1), w = i - h * (n1 - 1);
        const float c = im[(size_t)h * n1 + w];
        acc += fabsf(im[(size_t)h * n1 + w + 1] - c) + fabsf(im[(size_t)(h + 1) * n1 + w] - c);
    }
    const float tot = loss_block_sum(acc, red);
    if (threadIdx.x == 0) part[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = tot;
}

__device__ __forceinline__ float sgn(float v) { return (float)((v > 0.f) - (v < 0.f)); }

__global__ void __launch_bounds__(LOSS_THREADS)
tv_grad_kernel(const float *__restrict__ x, float *__restrict__ g, int n0, int n1)
{
    scd_pdl_wait();
    scd_pdl_trigger();
    const float *im = x + (size_t)blockIdx.y * n0 * n1;
    float *out = g + (size_t)blockIdx.y * n0 * n1;
    const int n = n0 * n1;
    for (int i = blockIdx.x * LOSS_THREADS + threadIdx.x; i < n; i += gridDim.x * LOSS_THREADS) {
        const int h = i / n1, w = i - h * n1;
        const float c = im[i];
        float v = 0.f;
        // terms |x[h,w+1]-x[h,w]| and |x[h+1,w]-x[h,w]| exist for h < n0-1, w < n1-1
        if (h < n0 - 1 && w < n1 - 1) v -= sgn(im[i + 1] - c) + sgn(im[i + n1] - c);
        if (h < n0 - 1 && w >= 1) v += sgn(c - im[i - 1]);          // |x[h,w]-x[h,w-1]|, column w-1 < n1-1
        if (h >= 1 && w < n1 - 1) v += sgn(c - im[i - n1]);         // |x[h,w]-x[h-1,w]|, row h-1 < n0-1
        out[i] = v;
    }
}

static int loss_blocks(int64_t n)
{
    int64_t nb = (n + LOSS_THREADS * 4 - 1) / (LOSS_THREADS * 4);
    return (int)(nb < 1 ? 1 : (nb > 1184 ? 1184 : nb));     // <= 8 CTAs per SM
}

extern "C" int scd_residual_sq_blocks(int64_t numel) { return loss_blocks(numel); }

int scd_launch_residual_sq(const float *ax, const float *y, const float *w, float *r, float *part, int64_t numel,
                           cudaStream_t st)
{
    if (!ax || !y || !r || !part) { scd_set_error("scd_residual_sq: null argument"); return SCD_E_INVALID; }
    if (numel <= 0) return 0;
    SCD_CUDA(scd_launch_kernel(residual_sq_kernel, dim3(loss_blocks(numel)), dim3(LOSS_THREADS), 0, st, 0,
                               ax, y, w, r, part, numel));
    SCD_LAUNCH_CHECK("residual_sq_kernel");
    return 0;
}

extern "C" int scd_residual_sq(const float *ax, const float *y, float *r, float *part, int64_t numel, void *stream)
{
    return scd_launch_residual_sq(ax, y, nullptr, r, part, numel, (cudaStream_t)stream);
}

extern "C" int scd_residual_sq_w(const float *ax, const float *y, const float *w, float *r, float *part, int64_t numel,
                                 void *stream)
{
    if (!w) { scd_set_error("scd_residual_sq_w: null weights"); return SCD_E_INVALID; }
    return scd_launch_residual_sq(ax, y, w, r, part, numel, (cudaStream_t)stream);
}

extern "C" int scd_tv_blocks(int n0, int n1)
{
    int nb = loss_blocks((int64_t)n0 * n1);
    return nb > 64 ? 64 : nb;
}

extern "C" int scd_tv_loss(const float *x, float *part, int images, int n0, int n1, void *stream)
{
    if (!x || !part) { scd_set_error("scd_tv_loss: null argument"); return SCD_E_INVALID; }
    if (images <= 0) return 0;
    if (n0 < 2 || n1 < 2 || images > 65535) { scd_set_error("scd_tv_loss: bad shape"); return SCD_E_INVALID; }
    SCD_CUDA(scd_launch_kernel(tv_fwd_kernel, dim3(scd_tv_blocks(n0, n1), images), dim3(LOSS_THREADS), 0,
                               (cudaStream_t)stream, 0, x, part, n0, n1));
    SCD_LAUNCH_CHECK("tv_fwd_kernel");
    return 0;
}

extern "C" int scd_tv_grad(const float *x, float *grad, int images, int n0, int n1, void *stream)
{
    if (!x || !grad) { scd_set_error("scd_tv_grad: null argument"); return SCD_E_INVALID; }
    if (images <= 0) return 0;
    if (n0 < 2 || n1 < 2 || images > 65535) { scd_set_error("scd_tv_grad: bad shape"); return SCD_E_INVALID; }
    SCD_CUDA(scd_launch_kernel(tv_grad_kernel, dim3(scd_tv_blocks(n0, n1), images), dim3(LOSS_THREADS), 0,
                               (cudaStream_t)stream, 0, x, grad, n0, n1));
    SCD_LAUNCH_CHECK("tv_grad_kernel");
    return 0;
}
