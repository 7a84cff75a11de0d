// K9  SCD adaptation objective as two library calls: forward (Tweedie -> data consistency -> loss) and the whole
// hand-written reverse sweep returning d loss / d s.
//
// Replaces, per Adam step of `_adapt` (reference src/samplers/utils.py:241-260), the chain
//     xhat0 = apTweedy(s, x)                               (:370-378)
//     xhat  = cg(op, xhat0, xhat0 + gamma*rhs, n_iter)     (src/utils/cg.py:11-39; or the `dc` gradient step, or none)
//     loss  = mean((A xhat - y)^2) + lambda * tv_loss(xhat) (src/utils/exp_utils.py:256-257, adaptation.py:7-11)
// and autograd's backward through all of it.  The reference differentiates the UNROLLED CG iterations (alpha and
// beta depend on the iterates), so the reverse sweep below differentiates the recurrences exactly -- it is not the
// adjoint linear solve.  With ODL's gradient pairing (grad of A = A*/c_w, grad of A* = c_w A, SURVEY.md 8b) the
// vector-Jacobian product of op(v) = v + gamma A*(A v) is op itself, so the sweep costs n_iter + 1 applications of
// op and a handful of vector kernels whose per-sample scalars never leave the device.
//
//   forward, per iteration k:   d_k = op(p_k), alpha_k = rho_k/<p_k,d_k>, x += alpha_k p_k, r_{k+1} = r_k - alpha_k d_k,
//                               rho_{k+1} = |r_{k+1}|^2, beta_k = rho_{k+1}/rho_k, p_{k+1} = r_{k+1} + beta_k p_k
//   kept for the sweep:         p_k, d_k, r_k (all k), alpha_k, beta_k, rho_k, <p_k,d_k>
//   reverse, k = K-1 .. 0       (gx, gr, gp, grho = adjoints of x, r_{k+1}, p_{k+1}, rho_{k+1}):
//       gbeta = <gp,p_k>; grho' = grho + gbeta/rho_k; gr' = gr + gp + 2 grho' r_{k+1}
//       galpha = <gx,p_k> - <gr',d_k>; gpd = -galpha alpha_k/<p,d>; gd = gpd p_k - alpha_k gr'
//       gp <- beta_k gp + alpha_k gx + gpd d_k + op(gd);  grho <- -gbeta beta_k/rho_k + galpha/<p,d>;  gr <- gr'
//   finally  gr <- gr + gp + 2 grho r_0;   d loss/d xhat0 = gx - gamma A*(A gr)   (start value + right-hand side)
//            d loss/d s = -(std_t/mean_t) * d loss/d xhat0
//
// Measurement weights (scd_adapt_fwd_w / _bwd_w): every op application projects with W (w_il, packed), and the
// loss is mean(W (A xhat - y)^2) + lambda tv: the residual kept for the sweep is r_w = W (A xhat - y), whose plain
// transpose backprojection is the gradient of the weighted data term, so the sweep itself is unchanged.
//
// All buffers live in one caller-provided workspace (scd_adapt_workspace_bytes), which carries the saved vectors
// from scd_adapt_fwd to scd_adapt_bwd.  No allocation, no synchronisation, no host read-back: both calls are
// CUDA-graph capturable.
#include "scd_internal.cuh"
#include <algorithm>
#include <cstring>

#define AD_THREADS 256
#define AD_MAXSUM 3

static inline size_t ad_align(size_t v) { return (v + 255) & ~(size_t)255; }

// up to AD_MAXSUM sums of per-block partials (warp w adds array w in a fixed order), broadcast through smem
struct AdSums { const float *part[AD_MAXSUM]; int n[AD_MAXSUM]; };

__device__ __forceinline__ void ad_sums(const AdSums &S, int count, float *slot /* [AD_MAXSUM] shared */)
{
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (w < count) {
        float v = 0.f;
        for (int i = lane; i < S.n[w]; i += 32) v += S.part[w][i];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if (lane == 0) slot[w] = v;
    }
    __syncthreads();
}

__device__ __forceinline__ float ad_block_sum(float v, float *red /* [AD_THREADS/32] shared */)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();                               // red may still be read from a previous call
    if (lane == 0) red[w] = v;
    __syncthreads();
    float t = 0.f;
    if (threadIdx.x < 32) {
        t = (threadIdx.x < (AD_THREADS >> 5)) ? red[threadIdx.x] : 0.f;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
    }
    return t;   // valid in thread 0
}

#define AD_LOOP(i) for (int64_t i = (int64_t)blockIdx.x * AD_THREADS + threadIdx.x; i < numel; i += (int64_t)gridDim.x * AD_THREADS)

// ---- forward: x += alpha p; r_out = r_in - alpha d; partial |r_out|^2; alpha, rho, <p,d> stored ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_update_kernel(float *__restrict__ x, const float *__restrict__ r_in, float *__restrict__ r_out,
                    const float *__restrict__ p, const float *__restrict__ d,
                    const float *__restrict__ rr_part, int rr_n, const float *__restrict__ pd_part, int pd_n, int stride,
                    float *__restrict__ rr_new_part, float *__restrict__ s_alpha, float *__restrict__ s_rho,
                    float *__restrict__ s_pd, int64_t numel)
{
    __shared__ float slot[AD_MAXSUM], red[AD_THREADS / 32];
    scd_pdl_wait();
    scd_pdl_trigger();
    const int b = blockIdx.y;
    AdSums S;
    S.part[0] = rr_part + (size_t)b * stride; S.n[0] = rr_n;
    S.part[1] = pd_part + (size_t)b * stride; S.n[1] = pd_n;
    ad_sums(S, 2, slot);
    const float rho = slot[0], pd = slot[1];
    const float alpha = __fdiv_rn(rho, pd);        // no guard: same as the reference
    if (blockIdx.x == 0 && threadIdx.x == 0) { s_alpha[b] = alpha; s_rho[b] = rho; s_pd[b] = pd; }
    const size_t base = (size_t)b * numel;
    float acc = 0.f;
    AD_LOOP(i) {
        x[base + i] = fmaf(alpha, p[base + i], x[base + i]);
        const float rv = fmaf(-alpha, d[base + i], r_in[base + i]);
        r_out[base + i] = rv;
        acc = fmaf(rv, rv, acc);
    }
    const float tot = ad_block_sum(acc, red);
    if (threadIdx.x == 0) rr_new_part[(size_t)b * stride + blockIdx.x] = tot;
}

// ---- forward: p_out = r + beta p_in, beta = |r|^2 / rho; beta stored ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_direction_kernel(const float *__restrict__ r, const float *__restrict__ p_in, float *__restrict__ p_out,
                       const float *__restrict__ rr_new_part, int rr_n, int stride, const float *__restrict__ s_rho,
                       float *__restrict__ s_beta, int64_t numel)
{
    __shared__ float slot[AD_MAXSUM];
    scd_pdl_wait();
    scd_pdl_trigger();
    const int b = blockIdx.y;
    AdSums S;
    S.part[0] = rr_new_part + (size_t)b * stride; S.n[0] = rr_n;
    ad_sums(S, 1, slot);
    const float beta = __fdiv_rn(slot[0], s_rho[b]);
    if (blockIdx.x == 0 && threadIdx.x == 0) s_beta[b] = beta;
    const size_t base = (size_t)b * numel;
    AD_LOOP(i) p_out[base + i] = fmaf(beta, p_in[base + i], r[base + i]);
}

// ---- loss = sum(res_part)/n_res + lambda*sum(tv_part), times nothing: one scalar on the device ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_loss_kernel(const float *__restrict__ res_part, int res_n, const float *__restrict__ tv_part, int tv_n,
                  float inv_numel, float lambda, float *__restrict__ loss)
{
    __shared__ float red[AD_THREADS / 32];
    scd_pdl_wait();
    scd_pdl_trigger();
    float a = 0.f, t = 0.f;
    for (int i = threadIdx.x; i < res_n; i += AD_THREADS) a += res_part[i];
    for (int i = threadIdx.x; i < tv_n; i += AD_THREADS) t += tv_part[i];
    const float sa = ad_block_sum(a, red);
    const float st = ad_block_sum(t, red);
    if (threadIdx.x == 0) loss[0] = fmaf(lambda, st, sa * inv_numel);
}

// ---- reverse: partial <a, b> ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_dot_kernel(const float *__restrict__ a, const float *__restrict__ bvec, float *__restrict__ part, int stride, int64_t numel)
{
    __shared__ float red[AD_THREADS / 32];
    scd_pdl_wait();
    scd_pdl_trigger();
    const int b = blockIdx.y;
    const size_t base = (size_t)b * numel;
    float acc = 0.f;
    AD_LOOP(i) acc = fmaf(a[base + i], bvec[base + i], acc);
    const float tot = ad_block_sum(acc, red);
    if (threadIdx.x == 0) part[(size_t)b * stride + blockIdx.x] = tot;
}

// ---- reverse: gr' = gr + gp + 2 (grho + gbeta/rho) r1; partial <gx,p>, <gr',d>   (gr, gp NULL = 0) ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_bw_residual_kernel(const float *__restrict__ gr, const float *__restrict__ gp, const float *__restrict__ r1,
                         const float *__restrict__ gx, const float *__restrict__ p, const float *__restrict__ d,
                         const float *__restrict__ gb_part, int gb_n, int stride, const float *__restrict__ s_grho,
                         const float *__restrict__ s_rho, float *__restrict__ gr_out, float *__restrict__ gxp_part,
                         float *__restrict__ grd_part, int64_t numel)
{
    __shared__ float slot[AD_MAXSUM], red[AD_THREADS / 32];
    scd_pdl_wait();
    scd_pdl_trigger();
    const int b = blockIdx.y;
    float gbeta = 0.f;
    if (gp) {
        AdSums S;
        S.part[0] = gb_part + (size_t)b * stride; S.n[0] = gb_n;
        ad_sums(S, 1, slot);
        gbeta = slot[0];
    }
    const float grho1 = (s_grho ? s_grho[b] : 0.f) + (gp ? __fdiv_rn(gbeta, s_rho[b]) : 0.f);
    const float two = 2.0f * grho1;
    const size_t base = (size_t)b * numel;
    float a1 = 0.f, a2 = 0.f;
    AD_LOOP(i) {
        float v = two * r1[base + i];
        if (gp) v += gp[base + i];
        if (gr) v += gr[base + i];
        gr_out[base + i] = v;
        a1 = fmaf(gx[base + i], p[base + i], a1);
        a2 = fmaf(v, d[base + i], a2);
    }
    const float t1 = ad_block_sum(a1, red);
    const float t2 = ad_block_sum(a2, red);
    if (threadIdx.x == 0) {
        gxp_part[(size_t)b * stride + blockIdx.x] = t1;
        grd_part[(size_t)b * stride + blockIdx.x] = t2;
    }
}

// ---- reverse: gd = gpd p - alpha gr'; gptmp = beta gp + alpha gx + gpd d; grho <- -gbeta beta/rho + galpha/pd ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_bw_direction_kernel(const float *__restrict__ gp, const float *__restrict__ gx, const float *__restrict__ p,
                          const float *__restrict__ d, const float *__restrict__ gr1,
                          const float *__restrict__ gxp_part, const float *__restrict__ grd_part, int n_part,
                          const float *__restrict__ gb_part, int gb_n, int stride,
                          const float *__restrict__ s_alpha, const float *__restrict__ s_beta, const float *__restrict__ s_rho,
                          const float *__restrict__ s_pd, float *__restrict__ s_grho,
                          float *__restrict__ gd, float *__restrict__ gptmp, int64_t numel)
{
    __shared__ float slot[AD_MAXSUM];
    scd_pdl_wait();
    scd_pdl_trigger();
    const int b = blockIdx.y;
    AdSums S;
    S.part[0] = gxp_part + (size_t)b * stride; S.n[0] = n_part;
    S.part[1] = grd_part + (size_t)b * stride; S.n[1] = n_part;
    S.part[2] = gb_part + (size_t)b * stride;  S.n[2] = gp ? gb_n : 0;
    ad_sums(S, 3, slot);
    const float galpha = slot[0] - slot[1], gbeta = slot[2];
    const float alpha = s_alpha[b], pd = s_pd[b], rho = s_rho[b];
    const float beta = gp ? s_beta[b] : 0.f;
    const float gpd = -galpha * alpha / pd;
    if (blockIdx.x == 0 && threadIdx.x == 0) s_grho[b] = (gp ? -gbeta * beta / rho : 0.f) + galpha / pd;
    const size_t base = (size_t)b * numel;
    AD_LOOP(i) {
        const float pv = p[base + i], g1 = gr1[base + i];
        gd[base + i] = fmaf(gpd, pv, -alpha * g1);
        float t = fmaf(alpha, gx[base + i], gpd * d[base + i]);
        if (gp) t = fmaf(beta, gp[base + i], t);
        gptmp[base + i] = t;
    }
}

// ---- reverse: gr <- gr + gp + 2 grho r0 ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_bw_final_kernel(const float *__restrict__ gr, const float *__restrict__ gp, const float *__restrict__ r0,
                      const float *__restrict__ s_grho, float *__restrict__ out, int64_t numel)
{
    scd_pdl_wait();
    scd_pdl_trigger();
    const int b = blockIdx.y;
    const float two = 2.0f * s_grho[b];
    const size_t base = (size_t)b * numel;
    AD_LOOP(i) out[base + i] = gr[base + i] + gp[base + i] + two * r0[base + i];
}

// ---- reverse: grad_s = -(std_t/mean_t) * g_loss * v ----
__global__ void __launch_bounds__(AD_THREADS)
adapt_bw_tweedie_kernel(const float *__restrict__ v, const float *__restrict__ t, const float *__restrict__ abar, int n_table,
                        const float *__restrict__ g_loss, float *__restrict__ grad_s, int64_t numel)
{
    scd_pdl_wait();
    scd_pdl_trigger();
    const int b = blockIdx.y;
    long long idx = (long long)t[b] + 1;
    idx = idx < 0 ? 0 : (idx >= n_table ? n_table - 1 : idx);
    const float ab = abar[idx];
    const float coef = -__fsqrt_rn(__fsub_rn(1.0f, ab)) * __fdiv_rn(1.0f, __fsqrt_rn(ab)) * (g_loss ? g_loss[0] : 1.0f);
    const size_t base = (size_t)b * numel;
    AD_LOOP(i) grad_s[base + i] = coef * v[base + i];
}

// ------------------------------------------------------------- host side ---
struct AdLayout {
    size_t img, sino, K, stride;
    int nblk, nbp, res_blocks, tv_blocks;
    size_t off_q, off_pack, off_ax, off_res;
    size_t off_xhat0, off_b, off_x, off_r, off_p, off_d;       // r: K+1 images, p, d: K images
    size_t off_gx, off_gra, off_grb, off_gp, off_gptmp, off_gd, off_val;
    size_t off_part, off_respart, off_tvpart, off_scal;
    size_t total;
};

static int ad_blocks(const scd_geom *g, int batch)
{
    const int64_t numel = (int64_t)g->n0 * g->n1;
    int64_t nb = (2L * g->sm_count + batch - 1) / batch;
    const int64_t cap = (numel + AD_THREADS * 4 - 1) / (AD_THREADS * 4);
    if (nb > cap) nb = cap;
    if (nb > 64) nb = 64;
    if (nb < 1) nb = 1;
    return (int)nb;
}

static AdLayout ad_layout(const scd_geom *g, int batch, int n_iter)
{
    AdLayout L;
    L.img = (size_t)g->n0 * g->n1 * batch * 4;
    L.sino = (size_t)g->n_angles * g->n_det * batch * 4;
    L.K = (size_t)std::max(n_iter, 0);
    L.nblk = ad_blocks(g, batch);
    L.nbp = scd_bp_ctas_per_sample_max(g, batch);
    L.stride = (size_t)std::max(L.nblk, L.nbp);
    L.res_blocks = scd_residual_sq_blocks((int64_t)g->n_angles * g->n_det * batch);
    L.tv_blocks = scd_tv_blocks(g->n0, g->n1);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o += ad_align(bytes); return at; };
    L.off_q = take(scd_sino_il_bytes(g, batch));
    L.off_pack = take(scd_fp_scratch_need(g, batch));
    L.off_ax = take(L.sino); L.off_res = take(L.sino);
    L.off_xhat0 = take(L.img); L.off_b = take(L.img); L.off_x = take(L.img);
    L.off_r = take(L.img * (L.K + 1)); L.off_p = take(L.img * std::max<size_t>(L.K, 1)); L.off_d = take(L.img * std::max<size_t>(L.K, 1));
    L.off_gx = take(L.img); L.off_gra = take(L.img); L.off_grb = take(L.img); L.off_gp = take(L.img);
    L.off_gptmp = take(L.img); L.off_gd = take(L.img); L.off_val = take(L.img);
    L.off_part = take(6 * L.stride * batch * 4);
    L.off_respart = take((size_t)L.res_blocks * 4);
    L.off_tvpart = take((size_t)L.tv_blocks * batch * 4);
    L.off_scal = take((4 * std::max<size_t>(L.K, 1) + 1) * batch * 4);
    L.total = o;
    return L;
}

extern "C" size_t scd_adapt_workspace_bytes(const scd_geom_t *g, int batch, int n_iter)
{
    if (!g || batch <= 0 || n_iter < 0) return 0;
    return ad_layout(g, batch, n_iter).total;
}

namespace {
struct AdCtx {
    const scd_geom *g; AdLayout L; char *w; int batch; cudaStream_t st; float gs; int64_t numel; dim3 grid;
    const float *w_il;     // packed measurement weights of op or NULL
    float *img(size_t off, size_t k = 0) const { return (float *)(w + off + k * L.img); }
    float *part(int k) const { return (float *)(w + L.off_part) + (size_t)k * L.stride * batch; }
    float *scal(int which, size_t k) const { return (float *)(w + L.off_scal) + ((size_t)which * std::max<size_t>(L.K, 1) + k) * batch; }
    float *grho() const { return (float *)(w + L.off_scal) + 4 * std::max<size_t>(L.K, 1) * batch; }
    // out = c_acc*BP(A v) + c1*add1 + c2*add2 (+ dot partials): pack/interleave, march, backprojection
    int op(const float *v, float *out, float c_acc, const float *add1, float c1, const float *add2, float c2,
           float *out2, float *dot_part, int dot_with_add1) const
    {
        float *q = (float *)(w + L.off_q);
        int rc = scd_launch_fp(g, v, nullptr, q, batch, 0, g->n_angles, w + L.off_pack, scd_fp_scratch_need(g, batch), st, nullptr,
                               w_il);
        if (rc) return rc;
        BpEpilogue e;
        e.c_acc = c_acc; e.add1 = add1; e.c1 = c1; e.add2 = add2; e.c2 = c2; e.out2 = out2;
        e.dot_part = dot_part; e.dot_stride = (int)L.stride; e.dot_with_add1 = dot_with_add1;
        return scd_launch_bp_il(g, q, out, batch, 0, g->n_angles, e, st);
    }
};

int ad_setup(AdCtx &c, const scd_geom_t *g, int batch, int n_iter, int dc_type, void *work, size_t work_bytes, double gamma,
             void *stream, const char *who, const float *w_il)
{
    if (n_iter < 0 || dc_type < 0 || dc_type > 2) { scd_set_error("%s: bad n_iter / dc_type", who); return SCD_E_INVALID; }
    if (((uintptr_t)w_il & 127) != 0) { scd_set_error("%s: w_il must be 128-byte aligned", who); return SCD_E_INVALID; }
    c.w_il = w_il;
    if (((uintptr_t)work & 255) != 0) { scd_set_error("%s: workspace must be 256-byte aligned", who); return SCD_E_INVALID; }
    c.g = g; c.L = ad_layout(g, batch, dc_type == 0 ? n_iter : 0); c.w = (char *)work; c.batch = batch; c.st = (cudaStream_t)stream;
    if (work_bytes < c.L.total) {
        scd_set_error("%s: workspace too small (%zu < %zu bytes)", who, work_bytes, c.L.total);
        return SCD_E_WORKSPACE;
    }
    c.gs = (float)gamma * (float)g->adj_scale;
    c.numel = (int64_t)g->n0 * g->n1;
    c.grid = dim3(c.L.nblk, batch);
    if (batch > 65535) { scd_set_error("%s: batch too large", who); return SCD_E_INVALID; }
    return 0;
}
}  // namespace

#define AD_LAUNCH(kernel, ...)                                                                         \
    do {                                                                                               \
        SCD_CUDA(scd_launch_kernel(kernel, c.grid, dim3(AD_THREADS), 0, c.st, 0, __VA_ARGS__));        \
        SCD_LAUNCH_CHECK(#kernel);                                                                     \
    } while (0)

// dc_type: 0 = cg (n_iter iterations), 1 = one gradient step (xhat = xhat0 - gamma A*(A xhat0) + gamma atb), 2 = none
extern "C" int scd_adapt_fwd(const scd_geom_t *g, const float *x, const float *s, const float *atb, const float *y,
                             const float *t, const float *abar, int n_table, double gamma, int n_iter, int dc_type,
                             double tv_lambda, float *loss, float *xhat_out, int batch, void *work, size_t work_bytes,
                             void *stream)
{
    return scd_adapt_fwd_w(g, x, s, atb, y, nullptr, nullptr, t, abar, n_table, gamma, n_iter, dc_type, tv_lambda, loss,
                           xhat_out, batch, work, work_bytes, stream);
}

extern "C" int scd_adapt_fwd_w(const scd_geom_t *g, const float *x, const float *s, const float *atb, const float *y,
                               const float *w, const float *w_il, const float *t, const float *abar, int n_table,
                               double gamma, int n_iter, int dc_type, double tv_lambda, float *loss, float *xhat_out,
                               int batch, void *work, size_t work_bytes, void *stream)
{
    if (!w != !w_il) { scd_set_error("scd_adapt_fwd_w: give both w and w_il, or neither"); return SCD_E_INVALID; }
    if (!g || !x || !s || !y || !t || !abar || !loss || !work || (dc_type != 2 && !atb)) {
        scd_set_error("scd_adapt_fwd: null argument"); return SCD_E_INVALID;
    }
    if (batch <= 0) { scd_set_error("scd_adapt_fwd: empty batch"); return SCD_E_INVALID; }
    AdCtx c;
    int rc = ad_setup(c, g, batch, n_iter, dc_type, work, work_bytes, gamma, stream, "scd_adapt_fwd", w_il);
    if (rc) return rc;
    const AdLayout &L = c.L;
    const int K = (int)L.K, ps = (int)L.stride;
    float *xhat0 = c.img(L.off_xhat0), *b = c.img(L.off_b), *xk = c.img(L.off_x);
    const int nbp = scd_bp_ctas_per_sample(g, batch);
    if (nbp > ps) { scd_set_error("scd_adapt_fwd: partial-sum stride"); return SCD_E_INVALID; }
    // Tweedie (+ right-hand side of the data-consistency system)
    if ((rc = scd_launch_tweedie_rhs(x, s, atb, t, abar, n_table, (float)gamma, xhat0, dc_type == 2 ? nullptr : b, batch, c.numel, c.st))) return rc;
    const float *xhat = xhat0;
    if (dc_type == 1) {
        // xhat = xhat0 - gamma A*(A xhat0) + gamma atb
        if ((rc = c.op(xhat0, xk, -c.gs, xhat0, 1.f, atb, (float)gamma, nullptr, nullptr, 0))) return rc;
        xhat = xk;
    } else if (dc_type == 0 && K > 0) {
        float *rr_a = c.part(0), *rr_b = c.part(1), *pd = c.part(2);
        // r_0 = b - x_0 - gamma A*(A x_0);  p_0 = r_0;  rho_0 = |r_0|^2
        if ((rc = c.op(xhat0, c.img(L.off_r, 0), -c.gs, xhat0, -1.f, b, 1.f, c.img(L.off_p, 0), rr_a, 0))) return rc;
        SCD_CUDA(cudaMemcpyAsync(xk, xhat0, L.img, cudaMemcpyDeviceToDevice, c.st));
        float *rr_cur = rr_a, *rr_nxt = rr_b;
        int rr_n = nbp;
        for (int k = 0; k < K; ++k) {
            float *pk = c.img(L.off_p, k), *dk = c.img(L.off_d, k);
            if ((rc = c.op(pk, dk, c.gs, pk, 1.f, nullptr, 0.f, nullptr, pd, 1))) return rc;          // d = op(p), <p,d>
            AD_LAUNCH(adapt_update_kernel, xk, (const float *)c.img(L.off_r, k), c.img(L.off_r, k + 1), (const float *)pk,
                      (const float *)dk, (const float *)rr_cur, rr_n, (const float *)pd, nbp, ps, rr_nxt,
                      c.scal(0, k), c.scal(2, k), c.scal(3, k), c.numel);
            if (k + 1 < K)
                AD_LAUNCH(adapt_direction_kernel, (const float *)c.img(L.off_r, k + 1), (const float *)pk, c.img(L.off_p, k + 1),
                          (const float *)rr_nxt, L.nblk, ps, (const float *)c.scal(2, k), c.scal(1, k), c.numel);
            std::swap(rr_cur, rr_nxt);
            rr_n = L.nblk;
        }
        xhat = xk;
    }
    if (xhat != xk) SCD_CUDA(cudaMemcpyAsync(xk, xhat, L.img, cudaMemcpyDeviceToDevice, c.st));   // the sweep reads xhat at off_x
    if (xhat_out) SCD_CUDA(cudaMemcpyAsync(xhat_out, xhat, L.img, cudaMemcpyDeviceToDevice, c.st));
    // loss = mean((A xhat - y)^2) + lambda tv(xhat)
    float *ax = (float *)(c.w + L.off_ax), *res = (float *)(c.w + L.off_res);
    float *respart = (float *)(c.w + L.off_respart), *tvpart = (float *)(c.w + L.off_tvpart);
    if ((rc = scd_launch_fp(g, xk, ax, nullptr, batch, 0, g->n_angles, c.w + L.off_pack, scd_fp_scratch_need(g, batch), c.st, nullptr))) return rc;
    const int64_t n_res = (int64_t)g->n_angles * g->n_det * batch;
    if ((rc = scd_launch_residual_sq(ax, y, w, res, respart, n_res, c.st))) return rc;
    if ((rc = scd_tv_loss(xk, tvpart, batch, g->n0, g->n1, stream))) return rc;
    SCD_CUDA(scd_launch_kernel(adapt_loss_kernel, dim3(1), dim3(AD_THREADS), 0, c.st, 0, (const float *)respart, L.res_blocks,
                               (const float *)tvpart, L.tv_blocks * batch, 1.0f / (float)n_res, (float)tv_lambda, loss));
    SCD_LAUNCH_CHECK("adapt_loss_kernel");
    return 0;
}

extern "C" int scd_adapt_bwd(const scd_geom_t *g, const float *grad_loss, const float *t, const float *abar, int n_table,
                             double gamma, int n_iter, int dc_type, double tv_lambda, double trafo_grad_scale,
                             float *grad_s, int batch, void *work, size_t work_bytes, void *stream)
{
    return scd_adapt_bwd_w(g, grad_loss, nullptr, t, abar, n_table, gamma, n_iter, dc_type, tv_lambda, trafo_grad_scale,
                           grad_s, batch, work, work_bytes, stream);
}

extern "C" int scd_adapt_bwd_w(const scd_geom_t *g, const float *grad_loss, const float *w_il, const float *t,
                               const float *abar, int n_table, double gamma, int n_iter, int dc_type, double tv_lambda,
                               double trafo_grad_scale, float *grad_s, int batch, void *work, size_t work_bytes,
                               void *stream)
{
    if (!g || !t || !abar || !grad_s || !work) { scd_set_error("scd_adapt_bwd: null argument"); return SCD_E_INVALID; }
    if (batch <= 0) { scd_set_error("scd_adapt_bwd: empty batch"); return SCD_E_INVALID; }
    AdCtx c;
    int rc = ad_setup(c, g, batch, n_iter, dc_type, work, work_bytes, gamma, stream, "scd_adapt_bwd", w_il);
    if (rc) return rc;
    const AdLayout &L = c.L;
    const int K = (int)L.K, ps = (int)L.stride;
    float *xk = c.img(L.off_x), *gx = c.img(L.off_gx), *val = c.img(L.off_val);
    float *res = (float *)(c.w + L.off_res);
    // gx = d loss / d xhat = (2/N) A*(res)/c_w + lambda d tv/d xhat     (gradient of A under ODL's pairing; res is
    // W (A xhat - y) when the forward call was weighted)
    float *tvg = c.img(L.off_gd);                                        // free until the sweep needs gd
    if ((rc = scd_tv_grad(xk, tvg, batch, g->n0, g->n1, stream))) return rc;
    const double n_res = (double)g->n_angles * g->n_det * batch;
    BpEpilogue e;
    e.c_acc = (float)(2.0 / n_res * trafo_grad_scale);                   // trafo_grad_scale = adj_scale / c_w
    e.add1 = tvg; e.c1 = (float)tv_lambda; e.add2 = nullptr; e.c2 = 0.f;
    e.out2 = nullptr; e.dot_part = nullptr; e.dot_stride = 0; e.dot_with_add1 = 0;
    // the transpose of A carries no view weights (a weighted geometry weights A* only)
    if ((rc = scd_launch_bp(g, res, gx, batch, 0, g->n_angles, e, c.w + L.off_q, scd_sino_il_bytes(g, batch), c.st,
                            false))) return rc;
    const float *gfinal = gx;                                            // d loss / d xhat0
    if (dc_type == 1) {
        // xhat = xhat0 - gamma A*(A xhat0) + const: adjoint gx - gamma A*(A gx)
        if ((rc = c.op(gx, val, -c.gs, gx, 1.f, nullptr, 0.f, nullptr, nullptr, 0))) return rc;
        gfinal = val;
    } else if (dc_type == 0 && K > 0) {
        float *gb = c.part(3), *gxp = c.part(4), *grd = c.part(5);
        float *gr_cur = nullptr, *gr_nxt = c.img(L.off_gra), *gr_other = c.img(L.off_grb);
        float *gp = nullptr, *gp_buf = c.img(L.off_gp), *gptmp = c.img(L.off_gptmp), *gd = c.img(L.off_gd);
        for (int k = K - 1; k >= 0; --k) {
            const float *pk = c.img(L.off_p, k), *dk = c.img(L.off_d, k), *r1 = c.img(L.off_r, k + 1);
            if (gp) AD_LAUNCH(adapt_dot_kernel, (const float *)gp, pk, gb, ps, c.numel);
            AD_LAUNCH(adapt_bw_residual_kernel, (const float *)gr_cur, (const float *)gp, r1, (const float *)gx, pk, dk,
                      (const float *)gb, L.nblk, ps, (const float *)(gp ? c.grho() : nullptr), (const float *)c.scal(2, k),
                      gr_nxt, gxp, grd, c.numel);
            AD_LAUNCH(adapt_bw_direction_kernel, (const float *)gp, (const float *)gx, pk, dk, (const float *)gr_nxt,
                      (const float *)gxp, (const float *)grd, L.nblk, (const float *)gb, L.nblk, ps,
                      (const float *)c.scal(0, k), (const float *)c.scal(1, k), (const float *)c.scal(2, k),
                      (const float *)c.scal(3, k), c.grho(), gd, gptmp, c.numel);
            // gp <- gptmp + op(gd) = gptmp + gd + gamma A*(A gd)
            if ((rc = c.op(gd, gp_buf, c.gs, gd, 1.f, gptmp, 1.f, nullptr, nullptr, 0))) return rc;
            gp = gp_buf;
            gr_cur = gr_nxt;
            std::swap(gr_nxt, gr_other);
        }
        // gr <- gr + gp + 2 grho r_0;  d loss/d xhat0 = gx - gamma A*(A gr)
        AD_LAUNCH(adapt_bw_final_kernel, (const float *)gr_cur, (const float *)gp, (const float *)c.img(L.off_r, 0),
                  (const float *)c.grho(), gr_nxt, c.numel);
        if ((rc = c.op(gr_nxt, val, -c.gs, gx, 1.f, nullptr, 0.f, nullptr, nullptr, 0))) return rc;
        gfinal = val;
    }
    AD_LAUNCH(adapt_bw_tweedie_kernel, gfinal, t, abar, n_table, grad_loss, grad_s, c.numel);
    return 0;
}
