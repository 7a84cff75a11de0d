// Batched CG on (I + gamma A*A) x = rhs and the fused DDS data-consistency step,
// expressed as a fixed launch sequence on the caller's stream (CUDA-graph
// capturable: no allocation, no synchronisation, no host<->device traffic).
//
// Follows reference src/utils/cg.py:11-39 step by step:
//   r = rhs - op(x); p = r; rr = ||r||^2
//   repeat n_iter: d = op(p); alpha = rr/<p,d>; x += alpha p; r -= alpha d;
//                  rr' = ||r||^2; beta = rr'/rr; p = r + beta p
// with op(v) = v + gamma*A*(A v) (src/samplers/utils.py:188-189).
// Groups of >= 4 samples (batch >= 3) and batch 1 (whose interleaved image is the reference layout): the vectors
// x, r, p, d, b are sample-interleaved images for the whole
// solve (il_ops.cu) and an iteration is THREE launches with no packed copy of anything:
//   fp_march   q = A r + beta q          (q_k = A p_k with p_k = r_k + beta p_{k-1}: the projector reads r through
//                                         tensor copies, its output phase carries the recurrence and forms beta)
//   bp_tile    p = r + beta p;  d = p + gamma A*(q);  partial <p,d>      (all in the backprojector's epilogue)
//   cg_update_xr_il   alpha = rr/<p,d>;  x += alpha p;  r -= alpha d;  partial ||r||^2
// Batches of 2 samples (and batch 1 when n1 is not a multiple of 4) keep the packed-copy sequence:
// fp_packq (p-update fused), fp_march, bp_tile(+axpy,+<p,d>), cg_update_xr (the last p-update is skipped).
// Measurement weights (the _w entry points): op(v) = v + gamma*A*(W A v).  W, packed once into the layout of q
// (scd_sino_weights_pack), multiplies the projector's interleaved output before the recurrence q = A r + beta q;
// both are linear, so the recurrence stays exact.  No other launch changes.
#include "scd_internal.cuh"
#include <algorithm>
#include <cstring>

struct CgLayout {
    size_t img, sino, part_stride;
    size_t off_q, off_r, off_p, off_d, off_b, off_xh, off_part, off_pack, pack_bytes, total;
    // interleaved-state solve (same buffer, other carving): five il images, partial sums, beta
    size_t il_bytes, il_q, il_x, il_r, il_p, il_d, il_b, il_part, il_beta, il_total;
};

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static CgLayout cg_layout(const scd_geom *g, int batch)
{
    CgLayout L;
    L.img = (size_t)g->n0 * g->n1;
    L.sino = (size_t)g->n_angles * g->n_det;
    const int nbp = scd_bp_ctas_per_sample_max(g, batch);
    const int nvec = scd_vec_blocks_per_sample((int64_t)L.img, batch);
    L.part_stride = (size_t)std::max(std::max(nbp, nvec), scd_il_vec_blocks(g, batch));
    size_t o = 0;
    // q = A p lives in the sample-interleaved layout the backprojector stages from
    L.off_q = o;  o += align256(scd_sino_il_bytes(g, batch));
    L.off_r = o;  o += align256(L.img * batch * 4);
    L.off_p = o;  o += align256(L.img * batch * 4);
    L.off_d = o;  o += align256(L.img * batch * 4);
    L.off_b = o;  o += align256(L.img * batch * 4);    // rhs of the fused step
    L.off_xh = o; o += align256(L.img * batch * 4);    // CG iterate of the fused step
    L.off_part = o; o += align256(3 * L.part_stride * batch * 4);
    L.pack_bytes = scd_fp_scratch_need(g, batch);
    L.off_pack = o; o += align256(L.pack_bytes);
    L.total = o;
    // il carving
    L.il_bytes = align256(scd_il_image_bytes(g, batch));
    o = 0;
    L.il_q = o; o += align256(scd_sino_il_bytes(g, batch));
    L.il_x = o; o += L.il_bytes;
    L.il_r = o; o += L.il_bytes;
    L.il_p = o; o += L.il_bytes;
    L.il_d = o; o += L.il_bytes;
    L.il_b = o; o += L.il_bytes;
    L.il_part = o; o += align256(3 * L.part_stride * batch * 4);
    L.il_beta = o; o += align256((size_t)batch * 4);
    L.il_total = o;
    L.total = std::max(L.total, L.il_total);
    return L;
}

extern "C" size_t scd_cg_workspace_bytes(const scd_geom_t *g, int batch)
{
    if (!g || batch <= 0) return 0;
    return cg_layout(g, batch).total;
}

int scd_cg_run(const scd_geom *g, const float *x_in, float *x, const float *rhs, float gamma,
               int n_iter, int batch, void *work, size_t work_bytes, cudaStream_t st,
               const FpPrologue *first, const float *w_il)
{
    if (!g || !x || !x_in || !rhs || !work) { scd_set_error("scd_cg: null argument"); return SCD_E_INVALID; }
    if (batch <= 0) return 0;
    if (n_iter < 0) { scd_set_error("scd_cg: n_iter < 0"); return SCD_E_INVALID; }
    if (((uintptr_t)work & 255) != 0) { scd_set_error("scd_cg: workspace must be 256-byte aligned"); return SCD_E_INVALID; }
    const CgLayout L = cg_layout(g, batch);
    if (work_bytes < L.total) {
        scd_set_error("scd_cg: workspace too small (%zu < %zu bytes)", work_bytes, L.total);
        return SCD_E_WORKSPACE;
    }
    char *w = (char *)work;
    float *q = (float *)(w + L.off_q), *r = (float *)(w + L.off_r);
    float *p = (float *)(w + L.off_p), *d = (float *)(w + L.off_d);
    float *part = (float *)(w + L.off_part);
    void *pack = (void *)(w + L.off_pack);
    const int ps = (int)L.part_stride;
    float *rr_a = part, *rr_b = part + (size_t)ps * batch, *pd = part + 2 * (size_t)ps * batch;
    const int nbp = scd_bp_ctas_per_sample(g, batch);
    const int nvec = scd_vec_blocks_per_sample((int64_t)L.img, batch);
    if ((size_t)nbp > L.part_stride || (size_t)nvec > L.part_stride) {
        scd_set_error("scd_cg: %d partial sums per sample exceed the workspace stride %zu", std::max(nbp, nvec), L.part_stride);
        return SCD_E_INVALID;
    }
    const float gs = gamma * (float)g->adj_scale;
    int rc;
    float *q_user = nullptr, *q_il = q;            // q = A p: interleaved layout only
    auto bp = [&](float *out, const BpEpilogue &e) {
        return scd_launch_bp_il(g, q, out, batch, 0, g->n_angles, e, st);
    };

    // r = rhs - x - gamma A*(A x);  p = r;  rr = ||r||^2
    // (the Tweedie step that produces x_in and rhs may be fused into this projection's pack pass)
    if ((rc = scd_launch_fp(g, x_in, q_user, q_il, batch, 0, g->n_angles, pack, L.pack_bytes, st, first, w_il))) return rc;
    BpEpilogue e0;
    e0.c_acc = -gs; e0.add1 = x_in; e0.c1 = -1.f; e0.add2 = rhs; e0.c2 = 1.f;
    e0.out2 = p; e0.dot_part = rr_a; e0.dot_stride = ps; e0.dot_with_add1 = 0;
    if ((rc = bp(r, e0))) return rc;
    float *rr_old = rr_a, *rr_new = rr_b;
    int rr_old_n = nbp, rr_prev_n = nbp;

    for (int it = 0; it < n_iter; ++it) {
        // p = r + beta p (fused into the pack pass, it >= 1);  d = p + gamma A*(A p);  pd = <p,d>
        FpPrologue up;
        memset(&up, 0, sizeof(up));
        if (it > 0) {
            up.mode = 1; up.p = p; up.r = r;
            up.rr_new_part = rr_old; up.rr_new_n = rr_old_n;        // after the swap below: newest ||r||^2
            up.rr_old_part = rr_new; up.rr_old_n = rr_prev_n;       // and the one before it
            up.part_stride = ps;
        }
        if ((rc = scd_launch_fp(g, p, q_user, q_il, batch, 0, g->n_angles, pack, L.pack_bytes, st, it > 0 ? &up : nullptr,
                                w_il))) return rc;
        BpEpilogue e1;
        e1.c_acc = gs; e1.add1 = p; e1.c1 = 1.f; e1.add2 = nullptr; e1.c2 = 0.f;
        e1.out2 = nullptr; e1.dot_part = pd; e1.dot_stride = ps; e1.dot_with_add1 = 1;
        if ((rc = bp(d, e1))) return rc;
        // the first update reads the start iterate and writes the result buffer
        if ((rc = scd_launch_cg_update_xr(it == 0 ? x_in : x, x, r, p, d, rr_old, rr_old_n, pd, nbp, ps, rr_new,
                                          batch, (int64_t)L.img, st))) return rc;
        rr_prev_n = rr_old_n;
        std::swap(rr_old, rr_new);
        rr_old_n = nvec;
    }
    if (n_iter == 0 && x != x_in)
        SCD_CUDA(cudaMemcpyAsync(x, x_in, L.img * batch * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

// ---- interleaved-state solve ---------------------------------------------------------------------
// x_in: start iterate (read only), x: result (may be x_in), b: right-hand side -- all il images; q, r, p, d, the
// partial sums and beta live in the workspace.  With one sample per group (batch 1) an il image IS the reference
// layout, so the caller's tensors are used directly and the update kernel is the reference-layout one.
static int cg_run_il(const scd_geom *g, const CgLayout &L, const float *x_in, float *x, const float *b, float gamma,
                     int n_iter, int batch, char *w, cudaStream_t st, const float *w_il)
{
    float *q = (float *)(w + L.il_q), *r = (float *)(w + L.il_r);
    float *p = (float *)(w + L.il_p), *d = (float *)(w + L.il_d);
    float *part = (float *)(w + L.il_part), *beta = (float *)(w + L.il_beta);
    const int ps = (int)L.part_stride;
    float *rr_a = part, *rr_b = part + (size_t)ps * batch, *pd = part + 2 * (size_t)ps * batch;
    const int SB = scd_group_samples(g, batch);
    const int nbp = scd_bp_ctas_per_sample(g, batch);
    const int nvec = SB == 1 ? scd_vec_blocks_per_sample((int64_t)L.img, batch) : scd_il_vec_blocks(g, batch);
    if (nbp > ps || nvec > ps) {
        scd_set_error("scd_cg: %d partial sums per sample exceed the workspace stride %d", std::max(nbp, nvec), ps);
        return SCD_E_INVALID;
    }
    const float gs = gamma * (float)g->adj_scale;
    const int na = g->n_angles;
    int rc;
    // r = b - x - gamma A*(A x);  rr = ||r||^2
    if ((rc = scd_launch_fp_ilimg(g, x_in, nullptr, q, batch, 0, na, st, nullptr, w_il))) return rc;
    BpEpilogue e0;
    e0.il = 1; e0.mode = 0;
    e0.c_acc = -gs; e0.add1 = x_in; e0.c1 = -1.f; e0.add2 = b; e0.c2 = 1.f;
    e0.out2 = nullptr; e0.dot_part = rr_a; e0.dot_stride = ps; e0.dot_with_add1 = 0;
    if ((rc = scd_launch_bp_il(g, q, r, batch, 0, na, e0, st))) return rc;
    float *rr_new = rr_a, *rr_old = rr_b;          // newest ||r||^2 partials / the ones before
    int rr_new_n = nbp, rr_old_n = 0;
    for (int it = 0; it < n_iter; ++it) {
        // q = A r + beta q   (= A p with p = r + beta p; first iteration: p = r)
        FpAccumulate acc;
        acc.rr_new_part = rr_new; acc.rr_new_n = rr_new_n; acc.rr_old_part = rr_old; acc.rr_old_n = rr_old_n;
        acc.part_stride = ps; acc.beta_out = beta;
        if ((rc = scd_launch_fp_ilimg(g, r, nullptr, q, batch, 0, na, st, it > 0 ? &acc : nullptr, w_il))) return rc;
        // p = r + beta p;  d = p + gamma A*(q);  pd = <p,d>
        BpEpilogue e1;
        e1.il = 1; e1.mode = 1;
        e1.c_acc = gs; e1.add1 = r; e1.c1 = 1.f; e1.add2 = it > 0 ? p : nullptr; e1.c2 = 0.f;
        e1.beta = it > 0 ? beta : nullptr;
        e1.out2 = p; e1.dot_part = pd; e1.dot_stride = ps; e1.dot_with_add1 = 0;
        if ((rc = scd_launch_bp_il(g, q, d, batch, 0, na, e1, st))) return rc;
        // alpha = rr/pd;  x += alpha p;  r -= alpha d;  rr' = ||r||^2   (the first update reads the start iterate)
        const float *xi = it == 0 ? x_in : x;
        if (SB == 1)
            rc = scd_launch_cg_update_xr(xi, x, r, p, d, rr_new, rr_new_n, pd, nbp, ps, rr_old, batch, (int64_t)L.img, st);
        else
            rc = scd_launch_cg_update_xr_il(g, xi, x, r, p, d, rr_new, rr_new_n, pd, nbp, ps, rr_old, batch, st);
        if (rc) return rc;
        std::swap(rr_new, rr_old);                 // the kernel wrote the newest partials into the older array
        rr_old_n = rr_new_n;
        rr_new_n = nvec;
    }
    return 0;
}

static int cg_check(const scd_geom *g, const void *work, size_t work_bytes, int n_iter, const CgLayout &L, const char *who)
{
    if (n_iter < 0) { scd_set_error("%s: n_iter < 0", who); return SCD_E_INVALID; }
    if (((uintptr_t)work & 255) != 0) { scd_set_error("%s: workspace must be 256-byte aligned", who); return SCD_E_INVALID; }
    if (work_bytes < L.total) {
        scd_set_error("%s: workspace too small (%zu < %zu bytes)", who, work_bytes, L.total);
        return SCD_E_WORKSPACE;
    }
    (void)g;
    return 0;
}

// packed measurement weights: 128-byte aligned like every sino_il buffer (the projector reads them as vectors)
static int w_il_ok(const float *w_il, const char *who)
{
    if (((uintptr_t)w_il & 127) != 0) { scd_set_error("%s: w_il must be 128-byte aligned", who); return SCD_E_INVALID; }
    return 0;
}

extern "C" int scd_sino_weights_pack(const scd_geom_t *g, const float *w, float *w_il, int batch, void *stream)
{
    if (!g || !w || !w_il) { scd_set_error("scd_sino_weights_pack: null argument"); return SCD_E_INVALID; }
    if (batch <= 0) { scd_set_error("scd_sino_weights_pack: empty batch"); return SCD_E_INVALID; }
    int rc = w_il_ok(w_il, "scd_sino_weights_pack");
    if (rc) return rc;
    // the view weights of A* are applied by the projector's output scale: the pack must not apply them again
    return scd_launch_sino_pack(g, w, w_il, batch, 0, g->n_angles, (cudaStream_t)stream, false);
}

extern "C" int scd_cg(const scd_geom_t *g, float *x, const float *rhs, double gamma, int n_iter,
                      int batch, void *work, size_t work_bytes, void *stream)
{
    return scd_cg_w(g, x, rhs, nullptr, gamma, n_iter, batch, work, work_bytes, stream);
}

extern "C" int scd_cg_w(const scd_geom_t *g, float *x, const float *rhs, const float *w_il, double gamma, int n_iter,
                        int batch, void *work, size_t work_bytes, void *stream)
{
    if (w_il && w_il_ok(w_il, "scd_cg_w")) return SCD_E_INVALID;
    if (g && x && rhs && work && batch > 0 && scd_il_image_ok(g, batch)) {
        const CgLayout L = cg_layout(g, batch);
        int rc = cg_check(g, work, work_bytes, n_iter, L, "scd_cg");
        if (rc) return rc;
        if (n_iter == 0) return 0;                // the result is the start iterate (x is updated in place)
        char *w = (char *)work;
        cudaStream_t st = (cudaStream_t)stream;
        if (scd_group_samples(g, batch) == 1 && (((uintptr_t)x | (uintptr_t)rhs) & 15) == 0)
            return cg_run_il(g, L, x, x, rhs, (float)gamma, n_iter, batch, w, st, w_il);      // the layouts coincide: in place
        float *xi = (float *)(w + L.il_x), *bi = (float *)(w + L.il_b);
        if ((rc = scd_launch_il_pack(g, x, xi, rhs, bi, batch, st))) return rc;
        if ((rc = cg_run_il(g, L, xi, xi, bi, (float)gamma, n_iter, batch, w, st, w_il))) return rc;
        return scd_launch_il_unpack(g, xi, x, batch, st);
    }
    return scd_cg_run(g, x, x, rhs, (float)gamma, n_iter, batch, work, work_bytes, (cudaStream_t)stream, nullptr, w_il);
}

extern "C" size_t scd_fp_scratch_bytes(const scd_geom_t *g, int batch)
{
    return scd_fp_scratch_need(g, batch);
}

extern "C" int scd_fp(const scd_geom_t *g, const float *img, float *sino, int batch,
                      int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes, void *stream)
{
    return scd_launch_fp(g, img, sino, nullptr, batch, angle_lo, angle_hi, scratch, scratch_bytes, (cudaStream_t)stream);
}

// ---- operators on the sample-interleaved sinogram (the form A*A is composed in) ----
extern "C" size_t scd_sino_il_buffer_bytes(const scd_geom_t *g, int batch)
{
    return scd_sino_il_bytes(g, batch);
}

extern "C" int scd_fp_il(const scd_geom_t *g, const float *img, float *sino_il, int batch,
                         int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes, void *stream)
{
    return scd_fp_il_w(g, img, sino_il, nullptr, batch, angle_lo, angle_hi, scratch, scratch_bytes, stream);
}

extern "C" int scd_fp_il_w(const scd_geom_t *g, const float *img, float *sino_il, const float *w_il, int batch,
                           int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes, void *stream)
{
    if (((uintptr_t)sino_il & 127) != 0) { scd_set_error("scd_fp_il: sino_il must be 128-byte aligned"); return SCD_E_INVALID; }
    if (w_il && w_il_ok(w_il, "scd_fp_il_w")) return SCD_E_INVALID;
    return scd_launch_fp(g, img, nullptr, sino_il, batch, angle_lo, angle_hi, scratch, scratch_bytes, (cudaStream_t)stream,
                         nullptr, w_il);
}

extern "C" int scd_bp_il(const scd_geom_t *g, const float *sino_il, float *out, int batch,
                         int angle_lo, int angle_hi, float c_acc, const float *addend, float c_add,
                         void *stream)
{
    if (g && batch == 0) return 0;
    if (!g || !sino_il || !out) { scd_set_error("scd_bp_il: null argument"); return SCD_E_INVALID; }
    if (((uintptr_t)sino_il & 127) != 0) { scd_set_error("scd_bp_il: sino_il must be 128-byte aligned"); return SCD_E_INVALID; }
    if (batch < 0 || angle_lo < 0 || angle_hi > g->n_angles || angle_lo > angle_hi) {
        scd_set_error("scd_bp_il: bad batch/angle range"); return SCD_E_INVALID;
    }
    BpEpilogue e;
    e.c_acc = c_acc; e.add1 = addend; e.c1 = c_add; e.add2 = nullptr; e.c2 = 0.f;
    e.out2 = nullptr; e.dot_part = nullptr; e.dot_stride = 0; e.dot_with_add1 = 0;
    return scd_launch_bp_il(g, sino_il, out, batch, angle_lo, angle_hi, e, (cudaStream_t)stream);
}

// ---- sample-interleaved images at the ABI (callers that keep their vectors in the library's layout) ----
extern "C" size_t scd_img_il_bytes(const scd_geom_t *g, int batch)
{
    if (!g || batch <= 0 || !scd_il_image_ok(g, batch)) return 0;
    return scd_il_image_bytes(g, batch);
}

static int il_args_ok(const scd_geom_t *g, const void *a, const void *b, int batch, const char *who)
{
    if (!g || !a || !b) { scd_set_error("%s: null argument", who); return SCD_E_INVALID; }
    if (batch < 0) { scd_set_error("%s: negative batch", who); return SCD_E_INVALID; }
    if (batch > 0 && !scd_il_image_ok(g, batch)) {
        scd_set_error("%s: batches of %d sample(s) have no interleaved-image form (scd_img_il_bytes returns 0)", who, batch);
        return SCD_E_INVALID;
    }
    return 0;
}

extern "C" int scd_img_il_pack(const scd_geom_t *g, const float *img, float *img_il, int batch, void *stream)
{
    int rc = il_args_ok(g, img, img_il, batch, "scd_img_il_pack");
    if (rc || batch == 0) return rc;
    if (((uintptr_t)img_il & 127) != 0) { scd_set_error("scd_img_il_pack: img_il must be 128-byte aligned"); return SCD_E_INVALID; }
    return scd_launch_il_pack(g, img, img_il, nullptr, nullptr, batch, (cudaStream_t)stream);
}

extern "C" int scd_img_il_unpack(const scd_geom_t *g, const float *img_il, float *img, int batch, void *stream)
{
    int rc = il_args_ok(g, img_il, img, batch, "scd_img_il_unpack");
    if (rc || batch == 0) return rc;
    return scd_launch_il_unpack(g, img_il, img, batch, (cudaStream_t)stream);
}

extern "C" int scd_fp_ilimg(const scd_geom_t *g, const float *img_il, float *sino_il, int batch,
                            int angle_lo, int angle_hi, void *stream)
{
    return scd_fp_ilimg_w(g, img_il, sino_il, nullptr, batch, angle_lo, angle_hi, stream);
}

extern "C" int scd_fp_ilimg_w(const scd_geom_t *g, const float *img_il, float *sino_il, const float *w_il, int batch,
                              int angle_lo, int angle_hi, void *stream)
{
    int rc = il_args_ok(g, img_il, sino_il, batch, "scd_fp_ilimg");
    if (rc || batch == 0) return rc;
    if (((uintptr_t)sino_il & 127) != 0) { scd_set_error("scd_fp_ilimg: sino_il must be 128-byte aligned"); return SCD_E_INVALID; }
    if (w_il && w_il_ok(w_il, "scd_fp_ilimg_w")) return SCD_E_INVALID;
    return scd_launch_fp_ilimg(g, img_il, nullptr, sino_il, batch, angle_lo, angle_hi, (cudaStream_t)stream, nullptr, w_il);
}

extern "C" int scd_bp_ilimg(const scd_geom_t *g, const float *sino_il, float *out_il, int batch,
                            int angle_lo, int angle_hi, float c_acc, const float *addend_il, float c_add, void *stream)
{
    int rc = il_args_ok(g, sino_il, out_il, batch, "scd_bp_ilimg");
    if (rc || batch == 0) return rc;
    if (((uintptr_t)sino_il & 127) != 0 || ((uintptr_t)out_il & 15) != 0 || ((uintptr_t)addend_il & 15) != 0) {
        scd_set_error("scd_bp_ilimg: misaligned buffer"); return SCD_E_INVALID;
    }
    if (angle_lo < 0 || angle_hi > g->n_angles || angle_lo > angle_hi) { scd_set_error("scd_bp_ilimg: bad angle range"); return SCD_E_INVALID; }
    BpEpilogue e;
    e.il = 1; e.mode = 0;
    e.c_acc = c_acc; e.add1 = addend_il; e.c1 = c_add; e.add2 = nullptr; e.c2 = 0.f;
    e.out2 = nullptr; e.dot_part = nullptr; e.dot_stride = 0; e.dot_with_add1 = 0;
    return scd_launch_bp_il(g, sino_il, out_il, batch, angle_lo, angle_hi, e, (cudaStream_t)stream);
}

extern "C" size_t scd_bp_scratch_bytes(const scd_geom_t *g, int batch)
{
    return scd_sino_il_bytes(g, batch);
}

extern "C" int scd_bp(const scd_geom_t *g, const float *sino, float *out, int batch,
                      int angle_lo, int angle_hi, float c_acc, const float *addend, float c_add,
                      void *scratch, size_t scratch_bytes, void *stream)
{
    BpEpilogue e;
    e.c_acc = c_acc; e.add1 = addend; e.c1 = c_add; e.add2 = nullptr; e.c2 = 0.f;
    e.out2 = nullptr; e.dot_part = nullptr; e.dot_stride = 0; e.dot_with_add1 = 0;
    return scd_launch_bp(g, sino, out, batch, angle_lo, angle_hi, e, scratch, scratch_bytes, (cudaStream_t)stream);
}

extern "C" int scd_tweedie_rhs(const float *x, const float *s, const float *atb, const float *t,
                               const float *abar, int n_table, double gamma, float *xhat0,
                               float *b, int batch, int64_t numel, void *stream)
{
    if (!x || !s || !t || !abar || !xhat0 || (b && !atb)) {
        scd_set_error("scd_tweedie_rhs: null argument"); return SCD_E_INVALID;
    }
    if (n_table < 1) { scd_set_error("scd_tweedie_rhs: empty alpha-bar table"); return SCD_E_INVALID; }
    return scd_launch_tweedie_rhs(x, s, atb, t, abar, n_table, (float)gamma, xhat0, b, batch, numel,
                                  (cudaStream_t)stream);
}

extern "C" int scd_ddim(const float *xhat, const float *s, const float *eps, const float *t,
                        const float *t_prev, const float *abar, int n_table, double eta, float *out,
                        int batch, int64_t numel, void *stream)
{
    if (!xhat || !s || !eps || !t || !t_prev || !abar || !out) {
        scd_set_error("scd_ddim: null argument"); return SCD_E_INVALID;
    }
    if (n_table < 1) { scd_set_error("scd_ddim: empty alpha-bar table"); return SCD_E_INVALID; }
    // `tbeta.pow(2)*eta**2`: eta**2 is evaluated in Python (fp64) and then rounded
    return scd_launch_ddim(xhat, s, eps, t, t_prev, abar, n_table, (float)eta, (float)(eta * eta), out,
                           batch, numel, (cudaStream_t)stream);
}

extern "C" int scd_dds_step(const scd_geom_t *g, const float *x, const float *s, const float *atb,
                            const float *eps, const float *t, const float *t_prev,
                            const float *abar, int n_table, double gamma, double eta, int n_iter,
                            float *x_next, float *xhat0, int batch, void *work, size_t work_bytes,
                            void *stream)
{
    return scd_dds_step_w(g, x, s, atb, nullptr, eps, t, t_prev, abar, n_table, gamma, eta, n_iter, x_next, xhat0, batch,
                          work, work_bytes, stream);
}

extern "C" int scd_dds_step_w(const scd_geom_t *g, const float *x, const float *s, const float *atb, const float *w_il,
                              const float *eps, const float *t, const float *t_prev,
                              const float *abar, int n_table, double gamma, double eta, int n_iter,
                              float *x_next, float *xhat0, int batch, void *work, size_t work_bytes,
                              void *stream)
{
    if (w_il && w_il_ok(w_il, "scd_dds_step_w")) return SCD_E_INVALID;
    if (!g || !x || !s || !atb || !eps || !t || !t_prev || !abar || !x_next || !xhat0 || !work) {
        scd_set_error("scd_dds_step: null argument"); return SCD_E_INVALID;
    }
    if (batch <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const CgLayout L = cg_layout(g, batch);
    if (work_bytes < L.total) {
        scd_set_error("scd_dds_step: workspace too small (%zu < %zu bytes)", work_bytes, L.total);
        return SCD_E_WORKSPACE;
    }
    char *w = (char *)work;
    int rc;
    if (scd_il_image_ok(g, batch)) {
        // Tweedie writes xhat0 for the caller and the CG start iterate / right-hand side as il images; DDIM reads
        // the CG result in that layout: 1 + 2 + 3*n_iter + 1 launches
        if ((rc = cg_check(g, work, work_bytes, n_iter, L, "scd_dds_step"))) return rc;
        float *xi = (float *)(w + L.il_x), *bi = (float *)(w + L.il_b);
        if (scd_group_samples(g, batch) == 1) {
            // one sample per group: il image = reference layout.  xhat0 (returned to the caller) is the start iterate,
            // read only; the first update writes the iterate into the workspace
            if ((rc = scd_launch_tweedie_rhs(x, s, atb, t, abar, n_table, (float)gamma, xhat0, bi, batch, (int64_t)L.img, st))) return rc;
            if (n_iter > 0 && (rc = cg_run_il(g, L, xhat0, xi, bi, (float)gamma, n_iter, batch, w, st, w_il))) return rc;
            return scd_launch_ddim(n_iter > 0 ? xi : xhat0, s, eps, t, t_prev, abar, n_table, (float)eta, (float)(eta * eta),
                                   x_next, batch, (int64_t)L.img, st);
        }
        if ((rc = scd_launch_tweedie_il(g, x, s, atb, t, abar, n_table, (float)gamma, xhat0, xi, bi, batch, st))) return rc;
        if (n_iter > 0 && (rc = cg_run_il(g, L, xi, xi, bi, (float)gamma, n_iter, batch, w, st, w_il))) return rc;
        return scd_launch_ddim_il(g, xi, s, eps, t, t_prev, abar, n_table, (float)eta, (float)(eta * eta), x_next, batch, st);
    }
    float *b = (float *)(w + L.off_b), *xh = (float *)(w + L.off_xh);
    const int64_t numel = (int64_t)L.img;
    // xhat0 = Tweedie(x, s) and b = xhat0 + gamma*A*y are produced inside the pack pass of the
    // first projection; CG starts from xhat0 but must not overwrite it (the predictor returns it)
    FpPrologue tw;
    memset(&tw, 0, sizeof(tw));
    tw.mode = 2; tw.x = x; tw.s = s; tw.atb = atb; tw.t = t; tw.abar = abar; tw.n_table = n_table;
    tw.gamma = (float)gamma; tw.xhat0 = xhat0; tw.b = b;
    if ((rc = scd_cg_run(g, xhat0, xh, b, (float)gamma, n_iter, batch, work, work_bytes, st, &tw, w_il))) return rc;
    return scd_launch_ddim(xh, s, eps, t, t_prev, abar, n_table, (float)eta, (float)(eta * eta), x_next,
                           batch, numel, st);
}

// ------------------------------------------------------ host-buffer calls ---
static int host_roundtrip(const scd_geom_t *g, const float *in_host, size_t in_elems,
                          float *out_host, size_t out_elems, int batch, bool forward)
{
    if (!g || !in_host || !out_host) { scd_set_error("scd_*_host: null argument"); return SCD_E_INVALID; }
    if (batch <= 0) return 0;
    float *d_in = nullptr, *d_out = nullptr;
    void *d_scr = nullptr;
    const size_t scr_bytes = forward ? scd_fp_scratch_need(g, batch) : scd_sino_il_bytes(g, batch);
    cudaStream_t st = nullptr;
    int rc = 0;
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)) != cudaSuccess) return scd_cuda_fail(e, "stream create");
    if ((e = cudaMalloc(&d_in, in_elems * 4)) != cudaSuccess) { rc = scd_cuda_fail(e, "cudaMalloc"); goto done; }
    if ((e = cudaMalloc(&d_out, out_elems * 4)) != cudaSuccess) { rc = scd_cuda_fail(e, "cudaMalloc"); goto done; }
    if ((e = cudaMemcpyAsync(d_in, in_host, in_elems * 4, cudaMemcpyHostToDevice, st)) != cudaSuccess) { rc = scd_cuda_fail(e, "H2D"); goto done; }
    if ((e = cudaMalloc(&d_scr, scr_bytes)) != cudaSuccess) { rc = scd_cuda_fail(e, "cudaMalloc"); goto done; }
    if (forward) rc = scd_fp(g, d_in, d_out, batch, 0, g->n_angles, d_scr, scr_bytes, st);
    else rc = scd_bp(g, d_in, d_out, batch, 0, g->n_angles, (float)g->adj_scale, nullptr, 0.f, d_scr, scr_bytes, st);
    if (rc) goto done;
    if ((e = cudaMemcpyAsync(out_host, d_out, out_elems * 4, cudaMemcpyDeviceToHost, st)) != cudaSuccess) { rc = scd_cuda_fail(e, "D2H"); goto done; }
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) { rc = scd_cuda_fail(e, "sync"); goto done; }
done:
    if (d_in) cudaFree(d_in);
    if (d_out) cudaFree(d_out);
    if (d_scr) cudaFree(d_scr);
    if (st) cudaStreamDestroy(st);
    return rc;
}

extern "C" int scd_fp_host(const scd_geom_t *g, const float *img_host, float *sino_host, int batch)
{
    if (!g) { scd_set_error("scd_fp_host: null handle"); return SCD_E_INVALID; }
    return host_roundtrip(g, img_host, (size_t)batch * g->n0 * g->n1, sino_host,
                          (size_t)batch * g->n_angles * g->n_det, batch, true);
}

extern "C" int scd_bp_host(const scd_geom_t *g, const float *sino_host, float *img_host, int batch)
{
    if (!g) { scd_set_error("scd_bp_host: null handle"); return SCD_E_INVALID; }
    return host_roundtrip(g, sino_host, (size_t)batch * g->n_angles * g->n_det, img_host,
                          (size_t)batch * g->n0 * g->n1, batch, false);
}
