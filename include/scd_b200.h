/*
 * scd_b200.h -- C ABI of libscd_b200.so
 *
 * B200 (sm_100a) implementation of the data-consistency hot path of the
 * SCD / DDS reverse sampler of educating-dip/diffusion_models_dev_project:
 *
 *   A   parallel-beam ray transform, ray-driven Joseph projector
 *   A*  pixel-driven linear-interpolation backprojector (weighted adjoint)
 *   CG  batched conjugate gradient on (I + gamma A*A) x = rhs
 *   Tweedie + rhs, DDIM update (DDPM schedule)
 *
 * The reference has no native code: the interfaces these entry points replace
 * are Python call sites, cited per function below (paths relative to the
 * reference checkout).  Calling convention:
 *
 *   - plain C, no C++/torch types; every buffer is a raw pointer.  Unless a
 *     function name ends in `_host`, buffers are DEVICE pointers owned by
 *     the caller (PyTorch), fp32, contiguous:
 *       image     [batch][n0][n1]            (n1 fastest; axis0 <-> x, axis1 <-> y)
 *       sinogram  [batch][n_angles][n_det]   (n_det fastest)
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued on it and
 *     the call returns without synchronising (graph-capture safe: no
 *     allocation, no sync, no host reads of device memory after create).
 *   - gamma / eta are passed as double (the Python floats of the reference's
 *     CLI); kernels round them to fp32 exactly where PyTorch would.
 *   - return value: 0 on success, < 0 on failure (negated cudaError_t, or
 *     SCD_E_* below); scd_last_error_string() describes the last failure on
 *     the calling thread.
 *   - there is no CPU fallback anywhere in this library.
 */
#ifndef SCD_B200_H
#define SCD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCD_E_INVALID   (-10001)  /* bad argument                           */
#define SCD_E_NODEVICE  (-10002)  /* no CUDA device / not sm_100            */
#define SCD_E_WORKSPACE (-10003)  /* caller workspace too small             */

typedef struct scd_geom scd_geom_t; /* opaque, immutable after create */

/* Geometry description.  Mirrors what SimpleTrafo.__init__ derives through
 * odl.uniform_discr + odl.tomo.parallel_beam_geometry
 * (src/physics/trafo.py:17-27): image grid, angle list, detector partition.
 * adj_scale is the factor applied by A* on top of the plain sum of
 * interpolated detector values (default of the Python layer: delta_phi).   */
typedef struct scd_geom_desc {
    int32_t n0, n1;        /* image shape (axis0 = x, axis1 = y)             */
    double  x_min, y_min;  /* lower corner of the image domain               */
    double  dx;            /* pixel size (square pixels)                     */
    int32_t n_angles;
    const double *angles;  /* [n_angles] radians, host pointer (copied)      */
    int32_t n_det;
    double  s_min;         /* lower edge of the detector partition (= -rho)  */
    double  ds;            /* detector cell size                             */
    double  adj_scale;     /* A* = adj_scale * sum_i lerp(sino[i], t_i(x))   */
} scd_geom_desc;

/* Build the device-side tables for one geometry on the current device.
 * Replaces: SimpleTrafo.__init__ (src/physics/trafo.py:17-51).              */
int scd_geom_create(const scd_geom_desc *desc, scd_geom_t **out);

/* Same geometry with a weight per view: A* = adj_scale * sum_i w_i * lerp(sino[i], t_i(x)).
 * angle_weights[n_angles] is the relative angular cell of each view (ODL's nonuniform_partition /
 * uniform_partition of a wedge, mean 1; finite and > 0).  It makes A* the quadrature of a
 * limited-angle or non-uniform view set.  A (scd_fp) stays unweighted.  The weight is applied where the
 * sinogram the backprojector reads is written: by the projector's interleaved output (scd_fp_il,
 * scd_fp_ilimg, scd_cg, scd_dds_step, the operator applications of scd_adapt_fwd/bwd) and by the
 * re-layout of a user sinogram (scd_bp, scd_bp_banded).  The gradient backprojection of
 * scd_adapt_bwd stays unweighted: it is the transpose of A.
 * angle_weights == NULL, or every entry exactly 1.0: identical to scd_geom_create.                      */
int scd_geom_create_weighted(const scd_geom_desc *desc, const double *angle_weights, scd_geom_t **out);
int scd_geom_destroy(scd_geom_t *g);

/* A: forward projection of angles [angle_lo, angle_hi) (rows outside that
 * range of `sino` are left untouched; sino always has n_angles rows).
 * `scratch` is a caller-owned device buffer of at least
 * scd_fp_scratch_bytes(g, batch) bytes: the projector first interleaves the samples
 * of a group per pixel (the layout its shared-memory strips are fetched from).
 * Replaces: SimpleTrafo.trafo -> ODL/ASTRA par_fp (src/physics/trafo.py:58). */
size_t scd_fp_scratch_bytes(const scd_geom_t *g, int batch);
int scd_fp(const scd_geom_t *g, const float *img, float *sino, int batch,
           int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes,
           void *stream);

/* A*: out = c_acc * BP(sino; angles [lo,hi)) + c_add * addend
 * where BP is the un-scaled pixel-driven sum; the plain adjoint is
 * c_acc = adj_scale, addend = NULL.
 * `scratch` is a caller-owned device buffer of at least scd_bp_scratch_bytes(g, batch)
 * bytes: the sinogram is first re-laid out with the samples interleaved per detector
 * bin, the form the backprojector's shared-memory segments are bulk-copied from.
 * Replaces: SimpleTrafo.trafo_adjoint -> ODL/ASTRA par_bp
 * (src/physics/trafo.py:61) and the axpy of `op` (src/samplers/utils.py:188-189). */
size_t scd_bp_scratch_bytes(const scd_geom_t *g, int batch);
int scd_bp(const scd_geom_t *g, const float *sino, float *out, int batch,
           int angle_lo, int angle_hi, float c_acc, const float *addend,
           float c_add, void *scratch, size_t scratch_bytes, void *stream);

/* The same operators on the sample-interleaved sinogram ("sino_il": [group][angle][bins +
 * zero pads][samples of the group], scd_sino_il_buffer_bytes(g, batch) bytes, 128-byte aligned),
 * the form in which A*(A x) is composed without re-laying-out the sinogram in between:
 * scd_fp_il writes it, scd_bp_il reads it.  The layout is internal to the library (it depends on
 * the batch size); a buffer written for one batch size must be read with the same one.
 * Replaces: the `ray_trafo.trafo_adjoint(ray_trafo(x))` pairs of `op`
 * (src/samplers/utils.py:188-189, 235-236, 302-303).                                      */
size_t scd_sino_il_buffer_bytes(const scd_geom_t *g, int batch);
int scd_fp_il(const scd_geom_t *g, const float *img, float *sino_il, int batch,
              int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes, void *stream);
int scd_bp_il(const scd_geom_t *g, const float *sino_il, float *out, int batch,
              int angle_lo, int angle_hi, float c_acc, const float *addend, float c_add,
              void *stream);

/* Sample-interleaved images ("il image": [group][n0][n1][samples of the group], 128-byte aligned, opaque like
 * sino_il).  For batches of >= 3 samples the projector reads this layout directly through tensor copies
 * (cp.async.bulk.tensor: no packed copy of the image) and the backprojector writes it with one 16-byte
 * store per lane; scd_cg / scd_dds_step keep x, r, p, d in it for the whole solve.  A caller that iterates
 * with A / A* itself can do the same:
 *   scd_img_il_bytes   bytes of one il image for `batch` samples; 0 if this batch size has no il form
 *                      (2 samples; 1 sample when n1 is not a multiple of 4).  For ONE sample the il image is the
 *                      [n0][n1] image itself: scd_fp / scd_cg / scd_dds_step then read the caller's tensors directly
 *   scd_img_il_pack / scd_img_il_unpack   [batch][n0][n1] <-> il image
 *   scd_fp_ilimg       sino_il = A(img_il)                                   -- ONE launch (fp_march)
 *   scd_bp_ilimg       out_il = c_acc * BP(sino_il) + c_add * addend_il      -- ONE launch (bp_tile)
 * Replaces: the same call sites as scd_fp_il / scd_bp_il.                                      */
size_t scd_img_il_bytes(const scd_geom_t *g, int batch);
int scd_img_il_pack(const scd_geom_t *g, const float *img, float *img_il, int batch, void *stream);
int scd_img_il_unpack(const scd_geom_t *g, const float *img_il, float *img, int batch, void *stream);
int scd_fp_ilimg(const scd_geom_t *g, const float *img_il, float *sino_il, int batch,
                 int angle_lo, int angle_hi, void *stream);
int scd_bp_ilimg(const scd_geom_t *g, const float *sino_il, float *out_il, int batch,
                 int angle_lo, int angle_hi, float c_acc, const float *addend_il, float c_add, void *stream);

/* Bytes of scratch scd_cg / scd_dds_step need for `batch` samples.           */
size_t scd_cg_workspace_bytes(const scd_geom_t *g, int batch);

/* Batched CG, fixed n_iter, per-sample alpha/beta, no tolerance test:
 * solves (I + gamma A*A) x = rhs starting from x (overwritten by the result).
 * Replaces: cg(op, x, rhs, n_iter) with op(v) = v + gamma*A*(A v)
 * (src/utils/cg.py:11-39, src/samplers/utils.py:188-189).                    */
int scd_cg(const scd_geom_t *g, float *x, const float *rhs, double gamma,
           int n_iter, int batch, void *work, size_t work_bytes, void *stream);

/* DDPM alpha-bar table: abar[k] = prod_{m<k}(1 - beta_m) rounded to fp32, k in
 * [0, n_table) with abar[0] = 1 (index t+1, so t = -1 -> 1).  Device pointer,
 * computed by the caller exactly like DDPM._compute_alpha_cumprod
 * (src/utils/sde.py:172-174).  t / t_prev are DEVICE float arrays [batch]
 * holding integer-valued time steps, as BaseSampler passes them
 * (src/samplers/base_sampler.py:83-87).                                      */

/* Tweedie + CG right-hand side in one pass:
 *   xhat0 = (x - s*sqrt(1-abar_t)) / sqrt(abar_t);  b = xhat0 + gamma*atb
 * Replaces: apTweedy (src/samplers/utils.py:370-378) + :197.                 */
int scd_tweedie_rhs(const float *x, const float *s, const float *atb,
                    const float *t, const float *abar, int n_table,
                    double gamma, float *xhat0, float *b, int batch,
                    int64_t numel_per_sample, void *stream);

/* DDIM update for the DDPM schedule:
 *   out = m' * xhat + sqrt(1 - m'^2 - tbeta^2 eta^2) * s + eta*tbeta*eps
 * (m' = sqrt(abar_{t_prev}); tbeta as in the reference, NaN -> 0).
 * Replaces: ddim(...) DDPM branch (src/samplers/utils.py:338-368).           */
int scd_ddim(const float *xhat, const float *s, const float *eps,
             const float *t, const float *t_prev, const float *abar,
             int n_table, double eta, float *out, int batch,
             int64_t numel_per_sample, void *stream);

/* One whole data-consistency step of the DDS predictor after the score call:
 * Tweedie -> b -> CG(n_iter) -> DDIM.  x_next and xhat0 are outputs.
 * Replaces: decomposed_diffusion_sampling_sde_predictor body after score()
 * (src/samplers/utils.py:195-216).                                           */
int scd_dds_step(const scd_geom_t *g, const float *x, const float *s,
                 const float *atb, const float *eps, const float *t,
                 const float *t_prev, const float *abar, int n_table,
                 double gamma, double eta, int n_iter, float *x_next,
                 float *xhat0, int batch, void *work, size_t work_bytes,
                 void *stream);

/* Adaptation loss of SCD, loss(x) = mean((A x - y)^2) + lambda*tv_loss(x)
 * (src/utils/exp_utils.py:256-257, src/samplers/adaptation.py:7-11):
 *   scd_residual_sq : r = ax - y, part[k] = block-k partial sum of r^2 (scd_residual_sq_blocks entries)
 *   scd_tv_loss     : part[image*scd_tv_blocks + k] = partial sums of the cropped |dh| + |dw|
 *   scd_tv_grad     : grad = d tv_loss / d x
 * The caller adds the partials (in index order: deterministic).                */
int scd_residual_sq_blocks(int64_t numel);
int scd_residual_sq(const float *ax, const float *y, float *r, float *part, int64_t numel, void *stream);
int scd_tv_blocks(int n0, int n1);
int scd_tv_loss(const float *x, float *part, int images, int n0, int n1, void *stream);
int scd_tv_grad(const float *x, float *grad, int images, int n0, int n1, void *stream);

/* The adaptation objective of SCD as two calls (forward, and the complete reverse sweep): per Adam step
 * `_adapt` (src/samplers/utils.py:241-260) evaluates
 *     xhat0 = apTweedy(s, x);  xhat = cg(op, xhat0, xhat0 + gamma*atb, n_iter)  [dc_type 0; 1: one gradient
 *     step xhat0 - gamma A*(A xhat0) + gamma atb; 2: xhat = xhat0];  loss = mean((A xhat - y)^2) + tv_lambda*tv(xhat)
 * and differentiates it with respect to the score output s (autograd through the unrolled CG iterations).
 *   scd_adapt_fwd : loss[0] (device scalar), optionally xhat; keeps what the sweep needs in `work`
 *   scd_adapt_bwd : grad_s = d(grad_loss[0] * loss)/d s  (grad_loss: device scalar or NULL = 1), from the
 *                   SAME `work` buffer, untouched since the forward call.  trafo_grad_scale is the factor between
 *                   the gradient of <g, A x> w.r.t. x and the plain backprojection sum: adj_scale/c_w under ODL's
 *                   pairing (c_w = dphi*ds/dx^2, SURVEY.md 8b).
 * `work`: scd_adapt_workspace_bytes(g, batch, n_iter) bytes, 256-byte aligned.  y: [batch][n_angles][n_det].
 * Nothing is allocated, synchronised or read back: both calls can be captured in a CUDA graph.            */
size_t scd_adapt_workspace_bytes(const scd_geom_t *g, int batch, int n_iter);
int scd_adapt_fwd(const scd_geom_t *g, const float *x, const float *s, const float *atb, const float *y,
                  const float *t, const float *abar, int n_table, double gamma, int n_iter, int dc_type,
                  double tv_lambda, float *loss, float *xhat_out, int batch, void *work, size_t work_bytes,
                  void *stream);
int scd_adapt_bwd(const scd_geom_t *g, const float *grad_loss, const float *t, const float *abar, int n_table,
                  double gamma, int n_iter, int dc_type, double tv_lambda, double trafo_grad_scale,
                  float *grad_s, int batch, void *work, size_t work_bytes, void *stream);

/* Ramp filter of the filtered back-projection: every sinogram row is convolved along the detector
 * axis with the band-limited ramp (Kak & Slaney / the "ramp" Fourier filter of the reference's recipe)
 * and divided by the detector cell size:
 *   out[b][i][k] = (1/ds) * sum_j sino[b][i][j] * h(|k-j|),  h(0) = 1/4, h(odd n) = -1/(pi n)^2, else 0
 * so that fbp(y) = scd_bp(scd_ramp_filter(y)) with c_acc = pi/n_angles satisfies fbp(A x) ~ x.
 * `out` may not alias `sino`.
 * Replaces: the filtering half of SimpleTrafo.fbp (src/physics/trafo.py:34,42,67); recipe
 * filter_sinogram (src/physics/utils.py:11-33: zero-padded FFT, ramp, pi/(2 n_angles)).        */
int scd_ramp_filter(const scd_geom_t *g, const float *sino, float *out, int batch, void *stream);

/* Angle-sharded backprojection of one large slice stack over the GPUs of a box (BASELINE.json
 * config 4; the reference is single-GPU, SURVEY.md section 8e): every GPU backprojects its angle
 * range and the partial images are summed.  Instead of writing a local partial image and handing
 * it to a collective, the backprojector can store every tile straight into the memory of the GPU
 * that owns the tile's band of image rows (peer memory mapped by the caller, e.g. CUDA IPC /
 * torch symmetric memory), and the owner adds the staged copies:
 *   scd_bp_banded / scd_bp_il_banded : like scd_bp / scd_bp_il without addend, but rows
 *       [i*band_rows, (i+1)*band_rows) of every sample go to band_ptrs[i] as a dense
 *       [batch][band_rows][n1] array (band_ptrs: HOST array of n_bands <= 8 device pointers;
 *       band_rows a multiple of 32 with n_bands*band_rows >= n0)
 *   scd_band_reduce : for the `rows` image rows starting at row_lo (the caller's band):
 *       out_p[sample][row_lo + r][k] = c_sum * sum_{src < n_src} stage[src*slot_stride + dense(sample, r, k)]
 *                                      + c_add * addend[sample][row_lo + r][k]      (addend may be NULL)
 *       for every p < n_out (out_ptrs: HOST array of device pointers to [batch][n0][n1] arrays,
 *       local or peer); the copies are added in src order (deterministic).  With
 *       out_is_multicast != 0, out_ptrs[0] is ONE NVSwitch multicast address of that array on all
 *       GPUs (CUDA multicast object / torch symmetric memory `multicast_ptr`): each value is
 *       stored once with multimem.st and replicated by the switch.
 * Ordering between GPUs (all stores of a band landed before its reduction; all reductions landed
 * before the result is read) is the caller's responsibility.                                   */
int scd_bp_banded(const scd_geom_t *g, const float *sino, int batch, int angle_lo, int angle_hi,
                  float c_acc, float *const *band_ptrs, int n_bands, int band_rows,
                  void *scratch, size_t scratch_bytes, void *stream);
int scd_bp_il_banded(const scd_geom_t *g, const float *sino_il, int batch, int angle_lo, int angle_hi,
                     float c_acc, float *const *band_ptrs, int n_bands, int band_rows, void *stream);
int scd_band_reduce(const float *stage, int n_src, int64_t slot_stride_floats, int batch, int band_rows,
                    int rows, int n1, int row_lo, int n0, float *const *out_ptrs, int n_out,
                    int out_is_multicast, const float *addend, float c_add, float c_sum, void *stream);

/* Host-buffer variants (pageable or pinned host memory): copy in, run, copy
 * out, synchronise the stream.  These are what a non-PyTorch caller binds.   */
int scd_fp_host(const scd_geom_t *g, const float *img_host, float *sino_host,
                int batch);
int scd_bp_host(const scd_geom_t *g, const float *sino_host, float *img_host,
                int batch);

/* Introspection used by the tests, the bench and the launch heuristics.      */
int scd_geom_info(const scd_geom_t *g, int32_t *n0, int32_t *n1,
                  int32_t *n_angles, int32_t *n_det);
/* Number of kernels this library has launched in this process (all threads) since
 * the last reset (the bench reports it as gpu_launches).                     */
int64_t scd_launch_count(void);
void    scd_launch_count_reset(void);
/* Override launch heuristics (tuning / tests).  key is one of
 * "fp_samples" (samples interleaved per pixel/bin: 1,2,4,8,16), "fp_angles", "fp_rows",
 * "fp_threads", "fp_nbuf", "fp_cluster", "fp_plan", "fp_source" (1 = packed copy + 1-D bulk copies for every
 * batch size instead of tensor copies from the interleaved image, 2 = only for single-sample groups), "fp_cls0" (class-0 strips pixel-major through
 * tensor copies: 1 = always, 2 = never), "fp_plan_cost" (fixed cost of a unit in the unit plan, percent of one angle), "bp_tile", "bp_share" (1 = plain
 * march, no tap sharing between the pixels of a column pair), "bp_rows" (rows in use per tile; 1 = always the
 * full tile); value 0
 * restores the heuristic.  Not thread-safe; intended for benchmarks.         */
int scd_set_tuning(scd_geom_t *g, const char *key, int value);

const char *scd_last_error_string(void);
const char *scd_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SCD_B200_H */
