// Internal declarations shared by the translation units of libscd_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <stdio.h>
#include "scd_b200.h"

// ---------------------------------------------------------------- errors ---
void scd_set_error(const char *fmt, ...);
int  scd_cuda_fail(cudaError_t e, const char *what);   // records + returns -(int)e
void scd_count_launch(int n = 1);

#define SCD_CUDA(call)                                                        \
    do {                                                                      \
        cudaError_t e__ = (call);                                             \
        if (e__ != cudaSuccess) return scd_cuda_fail(e__, #call);             \
    } while (0)

// SCD_SYNC_LAUNCHES=1 in the environment: synchronise the device after every launch of the library and report
// the first kernel that faults by name (debugging aid; breaks graph capture and every overlap)
bool scd_sync_launches();
#define SCD_LAUNCH_CHECK(name)                                                \
    do {                                                                      \
        cudaError_t e__ = cudaGetLastError();                                 \
        if (e__ == cudaSuccess && scd_sync_launches()) { e__ = cudaDeviceSynchronize(); fprintf(stderr, "[scd] %s -> %d\n", name, (int)e__); } \
        if (e__ != cudaSuccess) return scd_cuda_fail(e__, name);              \
        scd_count_launch();                                                   \
    } while (0)

// ------------------------------------------------- dependent launches ------
// Every kernel of the library is launched with programmatic stream serialisation (PDL): it may
// become resident while its predecessor in the stream drains, runs the part of its prologue that
// touches no global data produced by earlier kernels (mbarrier init, geometry tables) and then
// blocks in scd_pdl_wait() until the predecessor has completed and flushed its writes.  All
// global reads of produced data and ALL global writes come after scd_pdl_wait().
#ifdef __CUDACC__
__device__ __forceinline__ void scd_pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void scd_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
#endif
bool scd_pdl_enabled();
// Optional per-CTA time stamps (tools/timeline.py): compiled in only with -DSCD_DEBUG_STAMPS (the debug build
// `python -m diffusion_models_dev_project_b200.build --debug`, which also exports scd_debug_set_stamps, declared
// in include/scd_b200_debug.h); the default library carries neither the hook nor the stores.
#ifdef SCD_DEBUG_STAMPS
unsigned long long *scd_debug_stamps();      // device buffer of 8 x int64 per CTA, or NULL
#else
static inline unsigned long long *scd_debug_stamps() { return nullptr; }
#endif
#ifdef __CUDACC__
__device__ __forceinline__ void scd_stamp(unsigned long long *dbg, int slot)
{
#ifdef SCD_DEBUG_STAMPS
    if (dbg && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        dbg[(size_t)(blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z)) * 8 + slot] = t;
    }
#else
    (void)dbg; (void)slot;
#endif
}
#endif

template <typename... KArgs, typename... Args>
static inline cudaError_t scd_launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                            cudaStream_t st, int cluster_x, Args &&...args)
{
    cudaLaunchConfig_t cfg;
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[2];
    int n = 0;
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = scd_pdl_enabled() ? 1 : 0;
    ++n;
    if (cluster_x > 0) {
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = cluster_x; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = at; cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Opt-in dynamic shared memory is a per-device function attribute: remember, per device, the
// largest size a kernel instantiation has been configured for.
struct ScdSmemAttr { int configured[16]; };
template <typename K>
static inline cudaError_t scd_ensure_smem(K kernel, ScdSmemAttr &state, int device, size_t smem)
{
    const int slot = device >= 0 && device < 16 ? device : 0;
    if ((int)smem <= state.configured[slot] && device < 16) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) state.configured[slot] = (int)smem;
    return e;
}

// -------------------------------------------------------------- geometry ---
// Forward projector, per angle.  In "tile coordinates" the ray of detector bin
// j crosses marching row r at interpolation-axis position
//     u(r, j) = a*j + b*r + c          (pixel-index units, pixel 0 centred at 0)
// class 0: |sin| > |cos|, march along axis 0 (r = k0), interpolate along axis 1
// class 1: otherwise,      march along axis 1 (r = k1), interpolate along axis 0
struct FpAngle {
    double a, b, c;     // exact (host fp64) coefficients
    float  scale;       // dx / max(|cos|,|sin|)
    int    cls;
};

// Backprojector, per angle: detector coordinate (bin units, bin 0 centred at
// 0) of pixel (k0,k1):  v = ci*k0 + si*k1 + oi
struct BpAngle {
    double ci, si, oi;
};

struct scd_geom {
    int n0, n1, n_angles, n_det;
    double x_min, y_min, dx, s_min, ds, adj_scale;
    int device;
    unsigned long long id;  // unique per scd_geom_create (cache keys must not rely on the address: it can be reused)
    int sm_count;
    int smem_optin;       // max dynamic shared memory per block (opt-in), bytes
    // device tables
    FpAngle *d_fp;        // [n_angles]
    BpAngle *d_bp;        // [n_angles]
    int     *d_order;     // [n_angles] angle ids sorted by (class, index)
    float2  *d_rayt;      // [n_angles][n_det] (u0 + 1, b): start position (row 0) and slope of every ray, from fp64;
                          // rows in order[] order (position p holds angle order[p])
    float2  *d_angt;      // [n_angles] (scale, id as int bits) in order[] order
    // view weights (scd_geom_create_weighted), NULL when every view weighs 1: applied to the interleaved sinogram
    // the backprojector reads, never to A's user-layout output
    float   *d_angw;      // [n_angles] w_i in order[] order (projector output)
    float   *d_w;         // [n_angles] w_i by angle id (sinogram re-layout)
    float   *d_zero_row;  // max(n0, n1) * 16 zero floats: source of projector strip rows beyond the image
    // host copies
    FpAngle *h_fp;
    BpAngle *h_bp;
    int     *h_order;
    int n_cls0;           // number of class-0 angles (they come first in order[])
    // tuning overrides (0 = heuristic)
    int tune_fp_samples, tune_fp_angles, tune_fp_rows, tune_fp_threads, tune_fp_nbuf, tune_fp_cluster, tune_fp_plan, tune_fp_plan_cost;
    int tune_bp_tile, tune_bp_share, tune_bp_rows;
    int tune_fp_cls0;     // 1: class-0 strips pixel-major through tensor copies (like class 1) instead of bulk rows
    int tune_fp_source;   // 1: force the packed-copy path of the projector (A/B runs, tests)
    // sample-interleaved sinogram rows (bp_tile.cu): il_padl zero bins, n_det bins, zero bins up to il_nb
    int il_padl, il_nb;
};

// ------------------------------------------------------------ launchers ----
// scratch: caller-owned device buffer of >= scd_fp_scratch_need(g, batch) bytes that
// receives the packed ("tile-ready") copy of the image
// Optional producer fused into the pack pass of the projector (img may be NULL then):
//   mode 1: p = r + beta*p with beta = sum(rr_new_part)/sum(rr_old_part); writes p; projects p
//   mode 2: xhat0 = (x - s*std_t)/mean_t, b = xhat0 + gamma*atb; writes both; projects xhat0
struct FpPrologue {
    int mode;
    float *p; const float *r;
    const float *rr_new_part; int rr_new_n; const float *rr_old_part; int rr_old_n; int part_stride;
    const float *x, *s, *atb, *t, *abar; int n_table; float gamma;
    float *xhat0, *b;
};
// sino: user layout [batch][n_angles][n_det] (may be NULL); sino_il: sample-interleaved layout read
// by scd_launch_bp_il (may be NULL)
int scd_launch_fp(const scd_geom *g, const float *img, float *sino, float *sino_il, int batch,
                  int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes,
                  cudaStream_t st, const FpPrologue *prologue = nullptr);
// samples interleaved per pixel / detector bin for this batch (1, 2, 4, 8 or 16)
int scd_group_samples(const scd_geom *g, int batch);

// ---- sample-interleaved images ("il image": [group][k0][k1][SB], SB = scd_group_samples(batch) >= 4) ----
// The projector reads them with tensor copies (no packed copy); the CG vectors live in this layout for the whole solve.
bool   scd_il_image_ok(const scd_geom *g, int batch);         // does this batch run on the tensor-copy path?
size_t scd_il_image_bytes(const scd_geom *g, int batch);      // bytes of one il image (upper bound over the tuning)
// recurrence of the CG solve carried by the projector's output phase: q = A img + beta * q_old,
// beta[b] = sum(rr_new_part[b]) / sum(rr_old_part[b]); beta is also stored to beta_out[b] (may be NULL)
struct FpAccumulate {
    const float *rr_new_part; int rr_new_n; const float *rr_old_part; int rr_old_n; int part_stride;
    float *beta_out;
};
int scd_launch_fp_ilimg(const scd_geom *g, const float *img_il, float *sino, float *sino_il, int batch,
                        int angle_lo, int angle_hi, cudaStream_t st, const FpAccumulate *acc);
// user layout -> il image for up to two arrays in one launch (b_user / b_il may be NULL)
int scd_launch_il_pack(const scd_geom *g, const float *a_user, float *a_il, const float *b_user, float *b_il,
                       int batch, cudaStream_t st);
// il image -> user layout
int scd_launch_il_unpack(const scd_geom *g, const float *a_il, float *a_user, int batch, cudaStream_t st);
// Tweedie + rhs producing the CG start iterate and right-hand side in il layout (xhat0 also in user layout)
int scd_launch_tweedie_il(const scd_geom *g, const float *x, const float *s, const float *atb, const float *t,
                          const float *abar, int n_table, float gamma, float *xhat0_user, float *x_il, float *b_il,
                          int batch, cudaStream_t st);
// DDIM update reading the CG result in il layout, writing user layout
int scd_launch_ddim_il(const scd_geom *g, const float *xh_il, const float *s, const float *eps, const float *t,
                       const float *t_prev, const float *abar, int n_table, float eta, float eta2, float *out,
                       int batch, cudaStream_t st);
// alpha = rr/pd;  x = x_in + alpha p;  r -= alpha d;  per-block partials of ||r||^2 -- all vectors il images
int scd_il_vec_blocks(const scd_geom *g, int batch);           // partials per sample written by the kernel below
int scd_launch_cg_update_xr_il(const scd_geom *g, const float *x_in, float *x, float *r, const float *p, const float *d,
                               const float *rr_part, int rr_n, const float *pd_part, int pd_n, int part_stride,
                               float *rr_new_part, int batch, cudaStream_t st);
size_t scd_fp_scratch_need(const scd_geom *g, int batch);
int scd_launch_fp_v4(const scd_geom *g, const float *img, float *sino, float *sino_il, int batch,
                     int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes,
                     cudaStream_t st, const FpPrologue *prologue);
size_t scd_fp_scratch_need_v4(const scd_geom *g, int batch);

// Backprojection with fused epilogue:
//   val  = c_acc*BP + c1*add1 + c2*add2
//   out  = val; if (out2) out2 = val
//   if (dot_part): dot_part[b*dot_stride + cta] = sum over the CTA's pixels of
//        val * (dot_with_add1 ? add1 : val)
#define SCD_MAX_BANDS 8
struct BpEpilogue {
    float c_acc;
    const float *add1; float c1;
    const float *add2; float c2;
    float *out2;
    float *dot_part; int dot_stride; int dot_with_add1;
    // Banded output (angle-sharded multi-GPU backprojection, peer_reduce.cu): when n_bands > 0 the rows
    // [i*band_rows, (i+1)*band_rows) of every sample are written to band_out[i] -- typically memory of the
    // GPU that owns band i, mapped into this process -- as a dense [batch][band_rows][n1] array instead
    // of `out`; band_rows is a multiple of 32 (every tile lies inside one band).
    float *band_out[SCD_MAX_BANDS] = {};
    int n_bands = 0, band_rows = 0;
    // Sample-interleaved images (il != 0): out, out2, add1, add2 are il images [group][k0][k1][SB] and every lane
    // moves its V samples of a pixel with one vector access.
    //   mode 0: as above.
    //   mode 1 (direction step of CG, reference src/utils/cg.py:24-27,35-38):
    //           p  = add1 + beta[b]*add2      (add1 = r, add2 = previous p; beta == NULL: p = add1)  -> out2
    //           d  = p + c_acc*BP                                                                    -> out
    //           dot_part: <p, d>
    int il = 0, mode = 0;
    const float *beta = nullptr;
};
// sino in user layout; scratch (>= scd_sino_il_bytes) receives the interleaved copy, times the view weights unless
// weighted == false (the plain transpose of A, gradient of the adaptation objective)
int scd_launch_bp(const scd_geom *g, const float *sino, float *out, int batch,
                  int angle_lo, int angle_hi, const BpEpilogue &ep, void *scratch, size_t scratch_bytes,
                  cudaStream_t st, bool weighted = true);
int scd_launch_bp_il(const scd_geom *g, const float *sino_il, float *out, int batch,
                     int angle_lo, int angle_hi, const BpEpilogue &ep, cudaStream_t st);
// banded stores + rank-ordered reduction of the bands (peer_reduce.cu)
int scd_launch_band_reduce(const float *stage, int n_src, int64_t slot_stride, int batch, int band_rows, int rows,
                           int n1, int row_lo, int n0, float *const *out_ptrs, int n_out, int multicast,
                           const float *addend, float c_add, float c_sum, cudaStream_t st);
int scd_launch_sino_pack(const scd_geom *g, const float *sino, float *sino_il, int batch,
                         int angle_lo, int angle_hi, cudaStream_t st, bool weighted = true);
size_t scd_sino_il_bytes(const scd_geom *g, int batch);
// number of dot_part entries per sample the BP launch for this batch writes (current tuning) /
// an upper bound independent of the tuning (workspace sizing)
int scd_bp_ctas_per_sample(const scd_geom *g, int batch);
int scd_bp_ctas_per_sample_max(const scd_geom *g, int batch);

// Vector kernels of the CG recurrences (vec_ops.cu).  *_part arrays hold
// per-block partial sums [batch][part_stride]; consumers add them in index
// order (deterministic, no atomics).
int scd_vec_blocks_per_sample(int64_t numel, int batch);
int scd_launch_cg_update_xr(const float *x_in, float *x, float *r, const float *p, const float *d,
                            const float *rr_part, int rr_n,
                            const float *pd_part, int pd_n, int part_stride,
                            float *rr_new_part, int batch, int64_t numel,
                            cudaStream_t st);
int scd_launch_tweedie_rhs(const float *x, const float *s, const float *atb,
                           const float *t, const float *abar, int n_table,
                           float gamma, float *xhat0, float *b, int batch,
                           int64_t numel, cudaStream_t st);
int scd_launch_ddim(const float *xhat, const float *s, const float *eps,
                    const float *t, const float *t_prev, const float *abar,
                    int n_table, float eta, float eta2, float *out, int batch,
                    int64_t numel, cudaStream_t st);

// x_in: start iterate (read only), x_out: result (may alias x_in)
int scd_cg_run(const scd_geom *g, const float *x_in, float *x_out, const float *rhs,
               float gamma, int n_iter, int batch, void *work, size_t work_bytes,
               cudaStream_t st, const FpPrologue *first = nullptr);
