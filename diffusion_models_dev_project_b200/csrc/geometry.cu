// Geometry handle: host-side derivation of the per-angle projector constants
// (fp64) and their upload.  Follows the index-space specification of
// SURVEY.md Appendix A, which restates what SimpleTrafo.__init__
// (reference src/physics/trafo.py:17-34) obtains from ODL.
#include "scd_internal.cuh"
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <algorithm>
#include <atomic>

static thread_local char    g_err[512] = "";
static std::atomic<int64_t> g_launches{0};     // process-wide: autograd runs backward passes on its own threads

void scd_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int scd_cuda_fail(cudaError_t e, const char *what)
{
    scd_set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return -(int)e;
}

void scd_count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#ifdef SCD_DEBUG_STAMPS
static unsigned long long *g_stamps = nullptr;
unsigned long long *scd_debug_stamps() { return g_stamps; }
extern "C" void scd_debug_set_stamps(void *device_buffer) { g_stamps = (unsigned long long *)device_buffer; }
#endif

bool scd_sync_launches()
{
    static const bool on = getenv("SCD_SYNC_LAUNCHES") != nullptr;
    return on;
}

bool scd_pdl_enabled()
{
    static const bool on = getenv("SCD_NO_PDL") == nullptr;
    return on;
}

extern "C" const char *scd_last_error_string(void) { return g_err; }
extern "C" const char *scd_version(void) { return "scd_b200 0.1 (sm_100a)"; }
extern "C" int64_t scd_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" void scd_launch_count_reset(void) { g_launches.store(0, std::memory_order_relaxed); }

extern "C" int scd_geom_create(const scd_geom_desc *d, scd_geom_t **out)
{
    return scd_geom_create_weighted(d, nullptr, out);
}

extern "C" int scd_geom_create_weighted(const scd_geom_desc *d, const double *wts, scd_geom_t **out)
{
    return scd_geom_create_ex(d, wts, 0, out);
}

extern "C" int scd_geom_create_ex(const scd_geom_desc *d, const double *wts, uint32_t flags, scd_geom_t **out)
{
    if (!d || !out) { scd_set_error("scd_geom_create: null argument"); return SCD_E_INVALID; }
    *out = nullptr;
    if (flags & ~(uint32_t)SCD_GEOM_MATCHED_ADJOINT) {
        scd_set_error("scd_geom_create_ex: unknown flag bits 0x%x", (unsigned)(flags & ~(uint32_t)SCD_GEOM_MATCHED_ADJOINT));
        return SCD_E_INVALID;
    }
    // the matched backprojector's hat has half-width max(|cos|, |sin|) * dx/ds bins; its three taps around round(v)
    // cover it only while that stays below 1.5
    if ((flags & SCD_GEOM_MATCHED_ADJOINT) && d->dx > 0 && d->ds > 0 && !(d->dx / d->ds < 1.5)) {
        scd_set_error("scd_geom_create_ex: the matched adjoint needs dx/ds < 1.5 (got dx=%g ds=%g)", d->dx, d->ds);
        return SCD_E_INVALID;
    }
    if (wts && d->n_angles >= 1) {
        bool all_one = true;
        for (int i = 0; i < d->n_angles; ++i) {
            if (!std::isfinite(wts[i]) || !(wts[i] > 0.0)) {
                scd_set_error("scd_geom_create_weighted: angle weight %d is %g (must be finite and > 0)", i, wts[i]);
                return SCD_E_INVALID;
            }
            all_one = all_one && wts[i] == 1.0;
        }
        if (all_one) wts = nullptr;               // the unweighted geometry: no table, the same launches
    }
    if (d->n0 < 1 || d->n1 < 1 || d->n_angles < 1 || d->n_det < 2 || !d->angles ||
        !(d->dx > 0) || !(d->ds > 0)) {
        scd_set_error("scd_geom_create: invalid geometry (n0=%d n1=%d n_angles=%d n_det=%d dx=%g ds=%g)",
                      d->n0, d->n1, d->n_angles, d->n_det, d->dx, d->ds);
        return SCD_E_INVALID;
    }
    if (d->n0 > 8192 || d->n1 > 8192 || d->n_det > 16384) {
        scd_set_error("scd_geom_create: geometry too large for the fp32 index arithmetic");
        return SCD_E_INVALID;
    }
    int dev = 0, ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        scd_set_error("scd_geom_create: no CUDA device (%s); this library has no CPU path",
                      cudaGetErrorString(e));
        return SCD_E_NODEVICE;
    }
    SCD_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    SCD_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) {
        scd_set_error("scd_geom_create: device %d is sm_%d%d; this library is built for sm_100a only",
                      dev, prop.major, prop.minor);
        return SCD_E_NODEVICE;
    }

    scd_geom *g = (scd_geom *)calloc(1, sizeof(scd_geom));
    if (!g) { scd_set_error("out of host memory"); return SCD_E_INVALID; }
    g->n0 = d->n0; g->n1 = d->n1; g->n_angles = d->n_angles; g->n_det = d->n_det;
    g->x_min = d->x_min; g->y_min = d->y_min; g->dx = d->dx;
    g->s_min = d->s_min; g->ds = d->ds; g->adj_scale = d->adj_scale;
    g->device = dev;
    g->matched = (flags & SCD_GEOM_MATCHED_ADJOINT) ? 1 : 0;
    { const char *e = getenv("SCD_FP_SOURCE"); if (e && !strcmp(e, "packed")) g->tune_fp_source = 1; }   // A/B runs
    { static std::atomic<unsigned long long> next_id{1}; g->id = next_id.fetch_add(1); }
    g->sm_count = prop.multiProcessorCount;
    g->smem_optin = (int)prop.sharedMemPerBlockOptin;

    const int na = d->n_angles;
    g->h_fp = (FpAngle *)malloc(sizeof(FpAngle) * na);
    g->h_bp = (BpAngle *)malloc(sizeof(BpAngle) * na);
    g->h_order = (int *)malloc(sizeof(int) * na);
    std::vector<int> c0, c1;
    for (int i = 0; i < na; ++i) {
        const double phi = d->angles[i];
        const double cs = std::cos(phi), sn = std::sin(phi);
        FpAngle &f = g->h_fp[i];
        if (std::fabs(sn) > std::fabs(cs)) {
            // march along axis 0 (x), interpolate along axis 1 (y)
            f.cls = 0;
            f.a = d->ds / (sn * d->dx);
            f.b = -cs / sn;
            f.c = ((d->s_min + 0.5 * d->ds - (d->x_min + 0.5 * d->dx) * cs) / sn - d->y_min) / d->dx - 0.5;
            f.scale = (float)(d->dx / std::fabs(sn));
            c0.push_back(i);
        } else {
            // march along axis 1 (y), interpolate along axis 0 (x)
            f.cls = 1;
            f.a = d->ds / (cs * d->dx);
            f.b = -sn / cs;
            f.c = ((d->s_min + 0.5 * d->ds - (d->y_min + 0.5 * d->dx) * sn) / cs - d->x_min) / d->dx - 0.5;
            f.scale = (float)(d->dx / std::fabs(cs));
            c1.push_back(i);
        }
        BpAngle &b = g->h_bp[i];
        b.ci = d->dx * cs / d->ds;
        b.si = d->dx * sn / d->ds;
        b.oi = ((d->x_min + 0.5 * d->dx) * cs + (d->y_min + 0.5 * d->dx) * sn - d->s_min) / d->ds - 0.5;
    }
    {
        // extreme detector coordinates (bin units) of the image corners over all angles -> zero
        // bins either side of the interleaved sinogram rows so that every staged segment of
        // bp_tile (start rounded down to x4, up to 12 bins of slack) stays inside its row
        double vmin = 0.0, vmax = (double)(d->n_det - 1);
        for (int i = 0; i < na; ++i)
            for (int c = 0; c < 4; ++c) {
                const double k0 = (c & 1) ? d->n0 - 1 : 0, k1 = (c & 2) ? d->n1 - 1 : 0;
                const double v = g->h_bp[i].ci * k0 + g->h_bp[i].si * k1 + g->h_bp[i].oi;
                vmin = std::min(vmin, v); vmax = std::max(vmax, v);
            }
        g->il_padl = ((int)std::max(0.0, 4.0 - std::floor(vmin)) + 3) & ~3;
        g->il_nb = (g->il_padl + std::max(d->n_det, (int)std::ceil(vmax) + 1) + 13 + 3) & ~3;
    }
    g->n_cls0 = (int)c0.size();
    std::copy(c0.begin(), c0.end(), g->h_order);
    std::copy(c1.begin(), c1.end(), g->h_order + c0.size());

    // per-ray start position and slope of the forward march, evaluated in fp64 once; both tables are
    // stored in order[] order so that a CTA reads them without first looking the angle id up
    std::vector<float2> rayt((size_t)na * d->n_det), angt((size_t)na);
    for (int p = 0; p < na; ++p) {
        const int i = g->h_order[p];
        for (int j = 0; j < d->n_det; ++j)
            rayt[(size_t)p * d->n_det + j] = make_float2((float)(g->h_fp[i].a * (double)j + (g->h_fp[i].c + 1.0)),
                                                          (float)g->h_fp[i].b);
        float idbits;
        memcpy(&idbits, &i, sizeof(float));
        angt[p] = make_float2(g->h_fp[i].scale, idbits);
    }
    cudaError_t ce;
    if ((ce = cudaMalloc(&g->d_rayt, sizeof(float2) * rayt.size())) != cudaSuccess ||
        (ce = cudaMemcpy(g->d_rayt, rayt.data(), sizeof(float2) * rayt.size(), cudaMemcpyHostToDevice)) != cudaSuccess ||
        (ce = cudaMalloc(&g->d_angt, sizeof(float2) * na)) != cudaSuccess ||
        (ce = cudaMemcpy(g->d_angt, angt.data(), sizeof(float2) * na, cudaMemcpyHostToDevice)) != cudaSuccess ||
        (ce = cudaMalloc(&g->d_zero_row, (size_t)std::max(d->n0, d->n1) * 16 * sizeof(float))) != cudaSuccess ||
        (ce = cudaMemset(g->d_zero_row, 0, (size_t)std::max(d->n0, d->n1) * 16 * sizeof(float))) != cudaSuccess ||
        (ce = cudaMalloc(&g->d_fp, sizeof(FpAngle) * na)) != cudaSuccess ||
        (ce = cudaMalloc(&g->d_bp, sizeof(BpAngle) * na)) != cudaSuccess ||
        (ce = cudaMalloc(&g->d_order, sizeof(int) * na)) != cudaSuccess ||
        (ce = cudaMemcpy(g->d_fp, g->h_fp, sizeof(FpAngle) * na, cudaMemcpyHostToDevice)) != cudaSuccess ||
        (ce = cudaMemcpy(g->d_bp, g->h_bp, sizeof(BpAngle) * na, cudaMemcpyHostToDevice)) != cudaSuccess ||
        (ce = cudaMemcpy(g->d_order, g->h_order, sizeof(int) * na, cudaMemcpyHostToDevice)) != cudaSuccess) {
        scd_geom_destroy(g);
        return scd_cuda_fail(ce, "scd_geom_create upload");
    }
    if (wts) {
        std::vector<float> w_pos((size_t)na), w_id((size_t)na);
        for (int p = 0; p < na; ++p) w_pos[p] = (float)wts[g->h_order[p]];
        for (int i = 0; i < na; ++i) w_id[i] = (float)wts[i];
        if ((ce = cudaMalloc(&g->d_angw, sizeof(float) * na)) != cudaSuccess ||
            (ce = cudaMemcpy(g->d_angw, w_pos.data(), sizeof(float) * na, cudaMemcpyHostToDevice)) != cudaSuccess ||
            (ce = cudaMalloc(&g->d_w, sizeof(float) * na)) != cudaSuccess ||
            (ce = cudaMemcpy(g->d_w, w_id.data(), sizeof(float) * na, cudaMemcpyHostToDevice)) != cudaSuccess) {
            scd_geom_destroy(g);
            return scd_cuda_fail(ce, "scd_geom_create_weighted upload");
        }
    }
    *out = g;
    return 0;
}

extern "C" int scd_geom_destroy(scd_geom_t *g)
{
    if (!g) return 0;
    if (g->d_fp) cudaFree(g->d_fp);
    if (g->d_bp) cudaFree(g->d_bp);
    if (g->d_order) cudaFree(g->d_order);
    if (g->d_rayt) cudaFree(g->d_rayt);
    if (g->d_angt) cudaFree(g->d_angt);
    if (g->d_zero_row) cudaFree(g->d_zero_row);
    if (g->d_angw) cudaFree(g->d_angw);
    if (g->d_w) cudaFree(g->d_w);
    free(g->h_fp); free(g->h_bp); free(g->h_order);
    free(g);
    return 0;
}

extern "C" int scd_geom_info(const scd_geom_t *g, int32_t *n0, int32_t *n1,
                             int32_t *n_angles, int32_t *n_det)
{
    if (!g) { scd_set_error("scd_geom_info: null handle"); return SCD_E_INVALID; }
    if (n0) *n0 = g->n0;
    if (n1) *n1 = g->n1;
    if (n_angles) *n_angles = g->n_angles;
    if (n_det) *n_det = g->n_det;
    return 0;
}

extern "C" int scd_set_tuning(scd_geom_t *g, const char *key, int value)
{
    if (!g || !key) { scd_set_error("scd_set_tuning: null argument"); return SCD_E_INVALID; }
    if (!strcmp(key, "fp_samples")) g->tune_fp_samples = value;
    else if (!strcmp(key, "fp_angles")) g->tune_fp_angles = value;
    else if (!strcmp(key, "fp_rows")) g->tune_fp_rows = value;
    else if (!strcmp(key, "fp_threads")) g->tune_fp_threads = value;
    else if (!strcmp(key, "fp_nbuf")) g->tune_fp_nbuf = value;
    else if (!strcmp(key, "fp_cluster")) g->tune_fp_cluster = value;
    else if (!strcmp(key, "fp_plan")) g->tune_fp_plan = value;
    else if (!strcmp(key, "fp_source")) g->tune_fp_source = value;
    else if (!strcmp(key, "fp_plan_cost")) g->tune_fp_plan_cost = value;
    else if (!strcmp(key, "fp_cls0")) g->tune_fp_cls0 = value;
    else if (!strcmp(key, "bp_tile")) g->tune_bp_tile = value;
    else if (!strcmp(key, "bp_share")) g->tune_bp_share = value;
    else if (!strcmp(key, "bp_rows")) {
        // tiles of fewer than 4 rows would outgrow the per-CTA partial-sum arrays of the CG workspace
        if (value != 0 && value != 1 && value < 4) { scd_set_error("scd_set_tuning: bp_rows must be 0, 1 or >= 4"); return SCD_E_INVALID; }
        g->tune_bp_rows = value;
    }
    else { scd_set_error("scd_set_tuning: unknown key '%s'", key); return SCD_E_INVALID; }
    return 0;
}
