// K2 (v2)  bp_tile -- pixel-driven linear-interpolation backprojector A*, batched, with the CG
// axpy and dot product fused into its epilogue.
//
// Replaces SimpleTrafo.trafo_adjoint (reference src/physics/trafo.py:61 -> ODL -> ASTRA par_bp),
// the `x + gamma*A*(A x)` axpy of `op` (src/samplers/utils.py:188-189) and the <p,d> / ||r||^2
// reductions of cg (src/utils/cg.py:22,27).  Arithmetic: SURVEY.md Appendix A, "A*".
//
// Like the forward projector (fp_march.cu) the kernel is bound by the shared-memory pipe (two
// taps per pixel, angle and sample), so the sinogram is read in a sample-interleaved layout
//
//   sino_il[group][angle][NB bins][SB]     SB = V*LPR samples interleaved per bin,
//                                          PADL zero bins before the detector, zero bins after
//
// in which the detector segment a pixel tile projects onto is ONE contiguous, 16-byte aligned
// byte range per angle: it is staged by cp.async.bulk (TMA unit) into an mbarrier ring of angle
// chunks by a producer warp.  fp_march writes this layout directly inside the CG solve; user
// sinograms are converted by sino_pack_kernel first.
//
//   CTA     = (32 x TH pixel tile, group of SB samples); 16 marching warps + 1 producer warp
//   lanes   = LPR consecutive lanes share a pixel, each owns V samples (one LDS.(32V) per tap);
//             pixels of a warp are adjacent along k1 (the contiguous image axis): taps of
//             neighbouring pixels are <= 1.01 bins apart -> conflict-free / broadcast
//   thread  = PPT pixels in a column (k0 .. k0+PPT-1), accumulators in registers
//   angle range [lo,hi): the angle-sharded variant (multi-GPU config 4) is the same kernel;
//             partial images are summed by the caller (NCCL).
//
// Matched adjoint (MT = true, geometries created with SCD_GEOM_MATCHED_ADJOINT): the exact transpose of the
// Joseph projector, c_w * J^T y = dphi * sum_i w_i sum_j k_i max(0, 1 - k_i |j - v|) y_ij with
// k_i = 1 / max(|ci|, |si|) -- the same march with the unit hat (1-f, f) replaced by a hat of unit area and
// half-width h_i = 1/k_i <= dx/ds < 1.5.  Views with h_i <= 1 keep the two taps floor(v), floor(v)+1 (and the
// pair march); the few near-axis views with h_i > 1 take three taps around round(v).  k_i and the 2/3-tap
// choice are derived per view from (ci, si) of the shared-memory table: warp-uniform.
#include "scd_internal.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>

#define BQ_NW        16
#define BQ_THREADS   (32 * (BQ_NW + 1))
#define BQ_MAX_NBUF  8
#define BQ_MAGIC      12582912.0f
#define BQ_MAGIC_BITS 0x4B400000

struct BqParams {
    const float   *sino_il;
    float         *out;
    const BpAngle *bp;
    int n0, n1, n_angles, n_det, batch;
    int angle_lo, angle_hi;
    int SEG;                 // bins per staged segment (multiple of 4)
    int AC, nbuf;            // angles per chunk, ring depth
    int share_taps;          // pair march (3 loads per pixel pair) where |ci| < 1
    int th_eff;              // rows of the tile in use (<= TH): balances single-wave launches over the SMs
    int PADL, NB;            // interleaved sinogram row
    size_t group_floats;     // n_angles * NB * SB
    BpEpilogue ep;
    unsigned long long *dbg;     // time stamps (scd_debug_set_stamps) or NULL
};

// ------------------------------------------------------------ sino pack ---
// user sinogram [B][n_angles][n_det] -> sino_il (angles [lo,hi) only), times the view weight w[a] of A* when
// w != NULL
// grid = (bin chunks of 256, angles in range, groups)
__global__ void __launch_bounds__(256)
sino_pack_kernel(const float *sino, float *sino_il, int n_angles, int n_det, int batch,
                 int angle_lo, int SB, int PADL, int NB, size_t group_floats, const float *w)
{
    __shared__ float tile[16][257];
    scd_pdl_wait();                               // predecessor complete, its writes visible
    scd_pdl_trigger();
    const int tid = threadIdx.x;
    const int J0 = blockIdx.x * 256, a = angle_lo + blockIdx.y, grp = blockIdx.z;
    const int j = J0 + tid;
    const float wa = w ? __ldg(w + a) : 1.f;
    for (int s = 0; s < SB; ++s) {
        const int b = grp * SB + s;
        float v = 0.f;
        if (b < batch && j >= PADL && j < PADL + n_det)
            v = __ldg(sino + ((size_t)b * n_angles + a) * n_det + (j - PADL));
        tile[s][tid] = w ? v * wa : v;
    }
    __syncthreads();
    float *dst = sino_il + (size_t)grp * group_floats + ((size_t)a * NB + J0) * SB;
    const int nj = min(256, NB - J0);
    for (int idx = tid; idx < nj * SB; idx += 256) {
        const int jj = idx / SB, s = idx - jj * SB;
        dst[idx] = tile[s][jj];
    }
}

// ----------------------------------------------------------------- tile ---
__device__ __forceinline__ unsigned bq_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bq_mbar_init(unsigned long long *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(bq_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void bq_mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(bq_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bq_mbar_arrive(unsigned long long *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(bq_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bq_mbar_wait(unsigned long long *bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "BQ_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra BQ_DONE;\n"
        "bra BQ_WAIT;\n"
        "BQ_DONE:\n"
        "}\n" :: "r"(bq_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bq_bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bq_smem_u32(bar)) : "memory");
}

template <int V> struct BqVec;
template <> struct BqVec<1> {
    typedef float T;
    template <int OFF> static __device__ __forceinline__ T ld(unsigned a)
    { T v; asm volatile("ld.shared.f32 %0, [%1+%2];\n" : "=f"(v) : "r"(a), "n"(OFF)); return v; }
};
template <> struct BqVec<2> {
    typedef float2 T;
    template <int OFF> static __device__ __forceinline__ T ld(unsigned a)
    { T v; asm volatile("ld.shared.v2.f32 {%0,%1}, [%2+%3];\n" : "=f"(v.x), "=f"(v.y) : "r"(a), "n"(OFF)); return v; }
};
template <> struct BqVec<4> {
    typedef float4 T;
    template <int OFF> static __device__ __forceinline__ T ld(unsigned a)
    {
        T v;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4+%5];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a), "n"(OFF));
        return v;
    }
};

// acc += l*wl + r*w; V >= 2 uses the packed fp32x2 FMA of sm_100 (FFMA2)
__device__ __forceinline__ void bq_tap(float (&p)[1], float l, float r, float wl, float w)
{ p[0] = fmaf(r, w, fmaf(l, wl, p[0])); }
__device__ __forceinline__ void bq_tap(float (&p)[2], float2 l, float2 r, float wl, float w)
{
    float2 a = make_float2(p[0], p[1]);
    a = __ffma2_rn(l, make_float2(wl, wl), a);
    a = __ffma2_rn(r, make_float2(w, w), a);
    p[0] = a.x; p[1] = a.y;
}
__device__ __forceinline__ void bq_tap(float (&p)[4], float4 l, float4 r, float wl, float w)
{
    const float2 wl2 = make_float2(wl, wl), w2 = make_float2(w, w);
    float2 a = make_float2(p[0], p[1]), b = make_float2(p[2], p[3]);
    a = __ffma2_rn(make_float2(l.x, l.y), wl2, a);
    b = __ffma2_rn(make_float2(l.z, l.w), wl2, b);
    a = __ffma2_rn(make_float2(r.x, r.y), w2, a);
    b = __ffma2_rn(make_float2(r.z, r.w), w2, b);
    p[0] = a.x; p[1] = a.y; p[2] = b.x; p[3] = b.y;
}

// acc += t0*a0 + t1*a1 + t2*a2 (three consecutive bins; one of a0, a2 is zero, see the pair march)
__device__ __forceinline__ void bq_tap3(float (&p)[1], float t0, float t1, float t2, float a0, float a1, float a2)
{ p[0] = fmaf(t2, a2, fmaf(t1, a1, fmaf(t0, a0, p[0]))); }
__device__ __forceinline__ void bq_tap3(float (&p)[2], float2 t0, float2 t1, float2 t2, float a0, float a1, float a2)
{
    float2 a = make_float2(p[0], p[1]);
    a = __ffma2_rn(t0, make_float2(a0, a0), a);
    a = __ffma2_rn(t1, make_float2(a1, a1), a);
    a = __ffma2_rn(t2, make_float2(a2, a2), a);
    p[0] = a.x; p[1] = a.y;
}
__device__ __forceinline__ void bq_tap3(float (&p)[4], float4 t0, float4 t1, float4 t2, float a0, float a1, float a2)
{
    const float2 w0 = make_float2(a0, a0), w1 = make_float2(a1, a1), w2 = make_float2(a2, a2);
    float2 a = make_float2(p[0], p[1]), b = make_float2(p[2], p[3]);
    a = __ffma2_rn(make_float2(t0.x, t0.y), w0, a);
    b = __ffma2_rn(make_float2(t0.z, t0.w), w0, b);
    a = __ffma2_rn(make_float2(t1.x, t1.y), w1, a);
    b = __ffma2_rn(make_float2(t1.z, t1.w), w1, b);
    a = __ffma2_rn(make_float2(t2.x, t2.y), w2, a);
    b = __ffma2_rn(make_float2(t2.z, t2.w), w2, b);
    p[0] = a.x; p[1] = a.y; p[2] = b.x; p[3] = b.y;
}

// Matched adjoint: the normalised hat k * max(0, 1 - k*d) at distance d from the pixel's detector coordinate
__device__ __forceinline__ float bq_hat(float k, float d) { return k * fmaxf(0.0f, fmaf(-k, d, 1.0f)); }

// Weights of the two taps floor(z), floor(z)+1 at fraction w = z - floor(z): (1-w, w), or the normalised hat (MT)
template <bool MT>
__device__ __forceinline__ void bq_w2(float k, float w, float &wl, float &wr)
{
    if (MT) { wl = bq_hat(k, w); wr = bq_hat(k, 1.0f - w); }
    else    { wl = 1.0f - w; wr = w; (void)k; }
}

// Pair march of two pixels of a column whose detector coordinates satisfy zlo <= zhi < zlo + 1: their four taps lie
// in the three consecutive bins starting at floor(zlo) -- 3 loads instead of 4.  The lower pixel takes (1-w, w) on bins
// 0, 1; the upper one (1-w, w, 0) or (0, 1-w, w).  The product with the exact zero changes nothing and the real taps
// are added in the order of the plain march: bit-identical to it.  MT: the same with the two hat weights of bq_w2.
template <int V, int SB, bool MT>
__device__ __forceinline__ void bq_pair(float (&acc_lo)[V], float (&acc_hi)[V], float zlo, float zhi, unsigned seg, float k)
{
    typedef BqVec<V> LD;
    typedef typename LD::T VT;
    const float tlo = __fadd_rd(zlo, BQ_MAGIC), thi = __fadd_rd(zhi, BQ_MAGIC);
    const float wlo = zlo - (tlo - BQ_MAGIC), whi = zhi - (thi - BQ_MAGIC);
    const int ilo = __float_as_int(tlo), ihi = __float_as_int(thi);
    const unsigned ad = seg + (unsigned)ilo * (unsigned)(SB * 4);
    const VT b0 = LD::template ld<0>(ad);
    const VT b1 = LD::template ld<SB * 4>(ad);
    const VT b2 = LD::template ld<2 * SB * 4>(ad);
    float ll, lr, ul, ur;
    bq_w2<MT>(k, wlo, ll, lr);
    bq_tap(acc_lo, b0, b1, ll, lr);
    const bool s = ihi != ilo;                                   // the upper pixel's left tap is bin 1
    bq_w2<MT>(k, whi, ul, ur);
    bq_tap3(acc_hi, b0, b1, b2, s ? 0.0f : ul, s ? ul : ur, s ? ur : 0.0f);
}

// V samples per lane, LPR lanes per pixel (SB = V*LPR), PPT pixels per thread; IL: the epilogue's images are
// sample-interleaved (il images); MT: matched adjoint (exact transpose of the Joseph projector)
template <int V, int LPR, int PPT, bool IL, bool MT = false>
__global__ void __launch_bounds__(BQ_THREADS, 2)
bp_tile_kernel(const BqParams P)
{
    typedef BqVec<V> LD;
    typedef typename LD::T VT;
    constexpr int SB = V * LPR;
    constexpr int RPW = 32 / LPR;          // pixels of a warp along k1
    constexpr int WX = LPR;                // warps along k1 (32 pixels)
    constexpr int WY = BQ_NW / WX;         // warps along k0
    constexpr int TH = WY * PPT;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int K0 = blockIdx.y * P.th_eff, K1 = blockIdx.x * 32;
    const int grp = blockIdx.z, b0 = grp * SB;
    const int nang = P.angle_hi - P.angle_lo;
    const int AC = P.AC, NBUF = P.nbuf;
    const unsigned SEGB = (unsigned)(P.SEG * SB * 4);
    const int nchunks = (nang + AC - 1) / AC;

    // shared memory: ring[nbuf][AC][SEG*SB] | mbarriers | per-angle constants | dot partials
    const size_t ring_bytes = (size_t)NBUF * AC * SEGB;
    unsigned long long *full = reinterpret_cast<unsigned long long *>(smem_raw + ring_bytes);
    unsigned long long *empty = full + BQ_MAX_NBUF;
    float4 *cst = reinterpret_cast<float4 *>(empty + BQ_MAX_NBUF);
    float *red = reinterpret_cast<float *>(cst + nang);

    scd_stamp(P.dbg, 0);                          // CTA start
    if (tid == 0) {
        for (int i = 0; i < NBUF; ++i) { bq_mbar_init(&full[i], 1); bq_mbar_init(&empty[i], BQ_NW); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    // ---- per-angle constants re-centred on this tile (fp64): the fp32 index arithmetic then
    // works on magnitudes < SEG
    {
        const int th = min(TH, P.n0 - K0), tw = min(32, P.n1 - K1);
        for (int i = tid; i < nang; i += BQ_THREADS) {
            const BpAngle A = P.bp[P.angle_lo + i];
            const double v00 = A.ci * (double)K0 + A.si * (double)K1 + A.oi;
            const double vmin = v00 + fmin(0.0, A.ci * (double)(th - 1)) + fmin(0.0, A.si * (double)(tw - 1));
            int j0 = (int)floor(vmin) - 1;                 // one bin of slack below (fp32 rounding)
            j0 = ((j0 + P.PADL) & ~3) - P.PADL;            // 16-byte aligned source whatever SB
            // zf = v - j0 >= 1: floor(zf) = segment index of the left tap
            cst[i] = make_float4((float)A.ci, (float)A.si, (float)(v00 - (double)j0), __int_as_float(j0));
        }
    }
    __syncthreads();
    scd_stamp(P.dbg, 1);                          // tables done
    scd_pdl_wait();                               // the producer of the sinogram has completed
    scd_pdl_trigger();
    scd_stamp(P.dbg, 2);                          // predecessor complete

    float acc[PPT][V];
#pragma unroll
    for (int m = 0; m < PPT; ++m)
#pragma unroll
        for (int v = 0; v < V; ++v) acc[m][v] = 0.f;

    const int lr = lane / LPR, lq = lane - lr * LPR;
    const int wx = warp % WX, wy = warp / WX;
    const int k1 = K1 + wx * RPW + lr;
    const int k0b = K0 + wy * PPT;

    // The epilogue's addends are fetched before the march so that their latency hides behind it
    // (when they fit in a few registers; taller tiles load them in the epilogue, and so does the matched march,
    // whose extra weights would otherwise push the prefetched addends into local memory).
    constexpr bool PREF = PPT * V <= 8 && !MT;
    float pa1[PREF ? PPT : 1][V], pa2[PREF ? PPT : 1][V];
    if (IL) {
        if (PREF && warp < BQ_NW) {
#pragma unroll
            for (int m = 0; m < PPT; ++m) {
                const int k0 = k0b + m;
                const bool live = k0 < P.n0 && k1 < P.n1 && wy * PPT + m < P.th_eff;
                const size_t o = live ? (((size_t)grp * P.n0 + k0) * P.n1 + k1) * SB + lq * V : 0;
                VT v1, v2;
                float *f1 = reinterpret_cast<float *>(&v1), *f2 = reinterpret_cast<float *>(&v2);
#pragma unroll
                for (int v = 0; v < V; ++v) f1[v] = f2[v] = 0.f;
                if (live && P.ep.add1) v1 = *reinterpret_cast<const VT *>(P.ep.add1 + o);
                if (live && P.ep.add2) v2 = *reinterpret_cast<const VT *>(P.ep.add2 + o);
#pragma unroll
                for (int v = 0; v < V; ++v) { pa1[PREF ? m : 0][v] = f1[v]; pa2[PREF ? m : 0][v] = f2[v]; }
            }
        }
    } else
    if (PREF && warp < BQ_NW) {
#pragma unroll
        for (int m = 0; m < PPT; ++m)
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const int b = b0 + lq * V + v, k0 = k0b + m;
                const bool live = b < P.batch && k0 < P.n0 && k1 < P.n1 && wy * PPT + m < P.th_eff;
                const size_t o = live ? ((size_t)b * P.n0 + k0) * P.n1 + k1 : 0;
                pa1[PREF ? m : 0][v] = (live && P.ep.add1) ? P.ep.add1[o] : 0.f;
                pa2[PREF ? m : 0][v] = (live && P.ep.add2) ? P.ep.add2[o] : 0.f;
            }
    }

    if (warp == BQ_NW) {
        // ------------------------------ producer warp ------------------------------
        const float *src0 = P.sino_il + (size_t)grp * P.group_floats;
        const unsigned ring0 = bq_smem_u32(smem_raw);
        int bi = 0; unsigned ph = 0;
        for (int c = 0; c < nchunks; ++c) {
            if (c >= NBUF) bq_mbar_wait(&empty[bi], ph ^ 1u);
            const int nac = min(AC, nang - c * AC);
            if (lane == 0) bq_mbar_expect_tx(&full[bi], (unsigned)nac * SEGB);
            __syncwarp();
            for (int i = lane; i < nac; i += 32) {
                const int ia = c * AC + i;
                const int j0 = __float_as_int(cst[ia].w);
                const float *src = src0 + ((size_t)(P.angle_lo + ia) * P.NB + (size_t)(P.PADL + j0)) * SB;
                bq_bulk_g2s(ring0 + (unsigned)(bi * AC + i) * SEGB, src, SEGB, &full[bi]);
            }
            if (++bi == NBUF) { bi = 0; ph ^= 1u; }
        }
    } else {
        // ------------------------------ marching warps -----------------------------
        // pixels outside the image are computed at the clamped position and never stored
        const float lxf = (float)(min(k1, P.n1 - 1) - K1);
        float kyf[PPT];
#pragma unroll
        for (int m = 0; m < PPT; ++m) kyf[m] = (float)(min(k0b + m, P.n0 - 1) - K0);
        const unsigned lane_base = bq_smem_u32(smem_raw) + (unsigned)(lq * V * 4) - (unsigned)BQ_MAGIC_BITS * (unsigned)(SB * 4);
        const unsigned cst_base = bq_smem_u32(cst);
        const bool share_taps = (PPT % 2 == 0) && P.share_taps;
        const bool warp_rows_in_use = wy * PPT < P.th_eff;
        int bi = 0; unsigned ph = 0;
        for (int c = 0; c < nchunks; ++c) {
            bq_mbar_wait(&full[bi], ph);
            if (c == 0) scd_stamp(P.dbg, 3);      // first angle chunk landed (warp 0)
            const int nac = warp_rows_in_use ? min(AC, nang - c * AC) : 0;     // idle warps only keep the ring moving
            unsigned seg = lane_base + (unsigned)(bi * AC) * SEGB;
            unsigned ca = cst_base + (unsigned)(c * AC) * 16u;
#pragma unroll 2
            for (int i = 0; i < nac; ++i, seg += SEGB, ca += 16u) {
                const float4 cs = BqVec<4>::ld<0>(ca);
                const float vb = fmaf(lxf, cs.y, cs.z);
                float k = 1.0f;
                if (MT) {
                    const float h = fmaxf(fabsf(cs.x), fabsf(cs.y));     // half-width of the hat, < 1.5 bins
                    k = __fdividef(1.0f, h);
                    if (h > 1.0f) {
                        // near-axis view: three taps round(z)-1 .. round(z)+1 at distances 1+f, |f|, 1-f
                        // (f = z - round(z) in [-1/2, 1/2]); round(z)+-2 lie >= 1.5 > h away
#pragma unroll
                        for (int m = 0; m < PPT; ++m) {
                            const float z = fmaf(kyf[m], cs.x, vb);
                            const float t = __fadd_rd(z + 0.5f, BQ_MAGIC);  // round(z) in the mantissa (z >= 1)
                            const float f = z - (t - BQ_MAGIC);
                            const unsigned ad = seg + (unsigned)(__float_as_int(t) - 1) * (unsigned)(SB * 4);
                            const VT t0 = LD::template ld<0>(ad);
                            const VT t1 = LD::template ld<SB * 4>(ad);
                            const VT t2 = LD::template ld<2 * SB * 4>(ad);
                            bq_tap3(acc[m], t0, t1, t2, bq_hat(k, 1.0f + f), bq_hat(k, fabsf(f)), bq_hat(k, 1.0f - f));
                        }
                        continue;
                    }
                }
                if (PPT >= 2 && share_taps && fabsf(cs.x) <= 0.999f) {
                    // Pair march: the two pixels of a column pair are |ci| < 1 bins apart, so their four
                    // taps lie in THREE consecutive bins starting at the smaller left index: 3 loads
                    // instead of 4 (the shared-memory pipe is what bounds this kernel).  Each pixel
                    // weighs the three bins with (1-w, w, 0) or (0, 1-w, w); the products with an exact
                    // zero change nothing, the two real taps are added in the same order as in the
                    // plain march, so the results are bit-identical to it.
                    // The sign of ci is the same for the whole angle (warp-uniform), so it is known which pixel
                    // of the pair has the smaller detector coordinate: that one always weighs (1-w, w) on the first
                    // two bins -- two taps, no selects -- and only the other one needs the three-bin form.
                    if (cs.x >= 0.0f) {
#pragma unroll
                        for (int m = 0; m + 1 < PPT; m += 2)
                            bq_pair<V, SB, MT>(acc[m], acc[m + 1], fmaf(kyf[m], cs.x, vb), fmaf(kyf[m + 1], cs.x, vb), seg, k);
                    } else {
#pragma unroll
                        for (int m = 0; m + 1 < PPT; m += 2)
                            bq_pair<V, SB, MT>(acc[m + 1], acc[m], fmaf(kyf[m + 1], cs.x, vb), fmaf(kyf[m], cs.x, vb), seg, k);
                    }
                    continue;
                }
                float w[PPT];
                unsigned ad[PPT];
#pragma unroll
                for (int m = 0; m < PPT; ++m) {
                    const float z = fmaf(kyf[m], cs.x, vb);
                    const float t = __fadd_rd(z, BQ_MAGIC);                 // floor(z) in the mantissa
                    w[m] = z - (t - BQ_MAGIC);
                    ad[m] = seg + (unsigned)__float_as_int(t) * (unsigned)(SB * 4);
                }
                VT tl[PPT], tr[PPT];
#pragma unroll
                for (int m = 0; m < PPT; ++m) {
                    tl[m] = LD::template ld<0>(ad[m]);
                    tr[m] = LD::template ld<SB * 4>(ad[m]);
                }
#pragma unroll
                for (int m = 0; m < PPT; ++m) {
                    float wl, wr;
                    bq_w2<MT>(k, w[m], wl, wr);
                    bq_tap(acc[m], tl[m], tr[m], wl, wr);
                }
            }
            __syncwarp();
            if (lane == 0) bq_mbar_arrive(&empty[bi]);
            if (++bi == NBUF) { bi = 0; ph ^= 1u; }
        }
    }

    // ---- epilogue: axpy, second output, dot-product partials ---------------
    if (warp == 0 && lane == 0 && P.dbg) scd_stamp(P.dbg, 4);       // warp 0 done marching
    const BpEpilogue &E = P.ep;
    // banded output: the whole tile lies in band K0 / band_rows (band_rows is a multiple of the tile height)
    float *band_ptr = nullptr;
    int band_row0 = 0;
    if (E.n_bands) {
        const int band = K0 / E.band_rows;
        band_row0 = band * E.band_rows;
#pragma unroll
        for (int i = 0; i < SCD_MAX_BANDS; ++i) if (i == band) band_ptr = E.band_out[i];
    }
    if (band_ptr) {
        // Banded (peer) output: the tile goes through shared memory so that every warp stores whole
        // 128-byte runs of one image row -- the stores may cross NVLink, where 32-byte fragments are
        // expensive.  The ring and the tables are dead once every warp has finished marching.
        constexpr int TP = 33;                                     // padded row of 32 pixels
        float *tile = reinterpret_cast<float *>(smem_raw);         // [SB][TH][TP]
        __syncthreads();
        if (warp < BQ_NW) {
#pragma unroll
            for (int v = 0; v < V; ++v)
#pragma unroll
                for (int m = 0; m < PPT; ++m)
                    tile[((lq * V + v) * TH + wy * PPT + m) * TP + wx * RPW + lr] = E.c_acc * acc[m][v];
        }
        __syncthreads();
        for (int idx = tid; idx < SB * TH * 32; idx += BQ_THREADS) {
            const int x = idx & 31, sr = idx >> 5;
            const int row = sr % TH, sm = sr / TH;
            const int b = b0 + sm, k0 = K0 + row, kx = K1 + x;
            if (b < P.batch && k0 < P.n0 && kx < P.n1 && row < P.th_eff)
                band_ptr[((size_t)b * E.band_rows + (k0 - band_row0)) * P.n1 + kx] = tile[sr * TP + x];
        }
        scd_stamp(P.dbg, 5);
        return;
    }
    float dsum[V];
#pragma unroll
    for (int v = 0; v < V; ++v) dsum[v] = 0.f;
    if (IL) {
        if (warp < BQ_NW && k1 < P.n1) {
            float bet[V];
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const int b = b0 + lq * V + v;
                bet[v] = (E.mode == 1 && E.beta && b < P.batch) ? E.beta[b] : 0.f;
            }
#pragma unroll
            for (int m = 0; m < PPT; ++m) {
                const int k0 = k0b + m;
                if (k0 < P.n0 && wy * PPT + m < P.th_eff) {
                    const size_t o = (((size_t)grp * P.n0 + k0) * P.n1 + k1) * SB + lq * V;
                    VT v1, v2, vo, vp;
                    float *f1 = reinterpret_cast<float *>(&v1), *f2 = reinterpret_cast<float *>(&v2);
                    float *fo = reinterpret_cast<float *>(&vo), *fp = reinterpret_cast<float *>(&vp);
                    if (PREF) {
#pragma unroll
                        for (int v = 0; v < V; ++v) { f1[v] = pa1[PREF ? m : 0][v]; f2[v] = pa2[PREF ? m : 0][v]; }
                    } else {
#pragma unroll
                        for (int v = 0; v < V; ++v) f1[v] = f2[v] = 0.f;
                        if (E.add1) v1 = *reinterpret_cast<const VT *>(E.add1 + o);
                        if (E.add2) v2 = *reinterpret_cast<const VT *>(E.add2 + o);
                    }
                    if (E.mode == 1) {
#pragma unroll
                        for (int v = 0; v < V; ++v) {
                            const float pn = E.beta ? fmaf(bet[v], f2[v], f1[v]) : f1[v];     // p = r + beta p
                            const float dv = fmaf(E.c_acc, acc[m][v], pn);                    // d = p + gamma A*(q)
                            fp[v] = pn; fo[v] = dv;
                            dsum[v] = fmaf(pn, dv, dsum[v]);
                        }
                        *reinterpret_cast<VT *>(E.out2 + o) = vp;
                        *reinterpret_cast<VT *>(P.out + o) = vo;
                    } else {
#pragma unroll
                        for (int v = 0; v < V; ++v) {
                            float val = E.c_acc * acc[m][v];
                            if (E.add1) val = fmaf(E.c1, f1[v], val);
                            if (E.add2) val = fmaf(E.c2, f2[v], val);
                            fo[v] = val;
                            dsum[v] += val * (E.dot_with_add1 ? f1[v] : val);
                        }
                        *reinterpret_cast<VT *>(P.out + o) = vo;
                        if (E.out2) *reinterpret_cast<VT *>(E.out2 + o) = vo;
                    }
                }
            }
        }
    } else
    if (warp < BQ_NW && k1 < P.n1) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const int b = b0 + lq * V + v;
            if (b >= P.batch) continue;
#pragma unroll
            for (int m = 0; m < PPT; ++m) {
                const int k0 = k0b + m;
                if (k0 < P.n0 && wy * PPT + m < P.th_eff) {
                    const size_t o = ((size_t)b * P.n0 + k0) * P.n1 + k1;
                    float val = E.c_acc * acc[m][v];
                    float a1 = 0.f;
                    if (E.add1) { a1 = PREF ? pa1[PREF ? m : 0][v] : E.add1[o]; val = fmaf(E.c1, a1, val); }
                    if (E.add2) val = fmaf(E.c2, PREF ? pa2[PREF ? m : 0][v] : E.add2[o], val);
                    P.out[o] = val;
                    if (E.out2) E.out2[o] = val;
                    dsum[v] += val * (E.dot_with_add1 ? a1 : val);
                }
            }
        }
    }
    if (E.dot_part) {
        // lanes with equal lq hold the same samples: add over the pixels of the warp, then over warps
        if (warp < BQ_NW) {
#pragma unroll
            for (int v = 0; v < V; ++v) {
                float s = dsum[v];
#pragma unroll
                for (int off = 16; off >= LPR; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
                if (lr == 0) red[warp * SB + lq * V + v] = s;
            }
        }
        __syncthreads();
        if (tid < SB) {
            const int b = b0 + tid;
            if (b < P.batch) {
                float s = 0.f;
                for (int w = 0; w < BQ_NW; ++w) s += red[w * SB + tid];
                E.dot_part[(size_t)b * E.dot_stride + blockIdx.y * gridDim.x + blockIdx.x] = s;
            }
        }
    }
    scd_stamp(P.dbg, 5);                          // thread 0 done with the epilogue
}

// ------------------------------------------------------------- host side ---
struct BqConfig { int V, LPR, SB, PPT, TH, th_eff, SEG, AC, nbuf; size_t smem; dim3 grid; };

static BqConfig bq_choose(const scd_geom *g, int batch, int angle_lo, int angle_hi)
{
    BqConfig c;
    c.SB = scd_group_samples(g, batch);
    c.V = c.SB >= 4 ? 4 : c.SB;
    c.LPR = c.SB / c.V;
    const int WY = BQ_NW / c.LPR;
    // tile height: 8 rows when several lanes share a pixel (measured fastest at B = 8 .. 256: more,
    // shorter CTAs hide the staging latency), 16 rows for one lane per pixel
    const int groups = (batch + c.SB - 1) / c.SB;
    int th = c.LPR >= 2 ? 8 : 16;
    // 16 samples per group: 16-row tiles (two column pairs per thread: 6 tap loads in flight, 3 per pair)
    // once they still give >= ~3.5 waves of CTAs (measured at 256^2: B = 128: 162 -> 149 us, B = 256:
    // 310 -> 275 us, B = 64: 89 -> 95 us; 501^2 x 64 slices x 150 angles: 667 -> 579 us)
    if (c.LPR == 4 && (long)((g->n1 + 31) / 32) * ((g->n0 + 15) / 16) * groups >= 1024) th = 16;
    if (g->tune_bp_tile == 8 || g->tune_bp_tile == 16 || g->tune_bp_tile == 32) th = g->tune_bp_tile;
    if (c.LPR == 4 && th == 32) th = 16;       // 8 pixels x 4 samples per thread would not fit two CTAs per SM
    if (c.LPR == 1 && th == 8) th = 16;        // 16 warps along k0: at least one pixel each
    c.PPT = th / WY; c.TH = th;
    double span = 0.0;
    for (int i = angle_lo; i < angle_hi; ++i)
        span = std::max(span, std::fabs(g->h_bp[i].ci) * (th - 1) + std::fabs(g->h_bp[i].si) * 31.0);
    c.SEG = (((int)std::ceil(span) + 9) + 3) & ~3;
    const int nang = std::max(1, angle_hi - angle_lo);
    const size_t segb = (size_t)c.SEG * c.SB * 4;
    // chunks of ~28 KB, ring of ~90 KB (two CTAs per SM)
    c.AC = (int)std::max<size_t>(2, std::min<size_t>(32, (28 * 1024) / segb));
    c.AC = std::min(c.AC, nang);
    const int nchunks = (nang + c.AC - 1) / c.AC;
    c.nbuf = (int)std::max<size_t>(2, std::min<size_t>(BQ_MAX_NBUF, (90 * 1024) / (c.AC * segb)));
    c.nbuf = std::max(1, std::min(c.nbuf, nchunks));
    c.smem = (size_t)c.nbuf * c.AC * segb + 2 * BQ_MAX_NBUF * 8 + (size_t)nang * 16 + (size_t)BQ_NW * c.SB * 4 + 64;
    // Rows of the tile in use.  When the whole launch is a single wave of co-resident CTAs (two per SM) the
    // span is set by the SMs that host the most CTAs: with one pixel per thread, use fewer rows per tile
    // if that levels the load (256^2, B = 8: 256 tiles of 8 rows = two CTAs on 108 SMs and one on 40 ->
    // 296 tiles of 7 rows = two on every SM); the unused warps of a tile only keep the ring moving.
    c.th_eff = th;
    const long gx = (g->n1 + 31) / 32, slots = 2L * g->sm_count;
    if (c.PPT == 1 && g->tune_bp_rows != 1 && gx * ((g->n0 + th - 1) / th) * groups <= slots) {
        long best = ((gx * ((g->n0 + th - 1) / th) * groups + g->sm_count - 1) / g->sm_count) * th;
        for (int t = th - 1; t >= std::max(4, th / 2); --t) {
            const long tiles = gx * ((g->n0 + t - 1) / t) * groups;
            if (tiles > slots) break;
            const long cost = ((tiles + g->sm_count - 1) / g->sm_count) * t;
            if (cost < best) { best = cost; c.th_eff = t; }
        }
    }
    if (g->tune_bp_rows >= 4 && g->tune_bp_rows <= th && c.PPT == 1) c.th_eff = g->tune_bp_rows;
    c.grid = dim3((g->n1 + 31) / 32, (g->n0 + c.th_eff - 1) / c.th_eff, groups);
    return c;
}

int scd_bp_ctas_per_sample(const scd_geom *g, int batch)
{
    BqConfig c = bq_choose(g, batch, 0, g->n_angles);
    return (int)(c.grid.x * c.grid.y);
}

size_t scd_sino_il_bytes(const scd_geom *g, int batch)
{
    if (!g || batch <= 0) return 0;
    // the group size may be overridden by tuning: size for the worst case
    size_t need = 0;
    for (int SB = 1; SB <= 16; SB <<= 1)
        need = std::max(need, (size_t)((batch + SB - 1) / SB) * g->n_angles * g->il_nb * SB * 4);
    return need + 256;
}

template <int V, int LPR, int PPT, bool IL, bool MT>
static int bq_launch_mt(const BqParams &P, const BqConfig &c, cudaStream_t st, int device)
{
    static ScdSmemAttr attr = {};        // per instantiation
    SCD_CUDA(scd_ensure_smem(bp_tile_kernel<V, LPR, PPT, IL, MT>, attr, device, c.smem));
    SCD_CUDA(scd_launch_kernel(bp_tile_kernel<V, LPR, PPT, IL, MT>, c.grid, dim3(BQ_THREADS), c.smem, st, 0, P));
    SCD_LAUNCH_CHECK("bp_tile_kernel");
    return 0;
}

// the pixel-driven or the matched march, by the geometry
template <int V, int LPR, int PPT, bool IL>
static int bq_launch_t(const BqParams &P, const BqConfig &c, cudaStream_t st, const scd_geom *g)
{
    return g->matched ? bq_launch_mt<V, LPR, PPT, IL, true>(P, c, st, g->device)
                      : bq_launch_mt<V, LPR, PPT, IL, false>(P, c, st, g->device);
}

// banded output: every tile lies inside one band and every band has somewhere to go
static int bq_check_bands(const scd_geom *g, const BpEpilogue &ep)
{
    if (ep.n_bands > SCD_MAX_BANDS || ep.band_rows <= 0 || ep.band_rows % 32 != 0 ||
        (long)ep.n_bands * ep.band_rows < g->n0) {
        scd_set_error("scd_bp: bad band layout (%d bands of %d rows for %d image rows; rows must be a multiple of 32)",
                      ep.n_bands, ep.band_rows, g->n0);
        return SCD_E_INVALID;
    }
    for (int i = 0; i < ep.n_bands; ++i)
        if (!ep.band_out[i]) { scd_set_error("scd_bp: null band pointer"); return SCD_E_INVALID; }
    return 0;
}

int scd_launch_bp_il(const scd_geom *g, const float *sino_il, float *out, int batch,
                     int angle_lo, int angle_hi, const BpEpilogue &ep, cudaStream_t st)
{
    if (!g || !sino_il || (!out && !ep.n_bands)) { scd_set_error("scd_bp: null argument"); return SCD_E_INVALID; }
    if (batch <= 0) return 0;
    if (ep.n_bands) {
        const int rc = bq_check_bands(g, ep);
        if (rc) return rc;
    }
    BqConfig c = bq_choose(g, batch, angle_lo, angle_hi);
    if (ep.n_bands && c.th_eff != c.TH) {          // bands are aligned to whole tiles
        c.th_eff = c.TH;
        c.grid.y = (g->n0 + c.TH - 1) / c.TH;
    }
    if (c.grid.z > 65535) { scd_set_error("scd_bp: batch too large"); return SCD_E_INVALID; }
    if (c.smem > (size_t)g->smem_optin) { scd_set_error("scd_bp: angle table does not fit in shared memory"); return SCD_E_INVALID; }
    BqParams P = BqParams();                       // value-initialised (the epilogue carries default member initialisers)
    P.sino_il = sino_il; P.out = out; P.bp = g->d_bp;
    P.n0 = g->n0; P.n1 = g->n1; P.n_angles = g->n_angles; P.n_det = g->n_det; P.batch = batch;
    P.angle_lo = angle_lo; P.angle_hi = angle_hi; P.SEG = c.SEG; P.AC = c.AC; P.nbuf = c.nbuf;
    P.PADL = g->il_padl; P.NB = g->il_nb; P.group_floats = (size_t)g->n_angles * g->il_nb * c.SB;
    P.ep = ep; P.dbg = scd_debug_stamps();
    P.share_taps = g->tune_bp_share == 1 ? 0 : 1;
    P.th_eff = c.th_eff;
    if (ep.n_bands) c.smem = std::max(c.smem, (size_t)c.SB * c.TH * 33 * 4);     // staging tile of the banded epilogue
    const int WY = BQ_NW / c.LPR;
    (void)WY;
    if (ep.il) {
        if (c.V == 2 || ep.n_bands) { scd_set_error("scd_bp: interleaved images need groups of 1 or >= 4 samples and no bands"); return SCD_E_INVALID; }
        if (ep.mode == 1 && (!ep.add1 || !ep.out2 || (ep.beta && !ep.add2))) { scd_set_error("scd_bp: direction step needs r, p"); return SCD_E_INVALID; }
#define BQ_CASE_IL(LL, PP) if (c.V == 4 && c.LPR == LL && c.PPT == PP) return bq_launch_t<4, LL, PP, true>(P, c, st, g);
        BQ_CASE_IL(1, 1) BQ_CASE_IL(1, 2) BQ_CASE_IL(2, 1) BQ_CASE_IL(2, 2) BQ_CASE_IL(2, 4) BQ_CASE_IL(4, 2) BQ_CASE_IL(4, 4)
#undef BQ_CASE_IL
        if (c.V == 1 && c.PPT == 1) return bq_launch_t<1, 1, 1, true>(P, c, st, g);      // one sample per group
        if (c.V == 1 && c.PPT == 2) return bq_launch_t<1, 1, 2, true>(P, c, st, g);
    }
#define BQ_CASE(VV, LL, PP) if (c.V == VV && c.LPR == LL && c.PPT == PP) return bq_launch_t<VV, LL, PP, false>(P, c, st, g);
    BQ_CASE(1, 1, 1) BQ_CASE(1, 1, 2) BQ_CASE(2, 1, 1) BQ_CASE(2, 1, 2) BQ_CASE(4, 1, 1) BQ_CASE(4, 1, 2)
    BQ_CASE(4, 2, 1) BQ_CASE(4, 2, 2) BQ_CASE(4, 2, 4) BQ_CASE(4, 4, 2) BQ_CASE(4, 4, 4)
#undef BQ_CASE
    scd_set_error("scd_bp: unsupported config V=%d LPR=%d PPT=%d", c.V, c.LPR, c.PPT);
    return SCD_E_INVALID;
}

int scd_launch_sino_pack(const scd_geom *g, const float *sino, float *sino_il, int batch,
                         int angle_lo, int angle_hi, cudaStream_t st, bool weighted)
{
    if (batch <= 0 || angle_hi <= angle_lo) return 0;
    const int SB = scd_group_samples(g, batch);
    const int groups = (batch + SB - 1) / SB;
    dim3 grid((g->il_nb + 255) / 256, angle_hi - angle_lo, groups);
    if (grid.y > 65535 || grid.z > 65535) { scd_set_error("scd_bp: too many angles / samples"); return SCD_E_INVALID; }
    const float *w = weighted ? g->d_w : nullptr;
    SCD_CUDA(scd_launch_kernel(sino_pack_kernel, grid, dim3(256), 0, st, 0, sino, sino_il, g->n_angles, g->n_det, batch,
                               angle_lo, SB, g->il_padl, g->il_nb, (size_t)g->n_angles * g->il_nb * SB, w));
    SCD_LAUNCH_CHECK("sino_pack_kernel");
    return 0;
}

// ----------------------------------------------------- user-layout entry ---
int scd_launch_bp(const scd_geom *g, const float *sino, float *out, int batch,
                  int angle_lo, int angle_hi, const BpEpilogue &ep, void *scratch, size_t scratch_bytes,
                  cudaStream_t st, bool weighted)
{
    if (g && batch == 0) return 0;                 // empty batch: nothing to do (pointers may be null)
    if (!g || !sino || (!out && !ep.n_bands)) { scd_set_error("scd_bp: null argument"); return SCD_E_INVALID; }
    if (batch < 0 || angle_lo < 0 || angle_hi > g->n_angles || angle_lo > angle_hi) {
        scd_set_error("scd_bp: bad batch/angle range (batch=%d, angles [%d,%d) of %d)",
                      batch, angle_lo, angle_hi, g->n_angles);
        return SCD_E_INVALID;
    }
    if (batch == 0) return 0;
    if (ep.n_bands) {                              // before the re-layout: a rejected call writes nothing
        const int rc = bq_check_bands(g, ep);
        if (rc) return rc;
    }
    const uintptr_t sp = ((uintptr_t)scratch + 127) & ~(uintptr_t)127;
    const size_t need = scd_sino_il_bytes(g, batch) - 256;
    if (!scratch || sp + need > (uintptr_t)scratch + scratch_bytes) {
        scd_set_error("scd_bp: scratch too small (%zu bytes given, %zu needed; see scd_bp_scratch_bytes)",
                      scratch_bytes, need + 256);
        return SCD_E_WORKSPACE;
    }
    int rc = scd_launch_sino_pack(g, sino, (float *)sp, batch, angle_lo, angle_hi, st, weighted);
    if (rc) return rc;
    return scd_launch_bp_il(g, (const float *)sp, out, batch, angle_lo, angle_hi, ep, st);
}

int scd_bp_ctas_per_sample_max(const scd_geom *g, int batch)
{
    // workspace sizing: independent of the tuning knobs (smallest tile in use = 32 x 4 pixels)
    (void)batch;
    return ((g->n1 + 31) / 32) * ((g->n0 + 3) / 4);
}
