// K1 (v4)  fp_march -- ray-driven Joseph forward projector A, batched over samples.
//
// Replaces SimpleTrafo.trafo (reference src/physics/trafo.py:58), which reaches ASTRA's par_fp
// through ODL one image at a time.  Arithmetic follows SURVEY.md Appendix A: march along the
// dominant axis, linear interpolation across it, weight dx/max(|cos|,|sin|), zero outside.
//
// The binding resource of Joseph's method is the shared-memory pipe (8 B per ray-step and
// sample, DESIGN.md), so the layout is chosen to spend no wavefront on bank conflicts and none
// on rays that miss the image:
//
//   packed image  packed[group][class][row][pixel][SB]   (fp_packq_kernel)
//                 SB = V*LPR samples interleaved per pixel; class 1 is the transposed image so
//                 the march is class-agnostic; 1 zero pixel left, 2 right, rows padded to x8.
//   lanes         LPR consecutive lanes share one ray, each owns V samples (one LDS.(32V) per
//                 tap).  With SB = 16 a quarter-warp reads two pixels of 64 B: it conflicts only
//                 when neighbouring rays are two pixels apart (9 % of the wavefronts at 256^2).
//   warp          a "chunk" of RPW = 32/LPR adjacent rays; chunks of the NA angles of the CTA
//                 are dealt round-robin to the 15 marching warps (NSLOT chunks per warp).  A
//                 chunk whose rays all miss the image in a strip is skipped (warp vote).
//   accumulators  registers, for the whole march: NSLOT*V per thread.
//   strips        TR rows of the packed image = one contiguous byte range, fetched by a
//                 producer warp with cp.async.bulk (TMA unit) into an mbarrier ring
//                 (full/empty barriers; no CTA-wide barrier inside the march).
//   il image      groups of >= 4 samples (and a single sample) need no packed copy at all: the image is kept
//                 sample-interleaved, img_il[group][k0][k1][SB] (no pads).  Class 0 (strip rows = image
//                 rows): a row is one contiguous byte range -> one 1-D bulk copy per strip row into the
//                 row-major strip [row][pixel][SB] of the packed path (pad pixels zeroed once in shared
//                 memory).  Class 1 (strip rows = image columns): 3-D TENSOR copies
//                 (cp.async.bulk.tensor.3d, SASS UTMALDG) with boxes {TR*SB, pixels, 1} -- TR*SB*4-byte
//                 pieces gathered with the image's row stride -- which land PIXEL-MAJOR,
//                 [pixel][row][SB]: the transposed orientation is never materialised in HBM; its zero
//                 pad pixels / pad rows come from the unit's out-of-bounds fill.  In the
//                 pixel-major layout the rays of a quarter-warp visit the rows of a strip in
//                 different (XOR-rotated) orders, so their 128-byte wavefront never collides
//                 whatever the ray spacing (the row-major layout conflicts when two rays are two
//                 pixels apart).  Inside CG the vectors live in this layout for the whole solve
//                 (cg_solver.cu).
//   cluster       for small batches the rows are split over a cluster of CS CTAs; partial line
//                 integrals are exchanged through distributed shared memory and added in rank
//                 order (deterministic, no atomics).
#include "scd_internal.cuh"
#include <cuda.h>                 // CUtensorMap (the encoder is fetched through the runtime: no libcuda link)
#include <cooperative_groups.h>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <functional>
#include <vector>

namespace cg = cooperative_groups;

#define MQ_MAX_NBUF  8
#define MQ_MAX_RUNS  8
#define MQ_MAGIC      12582912.0f       /* 1.5 * 2^23: float add rounds to integer */
#define MQ_MAGIC_BITS 0x4B400000

struct MqRun { int cls, first, count, na, unit0; };   // `count` angles from order[first], `na` per unit

struct MqLayout {
    int SB;
    int pitch[2];            // pixels per packed row, per class (ncols + 3)
    int rows[2];             // packed rows per class (multiple of 8)
    size_t cls_off[2];       // float offset of class c inside a group
    size_t group_floats;     // floats per sample group
};

struct MqParams {
    const float   *img;
    float         *sino;     // user layout [batch][n_angles][n_det] or NULL
    float         *sino_il;  // interleaved layout [group][n_angles][il_nb][SB] (bp_tile.cu) or NULL
    float         *packed;
    const FpAngle *fp;
    const float2  *rayt;     // [order position][n_det] (u0 + 1, b) per ray
    const float2  *angt;     // [order position] (scale, angle id bits)
    const float   *angw;     // [order position] view weight of the interleaved output (A* quadrature) or NULL
    const float   *w_il;     // measurement weights W in the layout of sino_il (scd_sino_weights_pack) or NULL
    const int     *order;
    int n0, n1, n_angles, n_det, batch;
    int NA;                  // largest number of angles per CTA (sizes the tables)
    int nbuf;                // ring depth
    int CS;                  // cluster size = row split
    int rows_per_cta;        // multiple of 8
    int ring_bytes;          // strip ring (aliased by the partial sums), tables follow
    int il_padl, il_nb;      // interleaved sinogram row: zero bins before / total bins
    unsigned long long *dbg;     // time stamps (scd_debug_set_stamps) or NULL
    int groups, n_big, n_units;  // sample groups; units of the full NA angles (they come first); all units
    int need_cls[2];
    MqLayout L;
    int n_runs;
    MqRun runs[MQ_MAX_RUNS];
    // tensor-copy source (tma != 0): strip rows come from the sample-interleaved image through the two tensor
    // maps passed next to this struct; spitch = pixels per shared-memory strip row (nbox boxes of bw pixels)
    int tma;
    int spitch[2], nbox[2], bw[2];
    const float *zero_row;   // >= max(n0, n1) * 16 zero floats (source of the strip rows beyond the image)
    int lead;                // pixels before pixel 0 in a row-major class-0 strip row (bulk rows need a 16-byte aligned start)
    int cls0_pm;             // class 0 fetched pixel-major by tensor copies too (4-D map tm0) instead of row-major bulk rows
    // output recurrence of the CG solve (acc_mode != 0): q = A r + beta q_old with
    // beta = sum(rr_new_part) / sum(rr_old_part) per sample (q_{k} = A p_k, p_k = r_k + beta p_{k-1});
    // the per-sample beta is also stored to beta_out for the backprojector's direction update
    int acc_mode;
    const float *rr_new_part; int rr_new_n; const float *rr_old_part; int rr_old_n; int part_stride;
    float *beta_out;
};

// ------------------------------------------------------------------ pack ---
// One block = one 16x16 image tile of one sample group; it writes the tile into both packed
// orientations, including the pad pixels and the zero rows that round the row count up to x8.
// Optional prologue (the producer of the image is fused into the pack pass):
//   mode 1  CG direction update   p = r + beta p        (reference src/utils/cg.py:35-38)
//   mode 2  Tweedie + CG rhs      xhat0, b              (reference src/samplers/utils.py:370-378, :197)
#define PK_T 16
template <int MODE, int SB>
__global__ void __launch_bounds__(256)
fp_packq_kernel(const MqParams P, const FpPrologue Q)
{
    constexpr int SBP = SB >= 4 ? SB + 4 : SB + 1;
    __shared__ __align__(16) float tile[PK_T * (PK_T + 1) * SBP];
    __shared__ float coef[SB][2];
    scd_pdl_wait();                               // predecessor complete, its writes visible
    scd_pdl_trigger();
    const int grp = blockIdx.z;
    const int tid = threadIdx.x;
    const int K0 = blockIdx.y * PK_T, K1 = blockIdx.x * PK_T;
    const size_t isz = (size_t)P.n0 * P.n1;

    // thread = pixel; four samples per round, their loads issued together (memory-level parallelism)
    const int ty = tid >> 4, tx = tid & 15;
    const int k0 = K0 + ty, k1 = K1 + tx;
    const bool in_img = k0 < P.n0 && k1 < P.n1;
    float a[4], c[4], e[4];
    bool live[4];
    auto load_round = [&](int s0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int s = s0 + i, b = grp * SB + s;
            live[i] = in_img && s < SB && b < P.batch;
            a[i] = c[i] = e[i] = 0.f;
            if (live[i]) {
                const size_t o = b * isz + (size_t)k0 * P.n1 + k1;
                if (MODE == 0) a[i] = __ldg(P.img + o);
                else if (MODE == 1) { a[i] = Q.p[o]; c[i] = Q.r[o]; }
                else { a[i] = Q.x[o]; c[i] = Q.s[o]; e[i] = Q.atb[o]; }
            }
        }
    };
    load_round(0);                                // in flight while the per-sample scalars are formed

    if (MODE != 0) {
        // per-sample scalars, one warp per sample (8 warps, SB <= 16 samples)
        const int w = tid >> 5, lane = tid & 31;
        for (int s = w; s < SB; s += 8) {
            const int b = grp * SB + s;
            if (b >= P.batch) continue;
            if (MODE == 1) {
                float rn = 0.f, ro = 0.f;
                for (int i = lane; i < Q.rr_new_n; i += 32) rn += Q.rr_new_part[(size_t)b * Q.part_stride + i];
                for (int i = lane; i < Q.rr_old_n; i += 32) ro += Q.rr_old_part[(size_t)b * Q.part_stride + i];
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    rn += __shfl_xor_sync(0xffffffffu, rn, off);
                    ro += __shfl_xor_sync(0xffffffffu, ro, off);
                }
                if (lane == 0) coef[s][0] = __fdiv_rn(rn, ro);               // beta
            } else if (lane == 0) {
                long long idx = (long long)Q.t[b] + 1;                       // Tensor.long() + 1
                idx = idx < 0 ? 0 : (idx >= Q.n_table ? Q.n_table - 1 : idx);
                const float ab = Q.abar[idx];
                const float mean = __fsqrt_rn(ab);
                coef[s][0] = __fsqrt_rn(__fsub_rn(1.0f, ab));                // std_t
                coef[s][1] = __fdiv_rn(1.0f, mean);                          // mean_t^-1
            }
        }
        __syncthreads();
    }

    // ---- produce the tile ----
    {
        float *tp = tile + (ty * (PK_T + 1) + tx) * SBP;
        for (int s0 = 0; s0 < SB; s0 += 4) {
            if (s0 > 0) load_round(s0);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int s = s0 + i, b = grp * SB + s;
                float v = 0.f;
                if (live[i]) {
                    const size_t o = b * isz + (size_t)k0 * P.n1 + k1;
                    if (MODE == 0) {
                        v = a[i];
                    } else if (MODE == 1) {
                        v = fmaf(coef[s][0], a[i], c[i]);
                        Q.p[o] = v;
                    } else {
                        const float u = __fsub_rn(a[i], __fmul_rn(c[i], coef[s][0]));
                        v = __fmul_rn(u, coef[s][1]);
                        Q.xhat0[o] = v;
                        Q.b[o] = __fadd_rn(v, __fmul_rn(Q.gamma, e[i]));
                    }
                }
                if (s < SB) tp[s] = v;
            }
        }
    }
    __syncthreads();

    // ---- write both orientations: lanes = (pixel, quad of samples), 16 B (or 4*V B) per lane ----
    constexpr int VQ = SB >= 4 ? 4 : SB;          // floats per lane
    constexpr int LQ = SB / VQ;                   // lanes per pixel
    float *dst = P.packed + (size_t)grp * P.L.group_floats;
#pragma unroll 1
    for (int cls = 0; cls < 2; ++cls) {
        if (!P.need_cls[cls]) continue;
        const int pitch = P.L.pitch[cls];
        const int nrow_img = cls == 0 ? P.n0 : P.n1;     // rows with data
        const int ncol = cls == 0 ? P.n1 : P.n0;
        const int nrow_pk = P.L.rows[cls];
        float *d = dst + P.L.cls_off[cls];
        for (int idx = tid; idx < PK_T * PK_T * LQ; idx += 256) {
            const int q = idx % LQ, pix = idx / LQ;
            const int cl = pix % PK_T, rl = pix / PK_T;          // column fastest -> contiguous stores
            const int row = (cls == 0 ? K0 : K1) + rl, col = (cls == 0 ? K1 : K0) + cl;
            if (row >= nrow_pk || col >= ncol) continue;
            const float *tp = tile + (cls == 0 ? (rl * (PK_T + 1) + cl) : (cl * (PK_T + 1) + rl)) * SBP + q * VQ;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (row < nrow_img) {
#pragma unroll
                for (int i = 0; i < 4; ++i) if (i < VQ) v[i] = tp[i];
            }
            float *o = d + ((size_t)row * pitch + 1 + col) * SB + q * VQ;
            if (VQ == 4) *reinterpret_cast<float4 *>(o) = make_float4(v[0], v[1], v[2], v[3]);
            else if (VQ == 2) *reinterpret_cast<float2 *>(o) = make_float2(v[0], v[1]);
            else o[0] = v[0];
            if (col == 0) {
                for (int i = 0; i < VQ; ++i) o[i - SB] = 0.f;
            }
            if (col == ncol - 1) {
                for (int i = 0; i < VQ; ++i) { o[SB + i] = 0.f; o[2 * SB + i] = 0.f; }
            }
        }
    }
}

// ----------------------------------------------------------------- march ---
__device__ __forceinline__ unsigned mq_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mq_mbar_init(unsigned long long *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(mq_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mq_mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(mq_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mq_mbar_arrive(unsigned long long *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(mq_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mq_mbar_wait(unsigned long long *bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MQ_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MQ_DONE;\n"
        "bra MQ_WAIT;\n"
        "MQ_DONE:\n"
        "}\n" :: "r"(mq_smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared through the TMA unit, completion on an mbarrier
__device__ __forceinline__ void mq_bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 :: "r"(mq_smem_u32(dst)), "l"(src), "r"(bytes), "r"(mq_smem_u32(bar)) : "memory");
}

// 3-D tiled tensor copy global -> shared through the TMA unit (SASS UTMALDG), completion on an mbarrier;
// elements outside the tensor are filled with zeros
__device__ __forceinline__ void mq_tensor_g2s(unsigned dst, const CUtensorMap *tm, int c0, int c1, int c2,
                                              unsigned long long *bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n"
                 :: "r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(mq_smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mq_tensor4_g2s(unsigned dst, const CUtensorMap *tm, int c0, int c1, int c2, int c3,
                                               unsigned long long *bar)
{
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];\n"
                 :: "r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(mq_smem_u32(bar)) : "memory");
}

// Tap loads with explicit 32-bit shared-window addresses (a generic pointer would be re-mapped
// through the cluster window on every access).  volatile: they stay behind the mbarrier wait.
template <int V> struct MqVec;
template <> struct MqVec<1> {
    typedef float T;
    template <int OFF> static __device__ __forceinline__ T ld(unsigned a)
    { T v; asm volatile("ld.shared.f32 %0, [%1+%2];\n" : "=f"(v) : "r"(a), "n"(OFF)); return v; }
};
template <> struct MqVec<2> {
    typedef float2 T;
    template <int OFF> static __device__ __forceinline__ T ld(unsigned a)
    { T v; asm volatile("ld.shared.v2.f32 {%0,%1}, [%2+%3];\n" : "=f"(v.x), "=f"(v.y) : "r"(a), "n"(OFF)); return v; }
};
template <> struct MqVec<4> {
    typedef float4 T;
    template <int OFF> static __device__ __forceinline__ T ld(unsigned a)
    {
        T v;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4+%5];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a), "n"(OFF));
        return v;
    }
};

// acc += l*wl + r*w for the V samples of a lane.  V >= 2 uses the packed fp32x2 FMA of sm_100
// (FFMA2: two independent round-to-nearest FMAs per issue slot, same results as two FFMAs).
__device__ __forceinline__ void mq_tap(float (&p)[1], float l, float r, float wl, float w)
{ p[0] = fmaf(r, w, fmaf(l, wl, p[0])); }
__device__ __forceinline__ void mq_tap(float (&p)[2], float2 l, float2 r, float wl, float w)
{
    float2 a = make_float2(p[0], p[1]);
    a = __ffma2_rn(l, make_float2(wl, wl), a);
    a = __ffma2_rn(r, make_float2(w, w), a);
    p[0] = a.x; p[1] = a.y;
}
__device__ __forceinline__ void mq_tap(float (&p)[4], float4 l, float4 r, float wl, float w)
{
    const float2 wl2 = make_float2(wl, wl), w2 = make_float2(w, w);
    float2 a = make_float2(p[0], p[1]), b = make_float2(p[2], p[3]);
    a = __ffma2_rn(make_float2(l.x, l.y), wl2, a);
    b = __ffma2_rn(make_float2(l.z, l.w), wl2, b);
    a = __ffma2_rn(make_float2(r.x, r.y), w2, a);
    b = __ffma2_rn(make_float2(r.z, r.w), w2, b);
    p[0] = a.x; p[1] = a.y; p[2] = b.x; p[3] = b.y;
}

// The march of one warp over the strips of its CTA.  PM = pixel-major strips [pixel][row][SB] (tensor copies of
// class 1): the pixel stride is the compile-time TR*SB*4 and every ray visits the rows of a strip in the order
// rr ^ rot, rot = (ray index) mod (rays per quarter-warp) -- the rays that share a 128-byte wavefront then read
// different rows, i.e. different bank groups, wherever their pixels are.  Row-major strips: rot = 0.
template <int V, int LPR, int NSLOT, int TR, int NW, bool PM>
__device__ __forceinline__ void mq_march_rows(float (&acc)[NSLOT][V], const int (&eidx)[NSLOT], unsigned livemask, int NCH,
                                              int warp, int lane, int nst, int NBUF, int r_begin, int ncols,
                                              unsigned row_bytes, unsigned strip_bytes, unsigned char *tile0,
                                              const float2 *rays, unsigned long long *full, unsigned long long *empty,
                                              unsigned long long *dbg, unsigned lane_shift)
{
    typedef MqVec<V> LD;
    typedef typename LD::T VT;
    constexpr int SB = V * LPR;
    constexpr unsigned PS = PM ? TR * SB * 4 : SB * 4;           // bytes between neighbouring pixels of a row
    constexpr int QR = 8 / LPR < TR ? 8 / LPR : TR;              // rows the rotation spreads a quarter-warp over
    const int lr = lane / LPR, lq = lane - lr * LPR;
    const int rot = PM ? (lr & (QR - 1)) : 0;
    float cf[TR];                                                // row visited at unrolled step rr, as a float ...
    unsigned ro[TR];                                             // ... and its byte offset inside the strip
#pragma unroll
    for (int rr = 0; rr < TR; ++rr) {
        cf[rr] = (float)(rr ^ rot);
        ro[rr] = PM ? (unsigned)((rr ^ rot) * SB * 4) : (unsigned)rr * row_bytes;
    }
    const float zmax = (float)(ncols + 1);    // u = ncols: both taps on the right pads
    // shared-window address of this lane's samples in pixel 0 of row 0 of buffer 0, with the
    // mantissa offset of the floor trick folded in
    const unsigned lane_base = mq_smem_u32(tile0) + (unsigned)(lq * V * 4) - (unsigned)MQ_MAGIC_BITS * PS + lane_shift;
    const unsigned rays_base = mq_smem_u32(rays);
    int bi = 0; unsigned ph = 0;
    for (int st = 0; st < nst; ++st) {
        mq_mbar_wait(&full[bi], ph);
        if (st == 0) scd_stamp(dbg, 3);       // first strip landed (warp 0)
        const unsigned sbuf = lane_base + (unsigned)bi * strip_bytes;
        const float r0f = (float)(r_begin + st * TR);
#pragma unroll
        for (int k = 0; k < NSLOT; ++k) {
            if (warp + k * NW < NCH) {                              // warp-uniform
                const float2 ub = MqVec<2>::ld<0>(rays_base + (unsigned)eidx[k] * 8u);
                const float bf = ub.y;
                const float z0 = fmaf(r0f, bf, ub.x);
                const float z1 = fmaf((float)(TR - 1), bf, z0);
                // every ray of this chunk outside the image on every row of the strip
                const bool outside = !((livemask >> k) & 1u) || fmaxf(z0, z1) <= 0.0f || fminf(z0, z1) >= zmax;
                if (!__all_sync(0xffffffffu, outside)) {
                    float w[TR];
                    unsigned ad[TR];
#pragma unroll
                    for (int rr = 0; rr < TR; ++rr) {
                        // clamped position: outside the image both taps land on zero pad pixels
                        const float z = fminf(fmaxf(fmaf(cf[rr], bf, z0), 0.0f), zmax);
                        const float t = __fadd_rd(z, MQ_MAGIC);       // floor(z) in the mantissa
                        w[rr] = z - (t - MQ_MAGIC);
                        ad[rr] = sbuf + ro[rr] + (unsigned)__float_as_int(t) * PS;
                    }
                    VT tl[TR], tr[TR];
#pragma unroll
                    for (int rr = 0; rr < TR; ++rr) {
                        tl[rr] = LD::template ld<0>(ad[rr]);
                        tr[rr] = LD::template ld<PS>(ad[rr]);
                    }
#pragma unroll
                    for (int rr = 0; rr < TR; ++rr) mq_tap(acc[k], tl[rr], tr[rr], 1.0f - w[rr], w[rr]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mq_mbar_arrive(&empty[bi]);                   // this warp is done with buffer bi
        if (++bi == NBUF) { bi = 0; ph ^= 1u; }
    }
}

struct __align__(8) MqAng { float scale; int id; };

// V     samples per lane (vector width of a tap)
// LPR   lanes per ray            -> SB = V*LPR samples per group, RPW = 32/LPR rays per warp
// NSLOT ray chunks per warp      (accumulators: NSLOT*V registers)
// TR    rows per strip
// NWT   warps per CTA: NWT-1 marching warps + one producer warp
template <int V, int LPR, int NSLOT, int TR, int NWT>
__global__ void __launch_bounds__(32 * NWT, 1)
fp_march_kernel(const MqParams P, const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1)
{
    typedef MqVec<V> LD;
    typedef typename LD::T VT;
    constexpr int SB = V * LPR;
    constexpr int RPW = 32 / LPR;
    constexpr int NW = NWT - 1;
    constexpr int NTHR = 32 * NWT;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int CS = P.CS;
    const int rank = CS > 1 ? (int)cluster.block_rank() : 0;
    // linear CTA order: first the full-size units, group by group (the units of a group read
    // the same packed image: co-resident CTAs share it in L2), then the shorter units, largest
    // first across groups (they level the last round of the machine; measured: ordering them
    // by group instead costs 7 % at B = 256)
    int grp, unit;
    {
        const int lin = (int)blockIdx.x / CS;
        const int nbig_all = P.n_big * P.groups;
        if (lin < nbig_all) { grp = lin / P.n_big; unit = lin - grp * P.n_big; }
        else { const int l2 = lin - nbig_all; unit = P.n_big + l2 / P.groups; grp = l2 - (unit - P.n_big) * P.groups; }
    }

    // locate this unit's run without indexing the parameter array dynamically
    MqRun R = P.runs[0];
#pragma unroll
    for (int k = 1; k < MQ_MAX_RUNS; ++k)
        if (k < P.n_runs && unit >= P.runs[k].unit0) R = P.runs[k];
    const int pos0 = R.first + (unit - R.unit0) * R.na;
    const int na = min(R.na, R.first + R.count - pos0);
    const int cls = R.cls;
    const int nrows = cls == 0 ? P.n0 : P.n1;   // marching axis
    const int ncols = cls == 0 ? P.n1 : P.n0;   // interpolation axis
    const int pitch = P.tma ? P.spitch[cls] : P.L.pitch[cls];   // pixels per strip row in shared memory
    const int n_det = P.n_det;
    const int b0 = grp * SB;
    const unsigned row_bytes = (unsigned)(pitch * SB * 4);
    const unsigned strip_bytes = TR * row_bytes;

    // this CTA's rows: [r_begin, r_begin + nst*TR), inside the zero-padded packed rows
    const int r_begin = rank * P.rows_per_cta;
    const int r_end = min(r_begin + P.rows_per_cta, (nrows + 7) & ~7);
    const int nst = r_end > r_begin ? (r_end - r_begin) / TR : 0;

    // shared memory: strips[nbuf] (aliased by the partial line integrals red[SB][E] once the
    // march is over) | mbarriers | angle table | ray table (u0, b)
    const int NBUF = P.nbuf;
    unsigned char *tile0 = smem_raw;
    unsigned long long *full = reinterpret_cast<unsigned long long *>(smem_raw + P.ring_bytes);
    unsigned long long *empty = full + MQ_MAX_NBUF;
    MqAng *ang = reinterpret_cast<MqAng *>(empty + MQ_MAX_NBUF);
    float2 *rays = reinterpret_cast<float2 *>(ang + P.NA);
    float *red = reinterpret_cast<float *>(smem_raw);
    __shared__ float betas[16];

    const int E = na * n_det;
    const float *src = P.tma ? nullptr : P.packed + (size_t)grp * P.L.group_floats + P.L.cls_off[cls] +
                                         (size_t)r_begin * pitch * SB;

    scd_stamp(P.dbg, 0);                          // CTA start
    if (tid == 0) {
        for (int i = 0; i < NBUF; ++i) { mq_mbar_init(&full[i], 1); mq_mbar_init(&empty[i], NW); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    // ray table of this unit: zf = u + 1 (left pad pixel) at row 0 and the slope per row, both
    // evaluated in fp64 at geometry creation (constant data: read before the PDL wait)
    for (int e = tid; e < E; e += NTHR) rays[e] = __ldg(P.rayt + (size_t)pos0 * n_det + e);
    if (tid < na) {
        const float2 t = __ldg(P.angt + pos0 + tid);
        MqAng a; a.scale = t.x; a.id = __float_as_int(t.y); ang[tid] = a;
    }
    if (P.tma && cls == 0 && !P.cls0_pm) {
        // pad pixels (`lead` left, >= 2 right) of every row of every ring buffer: zero once, the row copies never touch them
        const int lead = P.lead;
        const int padr = pitch - lead - ncols;
        const int per_row = (lead + padr) * SB;
        for (int i = tid; i < NBUF * TR * per_row; i += NTHR) {
            const int row = i / per_row, k = i - row * per_row;
            float *rp = reinterpret_cast<float *>(tile0 + (size_t)row * row_bytes);
            rp[k < lead * SB ? k : (size_t)(ncols + lead) * SB + (k - lead * SB)] = 0.f;
        }
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");      // generic-proxy writes vs the async copies
    }
    __syncthreads();                              // mbarrier init + tables (+ pads) visible
    scd_stamp(P.dbg, 1);                          // tables done
    scd_pdl_wait();                               // the pack pass has completed: packed image visible
    scd_pdl_trigger();
    scd_stamp(P.dbg, 2);                          // predecessor complete

    float acc[NSLOT][V];
    int eidx[NSLOT];
    unsigned livemask = 0;
    const int nchunk = (n_det + RPW - 1) / RPW;
    const int NCH = na * nchunk;
    const int lr = lane / LPR, lq = lane - lr * LPR;
#pragma unroll
    for (int k = 0; k < NSLOT; ++k) {
#pragma unroll
        for (int v = 0; v < V; ++v) acc[k][v] = 0.f;
        const int C = warp + k * NW;
        eidx[k] = 0;
        if (warp < NW && C < NCH) {
            const int ai = C / nchunk, cc = C - ai * nchunk;
            const int j = cc * RPW + lr;
            if (j < n_det) livemask |= 1u << k;
            eidx[k] = ai * n_det + min(j, n_det - 1);
        }
    }

    if (warp == NW) {
        // ------------------------------ producer warp ------------------------------
        if (P.tma && cls == 0 && !P.cls0_pm) {
            // Class 0 (rows = image rows): a row of the interleaved image is one contiguous byte range -> one 1-D bulk
            // copy per strip row (lane rr), landing behind the left pad pixel of the row-major strip [row][pixel][SB];
            // the pad pixels of every ring buffer were zeroed above and are never overwritten.  Rows beyond the image
            // (the row count is rounded up to x8) are copied from a zero row.
            const bool mine = lane < TR;
            const unsigned dst0 = mq_smem_u32(tile0) + (unsigned)lane * row_bytes + (unsigned)(P.lead * SB * 4);
            const unsigned nbytes = (unsigned)ncols * (unsigned)(SB * 4);
            const float *img0 = P.img + (size_t)grp * nrows * ncols * SB;
            int bi = 0; unsigned ph = 0;
            for (int st = 0; st < nst; ++st) {
                if (st >= NBUF) mq_mbar_wait(&empty[bi], ph ^ 1u);      // previous use of this buffer released
                if (lane == 0) mq_mbar_expect_tx(&full[bi], TR * nbytes);
                __syncwarp();
                if (mine) {
                    const int row = r_begin + st * TR + lane;
                    const float *srow = row < nrows ? img0 + (size_t)row * ncols * SB : P.zero_row;
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                                 :: "r"(dst0 + (unsigned)bi * strip_bytes), "l"(srow), "r"(nbytes), "r"(mq_smem_u32(&full[bi])) : "memory");
                }
                if (++bi == NBUF) { bi = 0; ph ^= 1u; }
            }
        } else if (P.tma && cls == 0) {
            // Class 0, pixel-major: the image as the 4-D tensor (SB, n0, n1, groups) -- rows before pixels, i.e. with
            // the strides of dimensions 1 and 2 swapped -- and boxes {SB, TR, bw, 1}: SB*4-byte pieces that land
            // [pixel][row][SB] like class 1, so that the row rotation removes the bank conflicts here too
            const int nbox = P.nbox[0], bw = P.bw[0];
            const bool mine = lane < nbox;
            const unsigned dst0 = mq_smem_u32(tile0) + (unsigned)(lane * bw) * (unsigned)(TR * SB * 4);
            const int cpix = lane * bw - 1;
            int bi = 0; unsigned ph = 0;
            for (int st = 0; st < nst; ++st) {
                if (st >= NBUF) mq_mbar_wait(&empty[bi], ph ^ 1u);
                if (lane == 0) mq_mbar_expect_tx(&full[bi], strip_bytes);
                __syncwarp();
                if (mine) mq_tensor4_g2s(dst0 + (unsigned)bi * strip_bytes, &tm0, 0, r_begin + st * TR, cpix, grp, &full[bi]);
                if (++bi == NBUF) { bi = 0; ph ^= 1u; }
            }
        } else if (P.tma) {
            // Class 1 (rows = image columns): the image as a 3-D tensor (n1*SB, n0, groups); one copy per box of bw
            // pixels covering all TR rows, box {TR*SB, bw, 1}: the unit gathers TR*SB*4-byte pieces with the image's
            // row stride and lands them pixel-major [pixel][row][SB].  Pixel -1, pixels >= ncols and rows >= nrows
            // are out of bounds: zero fill.
            const int nbox = P.nbox[1], bw = P.bw[1];
            const bool mine = lane < nbox;
            const unsigned dst0 = mq_smem_u32(tile0) + (unsigned)(lane * bw) * (unsigned)(TR * SB * 4);
            const int cpix = lane * bw - 1;
            int bi = 0; unsigned ph = 0;
            for (int st = 0; st < nst; ++st) {
                if (st >= NBUF) mq_mbar_wait(&empty[bi], ph ^ 1u);      // previous use of this buffer released
                if (lane == 0) mq_mbar_expect_tx(&full[bi], strip_bytes);
                __syncwarp();
                if (mine) mq_tensor_g2s(dst0 + (unsigned)bi * strip_bytes, &tm1, (r_begin + st * TR) * SB, cpix, grp, &full[bi]);
                if (++bi == NBUF) { bi = 0; ph ^= 1u; }
            }
        } else if (lane == 0) {
            int bi = 0; unsigned ph = 0;
            for (int st = 0; st < nst; ++st) {
                if (st >= NBUF) mq_mbar_wait(&empty[bi], ph ^ 1u);      // previous use of this buffer released
                mq_mbar_expect_tx(&full[bi], strip_bytes);
                mq_bulk_g2s(tile0 + (size_t)bi * strip_bytes, src + (size_t)st * TR * pitch * SB, strip_bytes, &full[bi]);
                if (++bi == NBUF) { bi = 0; ph ^= 1u; }
            }
        }
    } else {
        // ------------------------------ marching warps -----------------------------
        if (P.acc_mode) {
            // beta of this group's samples from the per-block partial sums (fixed order: deterministic); the
            // loads overlap the flight of the first strip
            for (int s = warp; s < SB; s += NW) {
                const int b = b0 + s;
                float rn = 0.f, ro = 0.f;
                if (b < P.batch) {
                    for (int i = lane; i < P.rr_new_n; i += 32) rn += P.rr_new_part[(size_t)b * P.part_stride + i];
                    for (int i = lane; i < P.rr_old_n; i += 32) ro += P.rr_old_part[(size_t)b * P.part_stride + i];
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    rn += __shfl_xor_sync(0xffffffffu, rn, off);
                    ro += __shfl_xor_sync(0xffffffffu, ro, off);
                }
                if (lane == 0) {
                    const float be = b < P.batch ? __fdiv_rn(rn, ro) : 0.f;
                    betas[s] = be;
                    if (unit == 0 && rank == 0 && b < P.batch && P.beta_out) P.beta_out[b] = be;
                }
            }
        }
        if (P.tma && (cls == 1 || P.cls0_pm))
            mq_march_rows<V, LPR, NSLOT, TR, NW, true>(acc, eidx, livemask, NCH, warp, lane, nst, NBUF, r_begin, ncols,
                                                       row_bytes, strip_bytes, tile0, rays, full, empty, P.dbg, 0u);
        else
            // row-major strips of the bulk-row source start `lead` pixels into the row (pixel p sits at index p + lead)
            mq_march_rows<V, LPR, NSLOT, TR, NW, false>(acc, eidx, livemask, NCH, warp, lane, nst, NBUF, r_begin, ncols,
                                                        row_bytes, strip_bytes, tile0, rays, full, empty, P.dbg,
                                                        (P.tma && cls == 0) ? (unsigned)((P.lead - 1) * SB * 4) : 0u);
    }
    __syncthreads();                              // all strips consumed: the ring can be reused
    scd_stamp(P.dbg, 4);                          // march done

    // ---- partial line integrals -> red[e][SB] (the V samples of a lane: one vector store) ----
    if (warp < NW) {
#pragma unroll
        for (int k = 0; k < NSLOT; ++k) {
            if ((livemask >> k) & 1u) {
                VT pv;
                float *pf = reinterpret_cast<float *>(&pv);
#pragma unroll
                for (int v = 0; v < V; ++v) pf[v] = acc[k][v];
                *reinterpret_cast<VT *>(red + (size_t)eidx[k] * SB + lq * V) = pv;
            }
        }
    }
    if (CS > 1) cluster.sync(); else __syncthreads();
    scd_stamp(P.dbg, 5);                          // partials exchanged

    // ---- add the row-split partials in rank order, scale, write ------------------------------
    const int per = (E + CS - 1) / CS;
    const int e_lo = rank * per, e_hi = min(E, e_lo + per);
    const int cnt = max(e_hi - e_lo, 0);
    const size_t sino_sz = (size_t)P.n_angles * n_det;
    if (P.sino_il) {
        // interleaved rows for the backprojector (samples fastest, zero bins either side): one
        // vector of V samples per thread and rank
        float *dst = P.sino_il + (size_t)grp * ((size_t)P.n_angles * P.il_nb * SB);
        for (int idx = tid; idx < cnt * LPR; idx += NTHR) {
            const int el = idx / LPR, q = idx - el * LPR, e = e_lo + el;
            float sum[V];
#pragma unroll
            for (int v = 0; v < V; ++v) sum[v] = 0.f;
            for (int r = 0; r < CS; ++r) {
                const float *src = (CS > 1 ? cluster.map_shared_rank(red, r) : red) + (size_t)e * SB + q * V;
                const VT pv = *reinterpret_cast<const VT *>(src);
                const float *pf = reinterpret_cast<const float *>(&pv);
#pragma unroll
                for (int v = 0; v < V; ++v) sum[v] += pf[v];
            }
            const int ai = e / n_det, j = e - ai * n_det;
            // the view weight of A* rides on the output scale: linear, so the recurrence below stays exact
            const float sc = P.angw ? ang[ai].scale * __ldg(P.angw + pos0 + ai) : ang[ai].scale;
            VT ov;
            float *of = reinterpret_cast<float *>(&ov);
#pragma unroll
            for (int v = 0; v < V; ++v) of[v] = sum[v] * sc;
            const size_t qi = ((size_t)ang[ai].id * P.il_nb + P.il_padl + j) * SB + q * V;
            VT *qp = reinterpret_cast<VT *>(dst + qi);
            if (P.w_il) {                           // W A: per sample and bin, same place, same reason
                const VT wv = __ldg(reinterpret_cast<const VT *>(P.w_il + (size_t)grp * ((size_t)P.n_angles * P.il_nb * SB) + qi));
                const float *wf = reinterpret_cast<const float *>(&wv);
#pragma unroll
                for (int v = 0; v < V; ++v) of[v] *= wf[v];
            }
            if (P.acc_mode) {                       // q = A r + beta * q_old
                const VT old = *qp;
                const float *pf = reinterpret_cast<const float *>(&old);
#pragma unroll
                for (int v = 0; v < V; ++v) of[v] = fmaf(betas[q * V + v], pf[v], of[v]);
            }
            *qp = ov;
        }
        const int npad = P.il_nb - n_det;
        for (int ai = rank; ai < na; ai += CS) {
            float *row = dst + (size_t)ang[ai].id * P.il_nb * SB;
            for (int idx = tid; idx < npad * SB; idx += NTHR) {
                const int jp = idx / SB, s = idx - jp * SB;
                const int j = jp < P.il_padl ? jp : n_det + jp;
                row[(size_t)j * SB + s] = 0.f;
            }
        }
    }
    if (P.sino) {
        // user layout [sample][angle][bin]: 8 consecutive lanes take 8 consecutive bins of one sample
        // (one full 32-byte sector per store), the next 8 lanes the next sample (shared-memory reads
        // of red[e][s] then conflict at most SB/4-fold)
        const int nblk = (cnt + 7) >> 3;
        for (int idx = tid; idx < nblk * 8 * SB; idx += NTHR) {
            const int blk = idx / (8 * SB), rem = idx - blk * (8 * SB);
            const int s = rem >> 3, e = e_lo + blk * 8 + (rem & 7);
            if (e >= e_hi) continue;
            float v = 0.f;
            for (int r = 0; r < CS; ++r) v += (CS > 1 ? cluster.map_shared_rank(red, r) : red)[(size_t)e * SB + s];
            if (b0 + s < P.batch) {
                const int ai = e / n_det, j = e - ai * n_det;
                P.sino[(size_t)(b0 + s) * sino_sz + (size_t)ang[ai].id * n_det + j] = v * ang[ai].scale;
            }
        }
    }
    scd_stamp(P.dbg, 6);                          // output written
    if (CS > 1) cluster.sync();                   // keep red alive until every rank has read it
#ifdef SCD_DEBUG_STAMPS
    if (P.dbg && threadIdx.x == 0)                // slot 7: class and angle count of the unit (tools/timeline.py --by-class)
        P.dbg[(size_t)blockIdx.x * 8 + 7] = (unsigned long long)(cls * 1000 + na);
#endif
}

// ------------------------------------------------------------- host side ---
struct MqConfig {
    int V, LPR, SB, NSLOT, TR, NWT, NA, CS, nbuf, rows_per_cta, groups;
    MqLayout L;
    size_t smem, scratch_bytes, ring_bytes;
    int tma, spitch[2], nbox[2], bw[2];      // tensor-copy source: shared-memory strip rows of nbox boxes x bw pixels
};

// Strip-row geometry of the tensor-copy path: ncols + 3 pixels (1 zero pixel left, 2 right) split into boxes of at
// most 256 pixels (the box limit of a tensor map) whose byte size is a multiple of 128 (alignment of the copy's
// shared-memory destination)
static int mq_lead(int SB) { return SB >= 4 ? 1 : 4 / SB; }      // bulk rows start 16-byte aligned behind the pad pixels

static void mq_tma_rows(const scd_geom *g, int SB, int spitch[2], int nbox[2], int bw[2])
{
    const int nc[2] = {g->n1, g->n0};
    const int gran = std::max(1, 32 / SB);
    for (int c = 0; c < 2; ++c) {
        const int need = nc[c] + 2 + (c == 0 ? mq_lead(SB) : 1);
        nbox[c] = (need + 255) / 256;
        int w = (need + nbox[c] - 1) / nbox[c];
        w = ((w + gran - 1) / gran) * gran;
        if (w > 256) { nbox[c] += 1; w = (need + nbox[c] - 1) / nbox[c]; w = ((w + gran - 1) / gran) * gran; }
        bw[c] = w;
        spitch[c] = nbox[c] * w;
    }
}

static MqLayout mq_layout(const scd_geom *g, int SB)
{
    MqLayout L;
    L.SB = SB;
    const int nr[2] = {g->n0, g->n1}, nc[2] = {g->n1, g->n0};
    size_t off = 0;
    for (int c = 0; c < 2; ++c) {
        L.pitch[c] = nc[c] + 3;
        L.rows[c] = (nr[c] + 7) & ~7;
        L.cls_off[c] = off;
        off += (size_t)L.rows[c] * L.pitch[c] * SB;
        off = (off + 31) & ~(size_t)31;            // keep every class 128-byte aligned
    }
    L.group_floats = off;
    return L;
}

static size_t mq_fixed_smem(const scd_geom *g, int NA)
{
    return 2 * MQ_MAX_NBUF * 8 + sizeof(MqAng) * NA + 8 * (size_t)NA * g->n_det + 64;
}

static bool mq_have_tr(int V, int LPR, int TR)
{
    if (LPR == 1) return TR == 8 || (V == 4 && TR == 4);
    if (LPR == 2) return TR == 8 || TR == 4;
    return TR == 4 || TR == 2;                     // LPR == 4
}

// slot counts instantiated per CTA shape: 16 warps (15 marching, 128 registers) / 32 warps (31 marching, 64 registers)
static int mq_nslot(int nwt, int need)
{
    if (nwt == 16) return need <= 6 ? 6 : (need <= 13 ? 13 : 0);
    if (nwt == 24) return need <= 4 ? 4 : (need <= 8 ? 8 : 0);          // 80 registers per thread
    return need <= 3 ? 3 : (need <= 6 ? 6 : 0);
}

// Samples interleaved per pixel (packed image) and per detector bin (interleaved sinogram): one
// lane carries up to 4 samples, up to 4 lanes share a ray / pixel.
int scd_group_samples(const scd_geom *g, int batch)
{
    int sb = batch <= 1 ? 1 : (batch == 2 ? 2 : (batch <= 4 ? 4 : (batch <= 8 ? 8 : 16)));
    const int t = g->tune_fp_samples;
    if (t == 1 || t == 2 || t == 4 || t == 8 || t == 16) sb = t;
    // two strips of the thinnest kind must fit next to the tables, else fewer samples per group
    const int maxpitch = std::max(g->n0, g->n1) + 3;
    while (sb > 1) {
        const int trmin = sb >= 16 ? 2 : (sb >= 4 ? 4 : 8);
        if (2 * (size_t)trmin * maxpitch * sb * 4 + mq_fixed_smem(g, 1) <= (size_t)g->smem_optin) break;
        sb >>= 1;
    }
    return sb;
}

static MqConfig mq_choose(const scd_geom *g, int batch, int n_cls_max, bool tma = false)
{
    MqConfig c;
    c.SB = scd_group_samples(g, batch);
    c.V = c.SB >= 4 ? 4 : c.SB;
    c.LPR = c.SB / c.V;
    c.tma = tma ? 1 : 0;
    int maxpitch = std::max(g->n0, g->n1) + 3;
    if (tma) {
        mq_tma_rows(g, c.SB, c.spitch, c.nbox, c.bw);
        maxpitch = std::max(c.spitch[0], c.spitch[1]);
    } else {
        for (int k = 0; k < 2; ++k) c.spitch[k] = c.nbox[k] = c.bw[k] = 0;
    }
    const size_t budget = (size_t)g->smem_optin;
    c.SB = c.V * c.LPR;
    c.groups = (batch + c.SB - 1) / c.SB;
    const int RPW = 32 / c.LPR;
    const int nchunk = (g->n_det + RPW - 1) / RPW;

    // warps per CTA: 15, 23 or 31 marching warps + the producer.  The chunks of a CTA are dealt
    // round-robin to the marching warps, so the count that divides them most evenly wins (365 bins
    // = 46 chunks of 8 rays = 2 x 23; 711 bins = 89 chunks ~ 4 x 23): 23 unless told otherwise
    c.NWT = 16;
    if (c.V == 4 && c.LPR >= 2) {
        // few CTAs (at most one per SM even with the row split): latency-bound, more warps help
        // (B = 32: 72 -> 67 us); many CTAs: the 15-warp shape with more registers wins (B = 256)
        const int units4 = c.groups * ((n_cls_max + 3) / 4) * 2;
        if (units4 * 4 <= 2 * g->sm_count) c.NWT = 24;
        // many CTAs per SM in sequence (several waves): more warps per CTA hide the tap latency better as long as
        // four angles per CTA still fit the smaller register budget (measured on the tensor-copy path, 256^2:
        // B = 128: 198.7 -> 192.0 us with 24 warps, B = 256: 359.9 -> 340.9 us with 32; neutral or worse below)
        else if (c.LPR == 4 && units4 * 2 >= 3 * g->sm_count && 4 * nchunk <= 6 * 31) c.NWT = 32;
        else if (c.LPR == 4 && units4 * 4 >= 3 * g->sm_count && 4 * nchunk <= 8 * 23) c.NWT = 24;
        // wide detectors (501^2: 711 bins = 89 chunks): four angles per CTA fit no shape, two fit 24 warps as well
        // as 16 (501^2 x 128 slices x 150 angles: 2058 -> 1891 us)
        else if (c.LPR == 4 && units4 * 4 >= 3 * g->sm_count && 4 * nchunk > 13 * 15 && 2 * nchunk <= 8 * 23) c.NWT = 24;
    }
    if (g->tune_fp_threads == 1024 && c.V == 4 && c.LPR >= 2) c.NWT = 32;
    else if (g->tune_fp_threads == 768 && c.V == 4) c.NWT = 24;
    else if (g->tune_fp_threads == 512) c.NWT = 16;
    const int NW = c.NWT - 1;
    // angles per CTA and cluster row split.  Sharing a strip between NA angles divides the
    // L2 -> SM traffic by NA, but the machine wants >= ~3/4 * SMs CTAs: take the largest NA for
    // which a row split of at most 4 provides them (measured: tools/kbench.py --kernel fp --sweep)
    const int maxrows8 = (std::max(g->n0, g->n1) + 7) & ~7;
    int na = 4, cs = 1;
    for (na = 4; na >= 1; na >>= 1) {
        if (na > 1 && !mq_nslot(c.NWT, (na * nchunk + NW - 1) / NW)) continue;
        const int units = c.groups * ((n_cls_max + na - 1) / na) * 2;
        bool ok = false;
        for (cs = 1; cs <= 4; cs <<= 1)
            if (units * cs * 4 >= g->sm_count * 3 || maxrows8 / (cs * 2) < 16) { ok = units * cs * 4 >= g->sm_count * 3; break; }
        if (cs > 4) cs = 4;
        if (ok || na == 1) break;
    }
    na = std::max(na, 1);
    if (g->tune_fp_angles) { na = g->tune_fp_angles; }
    na = std::max(1, std::min(na, std::max(1, n_cls_max)));
    while (na > 1 && !mq_nslot(c.NWT, (na * nchunk + NW - 1) / NW)) --na;
    c.NA = na;
    c.NSLOT = mq_nslot(c.NWT, (c.NA * nchunk + NW - 1) / NW);

    // rows per strip / ring depth from the shared-memory budget
    const int trs[3] = {8, 4, 2};
    c.TR = 0;
    for (int i = 0; i < 3; ++i) {
        const int tr = trs[i];
        if (g->tune_fp_rows && tr != g->tune_fp_rows) continue;
        if (!mq_have_tr(c.V, c.LPR, tr)) continue;
        if (3 * (size_t)tr * maxpitch * c.SB * 4 + mq_fixed_smem(g, c.NA) <= budget || tr == 2 ||
            (tr == 4 && !mq_have_tr(c.V, c.LPR, 2))) { c.TR = tr; break; }
    }
    if (!c.TR) c.TR = mq_have_tr(c.V, c.LPR, 2) ? 2 : (mq_have_tr(c.V, c.LPR, 4) ? 4 : 8);
    c.L = mq_layout(g, c.SB);
    const size_t strip = (size_t)c.TR * maxpitch * c.SB * 4;

    const int maxrows = std::max(c.L.rows[0], c.L.rows[1]);
    if (g->tune_fp_cluster) cs = g->tune_fp_cluster;
    if (cs != 1 && cs != 2 && cs != 4 && cs != 8) cs = 1;
    c.CS = cs;
    c.rows_per_cta = (((maxrows + cs - 1) / cs) + 7) & ~7;

    int nstrips = (c.rows_per_cta + c.TR - 1) / c.TR;
    int nbuf = g->tune_fp_nbuf ? g->tune_fp_nbuf : MQ_MAX_NBUF;
    nbuf = std::max(2, std::min(std::min(nbuf, MQ_MAX_NBUF), nstrips));
    while (nbuf > 1 && nbuf * strip + mq_fixed_smem(g, c.NA) > budget) --nbuf;
    c.nbuf = nbuf;
    // the partials red[NA*n_det][SB] alias the ring
    c.ring_bytes = (std::max(nbuf * strip, (size_t)c.SB * c.NA * g->n_det * 4) + 127) & ~(size_t)127;
    c.smem = c.ring_bytes + mq_fixed_smem(g, c.NA);
    c.scratch_bytes = (size_t)c.groups * c.L.group_floats * 4;
    return c;
}

// ---- unit plan: which angles share a CTA ------------------------------------------------------
// All CTAs cost about (angles + const), and there are only a few hundred of them for ~148 SMs, so
// equal chunks of NA angles can leave a third of the machine idle in the last round.  The plan
// splits each class into chunks of NA angles followed by shorter ones (launched last, largest
// first: list scheduling) and keeps the split with the smallest simulated makespan.
struct MqPlan { int n_runs; MqRun runs[MQ_MAX_RUNS]; int units, n_big; };

static double mq_makespan(const int *sizes, const int *counts, int nkinds, int jobs_per_unit, int machines, double fixed)
{
    // machines take jobs in launch order; all jobs of one kind cost the same
    std::vector<double> load((size_t)machines, 0.0);
    std::make_heap(load.begin(), load.end(), std::greater<double>());
    for (int k = 0; k < nkinds; ++k) {
        const double cost = sizes[k] + fixed;         // angles + fixed share (strip fetches, tables, output) in units of one angle
        for (long j = 0; j < (long)counts[k] * jobs_per_unit; ++j) {
            std::pop_heap(load.begin(), load.end(), std::greater<double>());
            load.back() += cost;
            std::push_heap(load.begin(), load.end(), std::greater<double>());
        }
    }
    return *std::max_element(load.begin(), load.end());
}

static MqPlan mq_plan(const scd_geom *g, const MqConfig &c, int angle_lo, int angle_hi)
{
    // positions in order[] of the selected angles, per class (contiguous: order[] is sorted by
    // class then index and the selection is an index range)
    int first[2] = {-1, -1}, cnt[2] = {0, 0};
    for (int pos = 0; pos < g->n_angles; ++pos) {
        const int a = g->h_order[pos];
        if (a < angle_lo || a >= angle_hi) continue;
        const int cls = g->h_fp[a].cls;
        if (first[cls] < 0) first[cls] = pos;
        cnt[cls]++;
    }
    const int machines = std::max(1, g->sm_count / c.CS);
    const int NA = c.NA;
    // candidate: per class, `t1` angles alone, `t2` angles in pairs, the rest in chunks of NA
    // (plus one remainder chunk); the same (t1, t2) for both classes, clipped to the class size
    int best_t1 = 0, best_t2 = 0;
    double best = -1.0;
    const double fixed = g->tune_fp_plan_cost > 0 ? g->tune_fp_plan_cost / 100.0 : 0.25;
    const int nmax = std::max(cnt[0], cnt[1]);
    const bool search = NA > 2 && g->tune_fp_plan != 1 && (long)c.groups * nmax * 2 <= 4096;
    for (int t1 = 0; t1 <= (search ? std::min(nmax, 2 * NA) : 0); ++t1)
        for (int t2 = 0; t2 + t1 <= (search ? std::min(nmax, 6 * NA) : 0); t2 += 2) {
            int sizes[8], counts[8], nk = 0;
            // launch order: big chunks of both classes, remainders, pairs, singles
            int rem[2], big[2], pairs[2], single[2];
            for (int cl = 0; cl < 2; ++cl) {
                single[cl] = std::min(t1, cnt[cl]);
                pairs[cl] = std::min(t2, cnt[cl] - single[cl]) / 2;
                const int rest = cnt[cl] - single[cl] - 2 * pairs[cl];
                big[cl] = rest / NA; rem[cl] = rest % NA;
            }
            sizes[nk] = NA; counts[nk++] = big[0] + big[1];
            for (int cl = 0; cl < 2; ++cl) if (rem[cl]) { sizes[nk] = rem[cl]; counts[nk++] = 1; }
            sizes[nk] = 2; counts[nk++] = pairs[0] + pairs[1];
            sizes[nk] = 1; counts[nk++] = single[0] + single[1];
            const double m = mq_makespan(sizes, counts, nk, c.groups, machines, fixed);
            if (best < 0 || m < best - 1e-9) { best = m; best_t1 = t1; best_t2 = t2; }
        }
    MqPlan pl;
    pl.n_runs = 0; pl.units = 0;
    int used[2] = {0, 0};
    auto add = [&](int cl, int count, int na) {
        if (count <= 0) return;
        MqRun &r = pl.runs[pl.n_runs++];
        r.cls = cl; r.first = first[cl] + used[cl]; r.count = count; r.na = na; r.unit0 = pl.units;
        pl.units += (count + na - 1) / na;
        used[cl] += count;
    };
    int single[2], pairs[2], rest[2];
    for (int cl = 0; cl < 2; ++cl) {
        single[cl] = std::min(best_t1, cnt[cl]);
        pairs[cl] = std::min(best_t2, cnt[cl] - single[cl]) / 2;
        rest[cl] = cnt[cl] - single[cl] - 2 * pairs[cl];
    }
    for (int cl = 0; cl < 2; ++cl) add(cl, rest[cl], NA);          // includes the remainder chunk (run-local min)
    pl.n_big = pl.units;
    for (int cl = 0; cl < 2; ++cl) add(cl, 2 * pairs[cl], 2);
    for (int cl = 0; cl < 2; ++cl) add(cl, single[cl], 1);
    return pl;
}

size_t scd_fp_scratch_need_v4(const scd_geom *g, int batch)
{
    if (!g || batch <= 0) return 0;
    size_t need = 0;
    for (int SB = 1; SB <= 16; SB <<= 1) {
        const MqLayout L = mq_layout(g, SB);
        need = std::max(need, (size_t)((batch + SB - 1) / SB) * L.group_floats * 4);
    }
    return need + 256;
}

template <int V, int LPR, int NSLOT, int TR, int NWT>
static int mq_launch_t(const MqParams &P, const CUtensorMap *tms, dim3 grid, size_t smem, cudaStream_t st, int device)
{
    static ScdSmemAttr attr = {};        // per instantiation
    SCD_CUDA(scd_ensure_smem(fp_march_kernel<V, LPR, NSLOT, TR, NWT>, attr, device, smem));
    SCD_CUDA(scd_launch_kernel(fp_march_kernel<V, LPR, NSLOT, TR, NWT>, grid, dim3(32 * NWT), smem, st, P.CS, P, tms[0], tms[1]));
    SCD_LAUNCH_CHECK("fp_march_kernel");
    return 0;
}

// ---- tensor maps of the sample-interleaved image ---------------------------------------------
typedef CUresult (*MqEncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                               const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static MqEncodeFn mq_encoder()
{
    static MqEncodeFn fn = []() -> MqEncodeFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess ||
            qr != cudaDriverEntryPointSuccess)
            return nullptr;
        return (MqEncodeFn)p;
    }();
    return fn;
}

// tms[1], class-1 strips: img_il[group][k0][k1][SB] as a 3-D tensor (n1*SB, n0, groups) -- an image row is one
// contiguous run of n1*SB floats -- with boxes of TR image columns x bw pixels: {TR*SB, bw, 1}.
// tms[0], class-0 strips fetched pixel-major (optional): the 4-D tensor (SB, n0, n1, groups), boxes {SB, TR, bw, 1}.
static int mq_make_maps(const scd_geom *g, const float *img_il, const MqConfig &c, CUtensorMap tms[2], bool cls0_pm)
{
    MqEncodeFn enc = mq_encoder();
    if (!enc) { scd_set_error("scd_fp: cuTensorMapEncodeTiled is not available in this driver"); return SCD_E_NODEVICE; }
    {
        const cuuint64_t dims[3] = {(cuuint64_t)g->n1 * c.SB, (cuuint64_t)g->n0, (cuuint64_t)c.groups};
        const cuuint64_t strides[2] = {(cuuint64_t)g->n1 * c.SB * 4, (cuuint64_t)g->n0 * g->n1 * c.SB * 4};
        const cuuint32_t estr[3] = {1, 1, 1};
        const cuuint32_t box[3] = {(cuuint32_t)(c.TR * c.SB), (cuuint32_t)c.bw[1], 1u};
        const CUresult r = enc(&tms[1], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void *)img_il, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { scd_set_error("scd_fp: cuTensorMapEncodeTiled failed (%d)", (int)r); return SCD_E_INVALID; }
    }
    if (cls0_pm) {
        const cuuint64_t dims[4] = {(cuuint64_t)c.SB, (cuuint64_t)g->n0, (cuuint64_t)g->n1, (cuuint64_t)c.groups};
        const cuuint64_t strides[3] = {(cuuint64_t)g->n1 * c.SB * 4, (cuuint64_t)c.SB * 4, (cuuint64_t)g->n0 * g->n1 * c.SB * 4};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const cuuint32_t box[4] = {(cuuint32_t)c.SB, (cuuint32_t)c.TR, (cuuint32_t)c.bw[0], 1u};
        const CUresult r = enc(&tms[0], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void *)img_il, dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { scd_set_error("scd_fp: cuTensorMapEncodeTiled (class 0) failed (%d)", (int)r); return SCD_E_INVALID; }
    }
    return 0;
}

// plan (cached) + launch of the march for one configuration; P carries sources / destinations
static int mq_march(const scd_geom *g, const MqConfig &c, MqParams &P, const CUtensorMap *tms, int angle_lo, int angle_hi,
                    cudaStream_t st)
{
    // the plan depends only on the geometry, the configuration and the angle range: keep the last one
    // (the search simulates a few hundred schedules, too slow to repeat at every launch)
    struct PlanKey { unsigned long long g; int lo, hi, groups, NA, CS, plan, sm, cost; };
    static thread_local PlanKey last_key = {0ull, 0, 0, 0, 0, 0, 0, 0, 0};
    static thread_local MqPlan last_plan;
    const PlanKey key = {g->id, angle_lo, angle_hi, c.groups, c.NA, c.CS, g->tune_fp_plan, g->sm_count, g->tune_fp_plan_cost};
    const bool same = key.g == last_key.g && key.lo == last_key.lo && key.hi == last_key.hi && key.groups == last_key.groups &&
                      key.NA == last_key.NA && key.CS == last_key.CS && key.plan == last_key.plan && key.sm == last_key.sm && key.cost == last_key.cost;
    if (!same) {
        last_plan = mq_plan(g, c, angle_lo, angle_hi);
        last_key = key;
    }
    const MqPlan &pl = last_plan;
    if (pl.units == 0) return 0;
    if ((long)pl.units * c.groups * c.CS > 0x7fffffffL) { scd_set_error("scd_fp: too many CTAs"); return SCD_E_INVALID; }
    P.groups = c.groups; P.n_big = pl.n_big; P.n_units = pl.units; P.dbg = scd_debug_stamps();
    P.n_runs = pl.n_runs;
    for (int i = 0; i < pl.n_runs; ++i) P.runs[i] = pl.runs[i];
    const unsigned gx = (unsigned)c.groups * c.CS;
    dim3 grid(gx * pl.units);      // linear: see the index decoding at the top of the kernel
    int rc = SCD_E_INVALID;
#define MQ_CASE(VV, LL, TT)                                                                         \
    if (c.V == VV && c.LPR == LL && c.TR == TT && c.NWT == 16)                                      \
        rc = c.NSLOT == 6 ? mq_launch_t<VV, LL, 6, TT, 16>(P, tms, grid, c.smem, st, g->device)                     \
                          : mq_launch_t<VV, LL, 13, TT, 16>(P, tms, grid, c.smem, st, g->device);
#define MQ_CASE24(VV, LL, TT)                                                                       \
    if (c.V == VV && c.LPR == LL && c.TR == TT && c.NWT == 24)                                      \
        rc = c.NSLOT == 4 ? mq_launch_t<VV, LL, 4, TT, 24>(P, tms, grid, c.smem, st, g->device)                     \
                          : mq_launch_t<VV, LL, 8, TT, 24>(P, tms, grid, c.smem, st, g->device);
#define MQ_CASE32(VV, LL, TT)                                                                       \
    if (c.V == VV && c.LPR == LL && c.TR == TT && c.NWT == 32)                                      \
        rc = c.NSLOT == 3 ? mq_launch_t<VV, LL, 3, TT, 32>(P, tms, grid, c.smem, st, g->device)                     \
                          : mq_launch_t<VV, LL, 6, TT, 32>(P, tms, grid, c.smem, st, g->device);
    MQ_CASE(1, 1, 8) MQ_CASE(2, 1, 8) MQ_CASE(4, 1, 8) MQ_CASE(4, 1, 4)
    MQ_CASE(4, 2, 8) MQ_CASE(4, 2, 4) MQ_CASE(4, 4, 4) MQ_CASE(4, 4, 2)
    MQ_CASE24(4, 1, 8) MQ_CASE24(4, 1, 4) MQ_CASE24(4, 2, 8) MQ_CASE24(4, 2, 4) MQ_CASE24(4, 4, 4) MQ_CASE24(4, 4, 2)
    MQ_CASE32(4, 2, 8) MQ_CASE32(4, 2, 4) MQ_CASE32(4, 4, 4) MQ_CASE32(4, 4, 2)
#undef MQ_CASE24
#undef MQ_CASE
#undef MQ_CASE32
    if (rc == SCD_E_INVALID) scd_set_error("scd_fp: no kernel for V=%d LPR=%d TR=%d warps=%d", c.V, c.LPR, c.TR, c.NWT);
    return rc;
}

static void mq_fill_params(const scd_geom *g, const MqConfig &c, MqParams &P, float *sino, float *sino_il, int batch,
                           const int ncls[2])
{
    memset(&P, 0, sizeof(P));
    P.sino = sino; P.sino_il = sino_il; P.il_padl = g->il_padl; P.il_nb = g->il_nb;
    P.fp = g->d_fp; P.rayt = g->d_rayt; P.angt = g->d_angt; P.angw = g->d_angw; P.order = g->d_order;
    P.n0 = g->n0; P.n1 = g->n1; P.n_angles = g->n_angles; P.n_det = g->n_det; P.batch = batch;
    P.NA = c.NA; P.nbuf = c.nbuf; P.CS = c.CS; P.rows_per_cta = c.rows_per_cta; P.ring_bytes = (int)c.ring_bytes; P.L = c.L;
    P.need_cls[0] = ncls[0] > 0; P.need_cls[1] = ncls[1] > 0;
    P.tma = c.tma;
    for (int k = 0; k < 2; ++k) { P.spitch[k] = c.spitch[k]; P.nbox[k] = c.nbox[k]; P.bw[k] = c.bw[k]; }
}

// Packed-copy path (groups of 1 or 2 samples, whose 4/8-byte pixels are below the 16-byte granule of a tensor copy):
// pack pass (producer fused in) + march over 1-D bulk copies
int scd_launch_fp_v4(const scd_geom *g, const float *img, float *sino, float *sino_il, int batch,
                     int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes, cudaStream_t st,
                     const FpPrologue *prologue, const float *w_il)
{
    FpPrologue Q;
    if (prologue) Q = *prologue; else { memset(&Q, 0, sizeof(Q)); }
    // angles of each class inside the range
    int ncls[2] = {0, 0};
    for (int a = angle_lo; a < angle_hi; ++a) ncls[g->h_fp[a].cls]++;
    MqConfig c = mq_choose(g, batch, std::max(ncls[0], ncls[1]));
    if (c.smem > (size_t)g->smem_optin || !c.NSLOT) { scd_set_error("scd_fp: image too large for the shared-memory strip"); return SCD_E_INVALID; }
    const uintptr_t sp = ((uintptr_t)scratch + 127) & ~(uintptr_t)127;
    if (!scratch || sp + c.scratch_bytes > (uintptr_t)scratch + scratch_bytes) {
        scd_set_error("scd_fp: scratch too small (%zu bytes given, %zu needed; see scd_fp_scratch_bytes)",
                      scratch_bytes, c.scratch_bytes + 128);
        return SCD_E_WORKSPACE;
    }
    MqParams P;
    mq_fill_params(g, c, P, sino, sino_il, batch, ncls);
    P.img = img; P.packed = (float *)sp; P.w_il = w_il;

    // ---- pack: image -> tile-ready layout (both orientations), producer fused in ----
    {
        if (c.groups > 65535) { scd_set_error("scd_fp: batch too large"); return SCD_E_INVALID; }
        dim3 pg((std::max(g->n1, c.L.rows[1]) + PK_T - 1) / PK_T, (std::max(g->n0, c.L.rows[0]) + PK_T - 1) / PK_T, c.groups);
#define PK_CASE(SS)                                                                                  \
        if (c.SB == SS) {                                                                               \
            if (Q.mode == 0) SCD_CUDA(scd_launch_kernel(fp_packq_kernel<0, SS>, pg, dim3(256), 0, st, 0, P, Q));       \
            else if (Q.mode == 1) SCD_CUDA(scd_launch_kernel(fp_packq_kernel<1, SS>, pg, dim3(256), 0, st, 0, P, Q));  \
            else SCD_CUDA(scd_launch_kernel(fp_packq_kernel<2, SS>, pg, dim3(256), 0, st, 0, P, Q));                   \
        }
        PK_CASE(1) PK_CASE(2) PK_CASE(4) PK_CASE(8) PK_CASE(16)
#undef PK_CASE
        SCD_LAUNCH_CHECK("fp_packq_kernel");
    }
    CUtensorMap tms[2];
    memset(tms, 0, sizeof(tms));
    return mq_march(g, c, P, tms, angle_lo, angle_hi, st);
}

// Tensor-copy path: project a sample-interleaved image img_il[group][k0][k1][SB] (SB = scd_group_samples >= 4) --
// one launch, no packed copy.  acc != nullptr: q = A img + beta * q_old (see MqParams).
int scd_launch_fp_ilimg(const scd_geom *g, const float *img_il, float *sino, float *sino_il, int batch,
                        int angle_lo, int angle_hi, cudaStream_t st, const FpAccumulate *acc, const float *w_il)
{
    if (g && batch == 0) return 0;
    if (!g || !img_il || (!sino && !sino_il)) { scd_set_error("scd_fp: null argument"); return SCD_E_INVALID; }
    if (batch < 0 || angle_lo < 0 || angle_hi > g->n_angles || angle_lo > angle_hi) {
        scd_set_error("scd_fp: bad batch/angle range (batch=%d, angles [%d,%d) of %d)", batch, angle_lo, angle_hi, g->n_angles);
        return SCD_E_INVALID;
    }
    if (angle_lo == angle_hi) return 0;
    if (!scd_il_image_ok(g, batch)) { scd_set_error("scd_fp: no tensor-copy path for this batch / image size"); return SCD_E_INVALID; }
    if (((uintptr_t)img_il & 15) != 0) { scd_set_error("scd_fp: interleaved image must be 16-byte aligned"); return SCD_E_INVALID; }
    int ncls[2] = {0, 0};
    for (int a = angle_lo; a < angle_hi; ++a) ncls[g->h_fp[a].cls]++;
    MqConfig c = mq_choose(g, batch, std::max(ncls[0], ncls[1]), true);
    if (c.smem > (size_t)g->smem_optin || !c.NSLOT) { scd_set_error("scd_fp: image too large for the shared-memory strip"); return SCD_E_INVALID; }
    MqParams P;
    mq_fill_params(g, c, P, sino, sino_il, batch, ncls);
    P.img = img_il; P.zero_row = g->d_zero_row; P.lead = mq_lead(c.SB); P.w_il = w_il;
    if (acc) {
        P.acc_mode = 1;
        P.rr_new_part = acc->rr_new_part; P.rr_new_n = acc->rr_new_n;
        P.rr_old_part = acc->rr_old_part; P.rr_old_n = acc->rr_old_n; P.part_stride = acc->part_stride;
        P.beta_out = acc->beta_out;
    }
    // class 0 pixel-major as well: pays where the row-major layout conflicts most -- 8 samples per pixel (a
    // quarter-warp holds four rays: 30 % of its wavefronts were conflicts).  Measured at 256^2: B = 8 26.8 -> 24.8 us;
    // neutral at B = 16 .. 32, -1 % at B = 256, +4 % on the 501^2 shard (16 samples per pixel: 4.5 % conflicts
    // only, and SB*4-byte pieces instead of whole rows), +4 % at B = 4.  fp_cls0: 1 = always, 2 = never.
    P.cls0_pm = (g->tune_fp_cls0 == 1 || (g->tune_fp_cls0 == 0 && c.LPR == 2)) && c.nbox[0] <= 32;
    CUtensorMap tms[2];
    memset(tms, 0, sizeof(tms));
    int rc = mq_make_maps(g, img_il, c, tms, P.cls0_pm != 0);
    if (rc) return rc;
    return mq_march(g, c, P, tms, angle_lo, angle_hi, st);
}

// Whether batches of this size run on the tensor-copy path: groups of >= 4 samples (a pixel of the interleaved
// image is then >= 16 bytes, the granule of a tensor copy) whose strip rows need at most 32 copies per strip
// (one per lane of the producer warp)
bool scd_il_image_ok(const scd_geom *g, int batch)
{
    if (!g || batch <= 0) return false;
    if (g->tune_fp_source == 1) return false;          // tuning: force the packed-copy path
    const int SB = scd_group_samples(g, batch);
    if (!mq_encoder()) return false;
    // a single sample per group: the interleaved image IS the reference layout; rows and the TR-row pieces of the
    // class-1 gather are multiples of 16 bytes when n1 is a multiple of 4.  Pairs (SB = 2) have no interleaving
    // kernels: they keep the packed copy.
    if (SB == 2 || (SB == 1 && ((g->n1 & 3) || g->tune_fp_source == 2))) return false;
    int sp[2], nb[2], bw[2];
    mq_tma_rows(g, SB, sp, nb, bw);
    return nb[1] <= 32;                                 // one lane of the producer warp per class-1 box
}

size_t scd_il_image_bytes(const scd_geom *g, int batch)
{
    if (!g || batch <= 0) return 0;
    // the group size may be overridden by tuning: size for the worst case (a multiple of 16 samples)
    return (size_t)((batch + 15) / 16) * 16 * g->n0 * g->n1 * 4;
}

// ------------------------------------------------------------- entry point ---
int scd_launch_fp(const scd_geom *g, const float *img, float *sino, float *sino_il, int batch,
                  int angle_lo, int angle_hi, void *scratch, size_t scratch_bytes, cudaStream_t st,
                  const FpPrologue *prologue, const float *w_il)
{
    if (g && batch == 0) return 0;                 // empty batch: nothing to do (pointers may be null)
    if (!g || (!img && !(prologue && prologue->mode != 0)) || (!sino && !sino_il)) { scd_set_error("scd_fp: null argument"); return SCD_E_INVALID; }
    if (batch < 0 || angle_lo < 0 || angle_hi > g->n_angles || angle_lo > angle_hi) {
        scd_set_error("scd_fp: bad batch/angle range (batch=%d, angles [%d,%d) of %d)",
                      batch, angle_lo, angle_hi, g->n_angles);
        return SCD_E_INVALID;
    }
    if (batch == 0 || angle_lo == angle_hi) return 0;
    if (!(prologue && prologue->mode != 0) && scd_il_image_ok(g, batch)) {
        // user-layout images: one interleaving pass (1 x the image, instead of the 2.06 x packed copy), then the
        // tensor-copy march
        const uintptr_t sp = ((uintptr_t)scratch + 127) & ~(uintptr_t)127;
        const int SB = scd_group_samples(g, batch);
        const size_t need = (size_t)((batch + SB - 1) / SB) * SB * g->n0 * g->n1 * 4;
        if (!scratch || sp + need > (uintptr_t)scratch + scratch_bytes) {
            scd_set_error("scd_fp: scratch too small (%zu bytes given, %zu needed; see scd_fp_scratch_bytes)", scratch_bytes, need + 128);
            return SCD_E_WORKSPACE;
        }
        if (SB == 1 && ((uintptr_t)img & 15) == 0)      // one sample per group: the image already is its interleaved form
            return scd_launch_fp_ilimg(g, img, sino, sino_il, batch, angle_lo, angle_hi, st, nullptr, w_il);
        int rc = scd_launch_il_pack(g, img, (float *)sp, nullptr, nullptr, batch, st);
        if (rc) return rc;
        return scd_launch_fp_ilimg(g, (const float *)sp, sino, sino_il, batch, angle_lo, angle_hi, st, nullptr, w_il);
    }
    return scd_launch_fp_v4(g, img, sino, sino_il, batch, angle_lo, angle_hi, scratch, scratch_bytes, st, prologue, w_il);
}

size_t scd_fp_scratch_need(const scd_geom *g, int batch)
{
    return std::max(scd_fp_scratch_need_v4(g, batch), scd_il_image_bytes(g, batch) + 256);
}
