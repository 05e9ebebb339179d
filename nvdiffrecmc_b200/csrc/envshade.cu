// envshade.cu -- fused environment-light MIS sampling + shadow rays + PBR BSDF, forward and backward.
//
// Replaces the OptiX raygen program __raygen__rg / process_sample / shadow_test
// (render/optixutils/c_src/envsampling/kernel.cu:101-118, 403-542) and its launchers env_shade_fwd /
// env_shade_bwd (render/optixutils/c_src/torch_bindings.cpp:123-272).
//
// B200 mapping (no RT cores, 148 SMs):
//   * FOUR 8-WARP CTAs PER SM, ONE WARP PER PIXEL, ONE LANE PER SAMPLE, THREE CTA-SYNCHRONOUS PHASES PER BATCH OF 8 PIXELS
//     (history in profiles/: v1 traced inline at 10/32 active lanes; v2 per-warp queues, 13/32 lanes in the while-while loop;
//      v3 deferred leaf tests, 25/32 lanes but 22 % instruction-fetch stalls with 32 independent warps spread over all
//      phases; v4 one 32-warp CTA per SM in lock-step phases: no fetch stalls, L1 hit 88 %; final: 4 CTAs x 8 warps, so that
//      one CTA's ALU-heavy generate phase overlaps another's latency-heavy trace phase, +9 %):
//       G  generate, in two stages (round 2): every warp draws the directions of the 2N^2 samples of its pixel (exact path, all
//          lanes); rays that can contribute (n.wi > 0) are ballot-compacted into the warp's segment of a block-wide shared-memory
//          queue; the rest of the set-up (lat-long texel, light and BSDF pdf -> MIS weight) runs on the compacted entries only;
//       T  trace: all warps drain the queue together -- own segment first, then work stealing -- with one 4-wide quantised
//          BVH node step per lane per iteration (v6), leaf tests deferred to full-warp batches, dynamic ray fetch (a ray is picked up
//          with three MUFU.RCP: the culling constants are not part of the parity contract), and, once the queue is empty, idle lanes
//          take over pending subtrees of the walks still in flight (round 2); one bit per ray;
//       E  evaluate: each warp compacts the surviving rays (V != 0) of its pixel and only those evaluate the BSDF (forward)
//          or its adjoint + the env-map gradient scatter (backward); warp-shuffle reduction, one writer per pixel.
//     The reference runs one thread per pixel and loops 2*N^2 samples serially with an optixTrace per sample.
//   * The reference's per-pixel PCG stream is sequential (5 uniforms per stratum); lanes jump to their
//     position with a precomputed LCG skip table (state' = state*mul[k] + add[k]), so the random
//     numbers are bit-identical to the reference stream (kernel.cu:30-45, 504-524).
//   * Persistent warps: grid = #SMs x resident CTAs, each warp claims 32-pixel chunks from a global
//     counter (coverage is ~35 %: masked chunks cost one coalesced load + ballot).
//   * Rays whose unshadowed contribution is exactly zero (n.wi <= 0: Lambert and the GGX lobe both
//     vanish, and so do all their adjoints) are not traced; this is output-preserving and removes
//     about half of the light-sampled rays.
//   * Sampling decisions use exact.cuh arithmetic (bit-identical texel / direction / lobe choice vs
//     the oracle); BSDF evaluation, pdfs and adjoints use fast FMA math (bsdf.cuh).
//   * Backward: when forward and backward share the seed (the reference's training loop always does) the forward records the
//     rays it evaluated (direction, MIS weight, texel, occluded flag) and env_shade_replay_kernel walks that record: adjoint BSDF +
//     gradient scatter only, no sampling, no traversal.  Otherwise env_shade_kernel<1> replays the random stream and re-traces
//     like the reference.  Either way the per-pixel gradients are reduced in registers / shuffles (single writer per pixel like the
//     reference's `+=`, kernel.cu:442-456) and the env-map gradient is scattered with float atomics (kernel.cu:203-211),
//     skipping zero contributions.
#include "bsdf.cuh"
#include "bvh_traverse.cuh"
#include "ctx.h"
#include "exact.cuh"
#include <vector>

namespace {

constexpr float MIN_ROUGHNESS = 0.08f;     // kernel.cu:17

struct EnvParams {
    TView mask, ro, pos, nrm, view, kd, ks;
    const float *light; int l_s1, l_s2, l_s3;      // [Hl,Wl,3] strides
    const float *pdf; int p_s1, p_s2;
    const float *rows; int r_s;
    const float *cols; int c_s1, c_s2;
    const int32_t *perms; int pm_s1, pm_s3; uint32_t n_perms;
    int Hl, Wl, m_rows, m_cols;
    int B, H, W;
    int N, S;
    uint32_t bsdf, seed;
    const uint32_t *seed_dev;       // optional: added to `seed` at kernel start (CUDA-graph friendly seed advance)
    int batch_offset;
    float shadow_scale;
    BvhView bvh;
    const uint2 *skip;
    unsigned int *chunk_counter;
    // fwd
    float *diff, *spec;
    int32_t *rec_texel; uint8_t *rec_vis;
    uint32_t *hit_out;              // optional: per-pixel visibility record written by the forward pass
    const uint32_t *hit_in;         // optional: record replayed by the backward pass instead of tracing
    int hit_words;                  // uint32 words per pixel = ceil(2 N^2 / 32)
    uint32_t *rec_count;            // optional ray record written by the forward pass: evaluated rays per pixel ...
    float *rec_rays;                // ... and their (dx, dy, dz, mis, tex|occluded<<31) as [pixel][5][rec_slots] words
    int rec_slots;
    // bwd
    TView diff_grad, spec_grad;
    float *pos_grad, *nrm_grad, *kd_grad, *ks_grad, *light_grad;
};

// kernel.cu:30-35
__device__ __forceinline__ uint32_t rand_pcg(uint32_t &s)
{
    uint32_t word = ((s >> ((s >> 28u) + 4u)) ^ s) * 277803737u;
    s = s * 747796405u + 2891336453u;
    return (word >> 22u) ^ word;
}
__device__ __forceinline__ xf uniform_pcg(uint32_t &s)
{
    return xf((float)(rand_pcg(s) & 0xFFFFFFu) * (1.0f / 16777216.0f));      // exact: division by 2^24
}

// kernel.cu:140-169; cdf element i at cdf[i*stride].
// The reference bisects with a fixed iteration count, i.e. 9 DEPENDENT loads at 256 entries -- the top stall of the generate
// phase (profiles/r01_v4_*).  For a non-decreasing CDF that loop returns exactly min(upper_bound(x), size-1) (first index with
// cdf[idx] > x; verified exhaustively against the reference loop incl. plateaus and non-power-of-two sizes,
// tests/test_oracle_core.py::test_cdf_bisection_is_upper_bound), so the same index is found here with a 4-ary search:
// three independent probes per step, ceil(log4(size)) steps.
__device__ __forceinline__ xf sample_cdf(const float *__restrict__ cdf, int stride, int size, int steps4, xf x, uint32_t &idx)
{
    x = xmin(x, xf(0.99999994f));
    int lo = 0, hi = size - 1;                  // answer in [lo, hi]
    for (int i = 0; i < steps4; ++i) {
        const int span = hi - lo;
        const int m1 = lo + (span >> 2), m2 = lo + (span >> 1), m3 = lo + ((3 * span) >> 2);
        const float c1 = __ldg(cdf + (size_t)m1 * stride), c2 = __ldg(cdf + (size_t)m2 * stride), c3 = __ldg(cdf + (size_t)m3 * stride);
        if (span > 0) {
            if (x.v < c1) hi = m1;
            else if (x.v < c2) { lo = m1 + 1; hi = m2; }
            else if (x.v < c3) { lo = m2 + 1; hi = m3; }
            else lo = m3 + 1;
            lo = min(lo, hi);
        }
    }
    idx = (uint32_t)hi;
    xf pdf, sample;
    if (idx == 0) { pdf = xf(__ldg(cdf)); sample = x; }
    else {
        xf d0 = xf(__ldg(cdf + (size_t)idx * stride)), d1 = xf(__ldg(cdf + (size_t)(idx - 1) * stride));
        pdf = d0 - d1; sample = x - d1;
    }
    return xmin(sample / pdf, xf(0.99999994f));
}

// kernel.cu:124-129 + 177-178: direction -> lat-long coordinate -> nearest texel (decision path)
__device__ __forceinline__ void dir_to_texel(const EnvParams &p, xf3 dir, int &tx, int &ty, float &cy)
{
    xf a = det_atan2(dir.x, -dir.z);
    float u = __double2float_rn(xd_add(xd_div((double)a.v, 2.0 * XD_PI), 0.5));
    xf ac = det_acos(xclamp(dir.y, xf(-1.0f), xf(1.0f)));
    float v = __double2float_rn(xd_div((double)ac.v, XD_PI));
    tx = min(max(__float2int_rz(__fmul_rn(u, (float)p.Wl)), 0), p.Wl - 1);
    ty = min(max(__float2int_rz(__fmul_rn(v, (float)p.Hl)), 0), p.Hl - 1);
    cy = v;
}
// kernel.cu:131-138
__device__ __forceinline__ xf3 tc_to_dir(xf ux, xf uy)
{
    xf sphi, cphi, sth, cth;
    det_sincos(xf(__double2float_rn(xd_mul((double)(ux * xf(2.0f) - xf(1.0f)).v, XD_PI))), sphi, cphi);
    det_sincos(xf(__double2float_rn(xd_mul((double)uy.v, XD_PI))), sth, cth);
    return X3(sth * sphi, cth, -sth * cphi);
}
// kernel.cu:171-182 (value only; the texel comes from dir_to_texel)
__device__ __forceinline__ float light_pdf_value(const EnvParams &p, int tx, int ty, float cy)
{
    float w = (float)(p.Hl * p.Wl) / (2.0f * MCS_PI * MCS_PI * fmaxf(sinpif(cy), 0.0001f));
    return __ldg(p.pdf + (size_t)ty * p.p_s1 + (size_t)tx * p.p_s2) * w;
}

// kernel.cu:217-237
// (the denominator cancels catastrophically at the specular peak: exact order, see bsdf.cuh "conditioning note")
__device__ __forceinline__ float eval_ndf_ggx(float alpha, float c)
{
    xf a2 = xf(alpha) * xf(alpha);
    xf d = (xf(c) * a2 - xf(c)) * xf(c) + xf(1.0f);
    return a2.v / ((d * d).v * MCS_PI);
}
__device__ __forceinline__ float eval_g1_ggx(float alphaSqr, float c)
{
    if (c <= 0.0f) return 0.0f;
    float c2 = c * c;
    float t2 = fmaxf(1.0f - c2, 0.0f) / c2;
    return 2.0f / (1.0f + sqrtf(1.0f + alphaSqr * t2));
}

// Per-pixel shading frame and lobe probabilities (kernel.cu:490-502), shared by all items of a pixel
struct PixelFrame {
    xf3 N;            // gb_normal as given
    xf3 W, U, V;      // normalised normal + orthonormal basis
    xf3 wo;           // view direction
    xf3 wo_l_raw;     // tolocal(wo)      (ggx_pdf uses it un-normalised, kernel.cu:310)
    xf3 wo_l;         // normalised       (albedo / ggx_sample, kernel.cu:87,275)
    xf alpha;
    xf pDiffuse, pSpecular;
    xf NdotV;
};

__device__ __forceinline__ xf3 x_tolocal(xf3 a, const PixelFrame &f) { return X3(xdot(a, f.U), xdot(a, f.V), xdot(a, f.W)); }
__device__ __forceinline__ xf3 x_toworld(xf3 a, const PixelFrame &f) { return f.U * a.x + f.V * a.y + f.W * a.z; }

// kernel.cu:301-323 (value path)
__device__ __forceinline__ float ggx_pdf_value(const PixelFrame &f, f3 wi)
{
    const f3 wo_l = toF3(f.wo_l_raw);
    const xf3 wi_lx = x_tolocal(X3(wi), f);
    const f3 wi_l = toF3(wi_lx);
    float pdf = 0.0f;
    if (wo_l.z > 0.0f && wi_l.z > 0.0f) {
        const f3 m = toF3(xnormalize(wi_lx + f.wo_l_raw));
        float woDotH = dot(m, wo_l);
        float alpha = f.alpha.v;
        float D = eval_ndf_ggx(alpha, m.z);
        float G1 = eval_g1_ggx(alpha * alpha, wo_l.z);
        pdf = G1 * D * fmaxf(0.0f, woDotH) / wo_l.z;
        pdf /= (4.0f * woDotH);
    }
    return pdf;
}
__device__ __forceinline__ void update_pdf(float &pdf, float opdf, float b) { if (b > 0.000001f) pdf += opdf * b; }   // kernel.cu:325-332

// kernel.cu:374-397
__device__ __forceinline__ float bsdf_pdf_value(const PixelFrame &f, xf3 wi)
{
    xf NdotL = xdot(f.N, wi);
    if (xmin(f.NdotV, NdotL).v < 1e-6f) return 1.0f;
    float pdf = 0.0f;
    float pD = f.pDiffuse.v;
    if (pD > 0.0f) update_pdf(pdf, fmaxf(NdotL.v, 0.0f) * MCS_INV_PI, pD);
    if (f.pSpecular.v > 0.0f) update_pdf(pdf, ggx_pdf_value(f, toF3(wi)), 1.0f - pD);
    return pdf;
}

// kernel.cu:334-372 (direction on the exact path, pdf on the value path)
__device__ __forceinline__ xf3 bsdf_sample(const PixelFrame &f, xf sx, xf sy, xf sz, float &pdf)
{
    pdf = 0.0f;
    const float pD = f.pDiffuse.v;
    xf3 wi;
    if (sz < f.pDiffuse) {
        if (pD < 0.0001f) { pdf = 1.0f; return f.N; }
        // cosine_sample, kernel.cu:57-79
        xf phi = xf(__double2float_rn(xd_mul(2.0 * XD_PI, (double)sx.v)));
        xf ct = xsqrt(sy);
        xf st = xf(__double2float_rn(__dsqrt_rn(__dsub_rn(1.0, (double)sy.v))));
        xf sp, cp;
        det_sincos(phi, sp, cp);
        xf3 vec = f.U * (cp * st) + f.V * (sp * st) + f.W * ct;
        wi = xnormalize(vec);
        pdf = fmaxf(0.000001f, ct.v * MCS_INV_PI) * pD;
        if (f.pSpecular.v > 0.0f) update_pdf(pdf, ggx_pdf_value(f, toF3(wi)), 1.0f - pD);
    } else {
        // ggx_sample / sampleGGX_VNDF, kernel.cu:241-291
        if (!(f.wo_l.z.v > 0.0f)) { pdf = 0.0f; wi = X3(xf(0.0f), xf(0.0f), xf(0.0f)); }
        else {
            const xf alpha = f.alpha;
            xf3 Vh = xnormalize(X3(alpha * f.wo_l.x, alpha * f.wo_l.y, f.wo_l.z));
            xf3 T1 = (Vh.z.v < 0.9999f) ? xnormalize(xcross(X3(xf(0.0f), xf(0.0f), xf(1.0f)), Vh)) : X3(xf(1.0f), xf(0.0f), xf(0.0f));
            xf3 T2 = xcross(Vh, T1);
            xf r = xsqrt(sx);
            xf phi = (xf(2.0f) * xf(MCS_PI)) * sy;
            xf sp, cp;
            det_sincos(phi, sp, cp);
            xf t1 = r * cp, t2 = r * sp;
            xf s = xf(0.5f) * (xf(1.0f) + Vh.z);
            t2 = (xf(1.0f) - s) * xsqrt(xf(1.0f) - t1 * t1) + s * t2;
            xf3 Nh = T1 * t1 + T2 * t2 + Vh * xsqrt(xmax(xf(0.0f), xf(1.0f) - t1 * t1 - t2 * t2));
            xf3 h = xnormalize(X3(alpha * Nh.x, alpha * Nh.y, xmax(xf(0.0f), Nh.z)));
            xf woDotH = xdot(f.wo_l, h);
            xf3 wi_l = h * woDotH * xf(2.0f) - f.wo_l;
            wi = xnormalize(x_toworld(wi_l, f));
            // evalPdfGGX_VNDF, kernel.cu:232-237, then the reflection Jacobian (:287)
            float a = alpha.v, woz = f.wo_l.z.v;
            float G1 = eval_g1_ggx(a * a, woz);
            float D = eval_ndf_ggx(a, h.z.v);
            pdf = G1 * D * fmaxf(0.0f, woDotH.v) / woz;
            pdf /= (4.0f * woDotH.v);
        }
        pdf *= 1.0f - pD;
        if (pD > 0.0f) update_pdf(pdf, fmaxf(xdot(f.N, wi).v, 0.0f) * MCS_INV_PI, pD);
    }
    return wi;
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// CTA-wide ray queue in shared memory.  One CTA = NW warps (32/NW CTAs per SM, 64 registers/thread).
// All warps of the CTA move through the three phases TOGETHER (barriers in between):
//   * the instruction working set at any time is one phase, shared by all resident warps (profiles/r01_v3_*: with warps
//     spread over G/T/E code, 22 % of all stall samples were instruction-fetch misses);
//   * the trace phase load-balances over the CTA: warp w owns segment w of the queue (the live rays of "its" pixel),
//     drains it first and then steals from the other segments, so no lane idles while any ray of the batch is untraced.
// Layout is SoA, conflict-free: lane k of a warp touches word k of a segment.  tex bit 31 = "occluded" flag (trace phase).
// ---------------------------------------------------------------------------------------------
constexpr int REPLAY_MINB = 3;          // replay kernel: 80 registers, 3 CTAs/SM (2.93 -> 2.54 ms on 4 views; 4 CTAs/SM spills, software prefetch was slower)
constexpr int NW = 8;                    // warps per CTA (16-warp CTAs x 2 per SM measured +4 %)
constexpr int SPLIT_BELOW = 20;          // while a batch drains, idle lanes are handed subtrees when fewer than this many are walking
constexpr int QSTACK = 100;              // traversal stack entries per lane
constexpr int LEAF_BATCH = 32;           // deferred leaf tests are run when this many (ray, leaf) pairs are pending
constexpr int REFILL_BELOW = 24;         // idle lanes are refilled when fewer than this many are walking (picking up a ray is cheap: rayq_fetch)
constexpr int SEG = 128;                 // queue entries per warp segment (= one pixel at N = 8)
constexpr int QTOT = NW * SEG;
// pending (ray, leaf) pairs per warp: < LEAF_BATCH carried over + at most 128 appended per node step.  64 (flush inside the deferral
// loop, 6 KB less smem, 132 KB carve-out => 124 KB of L1) measured +5.6 %: profiles/r02_envshade_ab.json
constexpr int PCAP = 160;
static_assert(PCAP >= LEAF_BATCH + 4 * 32, "a node step appends up to four pairs per lane without a flush");
constexpr int PIXRING = 256;
static_assert(QTOT <= 65536, "queue entry index is stored in 16 bits");
static_assert(SEG <= 256 && SEG % 32 == 0, "sample slot within a fill is stored in 8 bits");

struct BlockQueue {
    float dx[QTOT], dy[QTOT], dz[QTOT], mis[QTOT];
    uint32_t tex[QTOT];
    uint16_t vlist[QTOT];                // per segment: dense list of entries that reach the eval phase
    uint8_t qitem[QTOT];                 // sample slot of the entry within the current queue fill (w - w0 < SEG)
    uint32_t hitw[NW][SEG / 32];         // per segment: occluded bits of the current queue fill
    uint2 pl[NW][PCAP];                  // per warp: deferred leaf tests, x = queue entry, y = leaf code
    float ro[NW][3];                     // per segment: ray origin / view vector / pixel id / live-ray count / fetch cursor
    float rog[NW][3];                    // per segment: quantisation-grid origin - ray origin (rounded once, rayq_fetch)
    float wo[NW][3];
    int pixid[NW];
    int seg_cnt[NW];
    int seg_head[NW];
    int pixring[PIXRING];                // active pixels waiting for a batch
    int ring_head, ring_tail, more_chunks;
};
struct BlockQueueRec { uint32_t slot[QTOT]; };   // MODE 2 only

struct PixelIn {
    f3 ro, pos, nrm, view, kd, ks;
    int ix, iy, iz;
    int64_t pix;
};

__device__ __forceinline__ PixelIn load_pixel(const EnvParams &p, int64_t pix)
{
    PixelIn q;
    q.pix = pix;
    q.ix = (int)(pix % p.W);
    const int64_t tt = pix / p.W;
    q.iy = (int)(tt % p.H); q.iz = (int)(tt / p.H);
    q.ro = p.ro.ld3(q.iz, q.iy, q.ix);
    q.pos = p.pos.ld3(q.iz, q.iy, q.ix);
    q.nrm = p.nrm.ld3(q.iz, q.iy, q.ix);
    q.view = p.view.ld3(q.iz, q.iy, q.ix);
    q.kd = p.kd.ld3(q.iz, q.iy, q.ix);
    q.ks = p.ks.ld3(q.iz, q.iy, q.ix);
    return q;
}

// ---------------------------------------------------------------------------------------------
// Per-ray and per-pixel code of phase E, shared by env_shade_kernel and env_shade_replay_kernel: the re-tracing backward and the
// record-replaying backward must give bit-identical per-pixel gradients, so they run the same code.  P = EnvParams or ReplayParams.
// ---------------------------------------------------------------------------------------------
// A ray's tex word: env texel ty << 16 | tx; bit 31 = occluded, set in phase T.
__device__ __forceinline__ uint32_t tex_pack(int tx, int ty) { return (uint32_t)((ty << 16) | tx); }
__device__ __forceinline__ void tex_unpack(uint32_t tex, int &tx, int &ty) { tx = tex & 0xFFFFu; ty = (tex >> 16) & 0x7FFFu; }

// Ray record written by the forward pass for the backward: per pixel (rr = rec_rays + pix * 5 * slots), the evaluated rays in
// evaluation order as coalesced SoA rows [5][slots] of (dx, dy, dz, mis, tex); k = the ray's position in that order.  Streaming
// (evict-first) stores and loads: 1.8 GB of record per launch must not push the BVH / probe tables out of the L2.
__device__ __forceinline__ void rec_store(float *rr, int slots, int k, const f3 &wi, float mis, uint32_t tex)
{
    __stcs(rr + k, wi.x); __stcs(rr + slots + k, wi.y); __stcs(rr + 2 * slots + k, wi.z);
    __stcs(rr + 3 * slots + k, mis); __stcs(rr + 4 * slots + k, __uint_as_float(tex));
}
__device__ __forceinline__ void rec_load(const float *rr, int slots, int k, f3 &wi, float &mis, uint32_t &tex)
{
    wi = F3(__ldcs(rr + k), __ldcs(rr + slots + k), __ldcs(rr + 2 * slots + k));
    mis = __ldcs(rr + 3 * slots + k);
    tex = __float_as_uint(__ldcs(rr + 4 * slots + k));
}

// process_sample, kernel.cu:403-461: radiance of the ray's env texel and the BSDF value
template <class P>
__device__ __forceinline__ f3 ray_eval(const P &p, bool diffuse_only, const f3 &kd, const f3 &ks, const f3 &wo, const f3 &nrm, const f3 &wi,
                                       int tx, int ty, float &diffv, f3 &specv)
{
    const float *lp = p.light + (size_t)ty * p.l_s1 + (size_t)tx * p.l_s2;
    const f3 light_col = F3(__ldg(lp), __ldg(lp + p.l_s3), __ldg(lp + 2 * p.l_s3));
    diffv = 0.0f; specv = F3(0.0f);
    if (diffuse_only) diffv = fwd_lambert(nrm, wi);
    else ox_fwd_pbr_bsdf(kd, ks, wo, nrm, wi, MIN_ROUGHNESS, diffv, specv);
    return light_col;
}

// One ray's adjoint (process_sample's backward branch, kernel.cu:422-457): light gradient scattered with float atomics, zero
// contributions skipped (kernel.cu:424-425 / 203-211), BSDF adjoint accumulated into the lane's per-pixel sums.
template <class P>
__device__ __forceinline__ void ray_adjoint(const P &p, bool diffuse_only, const f3 &kd, const f3 &ks, const f3 &wo, const f3 &nrm,
                                            const f3 &dgrad, const f3 &sgrad, const f3 &wi, int tx, int ty, float wgt,
                                            f3 &g_kd, f3 &g_ks, f3 &g_nrm, f3 &g_wo)
{
    float diffv; f3 specv;
    const f3 light_col = ray_eval(p, diffuse_only, kd, ks, wo, nrm, wi, tx, ty, diffv, specv);
    // (dgrad * diffv + sgrad * specv) * wgt, contracted explicitly so that the rounding does not depend on how the compiler fuses it
    const f3 lg = F3(fmaf(dgrad.x, diffv, sgrad.x * specv.x), fmaf(dgrad.y, diffv, sgrad.y * specv.y), fmaf(dgrad.z, diffv, sgrad.z * specv.z)) * wgt;
    float *gp = p.light_grad + ((size_t)ty * p.Wl + tx) * 3;
    if (lg.x != 0.0f) atomicAdd(gp, lg.x);
    if (lg.y != 0.0f) atomicAdd(gp + 1, lg.y);
    if (lg.z != 0.0f) atomicAdd(gp + 2, lg.z);
    const f3 dD = dgrad * light_col * wgt, dS = sgrad * light_col * wgt;
    if (diffuse_only) { f3 wi_grad = F3(0.0f); bwd_lambert(nrm, wi, g_nrm, wi_grad, sum(dD)); }
    else ox_bwd_pbr_bsdf(kd, ks, wo, nrm, wi, MIN_ROUGHNESS, g_kd, g_ks, g_wo, g_nrm, sum(dD), dS);
}

// Warp reduction of one pixel's adjoints, single writer per pixel (kernel.cu:442-456, 533-541).
template <class P>
__device__ __forceinline__ void pixel_grad_write(const P &p, int64_t pix, int lane, const f3 &pos, const f3 &view,
                                                 const f3 &g_kd, const f3 &g_ks, const f3 &g_nrm, const f3 &g_wo)
{
    f3 t_kd = F3(warp_sum(g_kd.x), warp_sum(g_kd.y), warp_sum(g_kd.z));
    f3 t_ks = F3(warp_sum(g_ks.x), warp_sum(g_ks.y), warp_sum(g_ks.z));
    f3 t_nrm = F3(warp_sum(g_nrm.x), warp_sum(g_nrm.y), warp_sum(g_nrm.z));
    f3 t_wo = F3(warp_sum(g_wo.x), warp_sum(g_wo.y), warp_sum(g_wo.z));
    if (lane == 0) {
        // wo = normalize(view_pos - pos): d_pos = -J^T d_wo (bsdf.h:270-274; d_view_pos is dropped, ops.py:105)
        f3 d__wo = F3(0.0f);
        bwd_safe_normalize(view - pos, d__wo, t_wo);
        float *a = p.pos_grad + pix * 3, *b = p.nrm_grad + pix * 3, *c = p.kd_grad + pix * 3, *d = p.ks_grad + pix * 3;
        a[0] = -d__wo.x; a[1] = -d__wo.y; a[2] = -d__wo.z;
        b[0] = t_nrm.x; b[1] = t_nrm.y; b[2] = t_nrm.z;
        c[0] = t_kd.x; c[1] = t_kd.y; c[2] = t_kd.z;
        d[0] = t_ks.x; d[1] = t_ks.y; d[2] = t_ks.z;
    }
}

// Gradients of a pixel that evaluates no ray (masked: the reference returns early on zero-initialised tensors, kernel.cu:478)
template <class P>
__device__ __forceinline__ void pixel_grad_zero(const P &p, int64_t pix)
{
    float *a = p.pos_grad + pix * 3, *b = p.nrm_grad + pix * 3, *c = p.kd_grad + pix * 3, *d = p.ks_grad + pix * 3;
    a[0] = a[1] = a[2] = 0.0f; b[0] = b[1] = b[2] = 0.0f; c[0] = c[1] = c[2] = 0.0f; d[0] = d[1] = d[2] = 0.0f;
}

// kernel.cu:490-502: shading frame + lobe probabilities
__device__ __forceinline__ void make_frame(const PixelIn &q, PixelFrame &f)
{
    f.N = X3(q.nrm);
    f.alpha = xf(q.ks.y) * xf(q.ks.y);
    f.wo = xnormalize(X3(q.view) - X3(q.pos));
    xf metallic = xf(q.ks.z);
    xf3 base = X3(q.kd);
    xf om = xf(1.0f) - metallic;
    xf3 specColor = X3(xf(0.04f) * om + base.x * metallic, xf(0.04f) * om + base.y * metallic, xf(0.04f) * om + base.z * metallic);
    xf lum = base.x * xf(0.2126f) + base.y * xf(0.7152f) + base.z * xf(0.0722f);
    xf diffuseWeight = om * lum;
    // albedo(), kernel.cu:81-94
    f.W = xnormalize(f.N);
    xONB(f.W, f.U, f.V);
    f.wo_l_raw = x_tolocal(f.wo, f);
    f.wo_l = xnormalize(f.wo_l_raw);
    xf specularWeight = xf(0.0f);
    if (f.wo_l.z.v > 0.0f) {
        xf c = xclamp(f.wo_l.z, xf(1e-4f), xf(1.0f) - xf(1e-4f));
        xf o = xf(1.0f) - c;
        xf o2 = o * o;
        xf scale = (o2 * o2) * o;
        xf os = xf(1.0f) - scale;
        xf3 F = X3(specColor.x * os + scale, specColor.y * os + scale, specColor.z * os + scale);
        specularWeight = F.x * xf(0.2126f) + F.y * xf(0.7152f) + F.z * xf(0.0722f);
    }
    xf sumw = diffuseWeight + specularWeight;
    f.pDiffuse = sumw.v > 0.0f ? diffuseWeight / sumw : xf(1.0f);
    f.pSpecular = xf(1.0f) - f.pDiffuse;
    f.NdotV = xdot(f.N, f.wo);
}

// Per-ray constants of the quantised node test (bvh.cu:k_emit_nodesq): plane t = (origin + q * cell - o) / d = q' * A + B with
// q' = 2^23 + q (the float whose low mantissa bits are the 16-bit coordinate), A = cell / d (exact: cell is a power of two),
// B = (origin - o) / d - 2^23 * A.  |error| < 0.51 cell (rounding of B), covered by the two-cell inflation of the stored boxes.
// The byte-permute that builds q' also picks the entry / exit plane from the (lo | hi << 16) word: its selector depends on the
// sign of d only, so the slab test needs no min/max per axis.  Zero direction components are nudged to +-1e-20 (keeps 2^23 * A
// finite for any sane scene; same conservative argument as ray_pre's 1e-30).
struct RayQ {
    float ax, ay, az, bx, by, bz;
    uint32_t nx, ny, nz, fx, fy, fz; // PRMT selectors of the entry / exit planes (0x7410 = low half, 0x7432 = high half)
};
// None of these constants is part of the parity contract: culling only has to be CONSERVATIVE (the boolean result comes from the
// exact triangle predicate), and the stored boxes carry a margin of two cells per side against a decode error of ~0.52 cell.  So
// 1/d is one MUFU.RCP (relative error 2^-23: < 0.02 cell over the whole grid) instead of an IEEE division -- picking up a ray
// costs half the instructions, which is what allows refilling idle lanes early (REFILL_BELOW).
__device__ __forceinline__ float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ RayQ rayq_fetch(const float *__restrict__ g, const float *rog, float dx, float dy, float dz)
{
    RayQ r;
    const float ix = rcp_approx(fabsf(dx) < 1e-20f ? copysignf(1e-20f, dx) : dx);
    const float iy = rcp_approx(fabsf(dy) < 1e-20f ? copysignf(1e-20f, dy) : dy);
    const float iz = rcp_approx(fabsf(dz) < 1e-20f ? copysignf(1e-20f, dz) : dz);
    r.ax = __ldg(g + 3) * ix; r.ay = __ldg(g + 4) * iy; r.az = __ldg(g + 5) * iz;
    r.bx = fmaf(-8388608.0f, r.ax, rog[0] * ix);
    r.by = fmaf(-8388608.0f, r.ay, rog[1] * iy);
    r.bz = fmaf(-8388608.0f, r.az, rog[2] * iz);
    r.nx = dx < 0.0f ? 0x7432u : 0x7410u; r.ny = dy < 0.0f ? 0x7432u : 0x7410u; r.nz = dz < 0.0f ? 0x7432u : 0x7410u;
    r.fx = dx < 0.0f ? 0x7410u : 0x7432u; r.fy = dy < 0.0f ? 0x7410u : 0x7432u; r.fz = dz < 0.0f ? 0x7410u : 0x7432u;
    return r;
}
// prmt.b32 directly: __byte_perm() masks its selector with 0x7777 first (one LOP3 per use); these selectors never set the
// sign-replication bits.
__device__ __forceinline__ float qplane(uint32_t w, uint32_t sel)
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(0x4B000000u), "r"(sel));
    return __uint_as_float(r);
}
// Slab test against one quantised child box.  Conservative without any relaxation of the comparison: every decoded plane is within
// 0.52 cell (in t * |d| units) of the true plane of the STORED box, and the stored box is the padded node box rounded outward and
// inflated by two more cells per side (bvh.cu:k_emit_nodesq), so each computed entry is below and each computed exit above the
// true ones of the node box: a ray that meets the node box at some t >= 0 always passes.  The upper end of the ray interval
// (t < 1e16) is enforced by the triangle test; not clamping the exit here only admits more boxes.
__device__ __forceinline__ bool qslab(const uint4 c, const RayQ &r)
{
    const float a0 = fmaf(qplane(c.x, r.nx), r.ax, r.bx), a1 = fmaf(qplane(c.x, r.fx), r.ax, r.bx);
    const float b0 = fmaf(qplane(c.y, r.ny), r.ay, r.by), b1 = fmaf(qplane(c.y, r.fy), r.ay, r.by);
    const float c0 = fmaf(qplane(c.z, r.nz), r.az, r.bz), c1 = fmaf(qplane(c.z, r.fz), r.az, r.bz);
    const float tn = fmaxf(fmaxf(a0, b0), fmaxf(c0, 0.0f));
    const float tf = fminf(fminf(a1, b1), c1);
    return tn <= tf;
}

// ---- phase G: generate the items [w0, w1) of one pixel, push the rays that can contribute into segment `seg` ----------
template <int MODE>
__device__ __forceinline__ void gen_segment(const EnvParams &p, BlockQueue &q, BlockQueueRec *qr, const PixelIn &px, const PixelFrame &f,
                                            int seg, int w0, int w1, int &qn, const int lane)
{
    const int S = p.S;
    const int qb = seg * SEG;
    const xf strata_frac = xf(1.0f) / xf((float)(unsigned)p.N);
    // RNG, kernel.cu:504-505
    uint32_t s_seed = p.seed + (p.seed_dev ? __ldg(p.seed_dev) : 0u), s_pix = (uint32_t)(((px.iz + p.batch_offset) * p.H + px.iy) * p.W + px.ix);
    uint32_t rng = rand_pcg(s_seed) ^ rand_pcg(s_pix);
    const uint32_t lightIdx = rand_pcg(rng) % p.n_perms;
    const uint32_t bsdfIdx = rand_pcg(rng) % p.n_perms;
    const uint32_t rng2 = rng;
    const f3 nrm = px.nrm;

    // Two stages (MODE 0 / 1).  Stage A draws the direction of every sample (all lanes busy) and ballot-compacts the LIVE ones --
    // n.wi > 0 -- into the queue; stage B runs the rest of the sample set-up (lat-long texel of the direction: atan2 + acos + two
    // double divisions, light pdf, and for light samples the BSDF pdf) on the compacted list only, i.e. not for the ~27 % of the
    // samples that are dropped anyway.  Same operations on the same values in the same order per sample: results are bit-identical
    // to the single-stage path, which MODE 2 keeps because it records the texel of every sample, dropped or not.
    for (int base = w0; base < w1; base += 32) {
        const int w = base + lane;
        const bool valid = w < w1;
        const bool is_bsdf = w >= S;
        const int i = is_bsdf ? w - S : w;
        xf3 dir = X3(xf(0.0f), xf(0.0f), xf(1.0f));
        float pdf_sum = 1.0f, pdf_b = 0.0f;
        int tx = 0, ty = 0;
        if (valid) {
            const uint2 sk = __ldg(p.skip + 5 * i + (is_bsdf ? 2 : 0));
            uint32_t st = rng2 * sk.x + sk.y;
            const uint32_t row = is_bsdf ? bsdfIdx : lightIdx;
            const uint32_t perm = (uint32_t)__ldg(p.perms + (size_t)row * p.pm_s1 + (size_t)i * p.pm_s3);
            const xf sx = (xf((float)(perm % (uint32_t)p.N)) + uniform_pcg(st)) * strata_frac;
            const xf sy = (xf((float)(perm / (uint32_t)p.N)) + uniform_pcg(st)) * strata_frac;
            if (!is_bsdf) {
                // lightSample, kernel.cu:184-193
                uint32_t cyi, cxi;
                xf ry = sample_cdf(p.rows, p.r_s, p.Hl, p.m_rows, sy, cyi);
                xf rx = sample_cdf(p.cols + (size_t)cyi * p.c_s1, p.c_s2, p.Wl, p.m_cols, sx, cxi);
                dir = tc_to_dir((xf((float)cxi) + rx) / xf((float)p.Wl), (xf((float)cyi) + ry) / xf((float)p.Hl));
            } else {
                const xf sz = uniform_pcg(st);
                dir = bsdf_sample(f, sx, sy, sz, pdf_b);
            }
            if (MODE == 2) {
                float cy;
                dir_to_texel(p, dir, tx, ty, cy);
                pdf_sum = light_pdf_value(p, tx, ty, cy) + (is_bsdf ? pdf_b : bsdf_pdf_value(f, dir));
            }
        }
        const f3 wi = toF3(dir);
        // A sample contributes (value and every adjoint) only if n.wi > 0: Lambert is max(n.wi/pi, 0) and the GGX lobe is gated by
        // wiDotN > 1e-4 (bsdf.h:21-30,160,186); everything else is multiplied by those.  Such rays are neither traced nor evaluated.
        const bool live = valid && dot(nrm, wi) > 0.0f;
        if (MODE == 2 && valid) {
            const size_t rec = (size_t)px.pix * (2 * S) + (size_t)(2 * i + (is_bsdf ? 1 : 0));
            p.rec_texel[rec] = (int32_t)tex_pack(tx, ty);
            if (!live) p.rec_vis[rec] = 2;
        }
        const unsigned m = __ballot_sync(0xFFFFFFFFu, live);
        if (live) {
            const int e = qb + qn + __popc(m & ((1u << lane) - 1u));
            q.dx[e] = wi.x; q.dy[e] = wi.y; q.dz[e] = wi.z;
            if (MODE == 2) {
                q.mis[e] = 1.0f / fmaxf(pdf_sum, 0.0001f);      // MIS balance heuristic, kernel.cu:409
                q.tex[e] = tex_pack(tx, ty);
                qr->slot[e] = (uint32_t)(2 * i + (is_bsdf ? 1 : 0));
            } else {
                q.mis[e] = pdf_b;                               // stage B turns these two into the MIS weight and the texel
                q.tex[e] = is_bsdf ? 1u : 0u;
            }
            q.qitem[e] = (uint8_t)(w - w0);
        }
        qn += __popc(m);
    }
    if (MODE != 2) {
        __syncwarp();
        for (int e0 = 0; e0 < qn; e0 += 32) {
            const int e = qb + e0 + lane;
            if (e0 + lane < qn) {
                const xf3 dir = X3(xf(q.dx[e]), xf(q.dy[e]), xf(q.dz[e]));
                int tx, ty; float cy;
                dir_to_texel(p, dir, tx, ty, cy);
                const float pdf_sum = light_pdf_value(p, tx, ty, cy) + (q.tex[e] ? q.mis[e] : bsdf_pdf_value(f, dir));
                q.mis[e] = 1.0f / fmaxf(pdf_sum, 0.0001f);      // MIS balance heuristic, kernel.cu:409
                q.tex[e] = tex_pack(tx, ty);
            }
        }
    }
}

// ---- phase T: any-hit traversal of all queued rays of the CTA: work stealing + dynamic fetch + deferred leaf tests ----
// SIMT-friendly organisation (profiles/r01_v2_*: a classic while-while loop ran at 13/32 lanes because lanes wait for each
// other at every leaf):
//   * node loop: every busy lane performs exactly one node step per iteration (fetch the quantised node -- 64 bytes, four
//     children, one 128-bit load per child -- four slab tests, push / continue / pop).  Leaf children that pass the slab test are NOT intersected here:
//     the (ray, leaf run) pair is appended to the warp's pending list (ballot compaction) and the lane keeps walking,
//     speculating that the leaf misses;
//   * as soon as 32 pairs are pending the warp intersects them with all lanes busy; a hit sets the ray's "occluded" bit
//     (tex bit 31), which the owning lane polls after each batch to abandon the walk;
//   * a lane whose walk ends pulls the next ray -- from the warp's own segment first, then from the other warps' segments --
//     as soon as fewer than REFILL_BELOW lanes are busy;
//   * when nothing is left to pull (the drain of a batch: the long walks), idle lanes are handed the BOTTOM stack entry of busy lanes
//     and walk that subtree for the same ray (below SPLIT_BELOW busy lanes);
//   * visibility of a ray = its occluded bit after all segments AND all pending lists have drained (block barrier).
// One visit = ~100 SASS instructions (round 1: ~150): raw prmt plane decode with six selector registers, no comparison relax, leaf
// flags from the node word, unconditional child stores with a conditional stack-pointer bump.
// What bounds it (profiles/r02_envshade_*): instruction issue + latency (73 % issue-active, 24 of 32 lanes = 54 % of the
// thread-instruction peak; no pipe above 60 %).  With fp32 64-byte binary nodes (4 loads
// per visit) the L1 data pipe was a co-limiter at 75 %; quantised nodes took it to 47 % and long-scoreboard stalls from 25 % to
// 18 % at equal run time; the 4-wide view then halves the visits (13.8 vs 28.8 per ray) for -8 % run time.  Measured and
// rejected: 4-wide fp32 nodes (7 loads per visit: L1-bound, +5 %), node fetch through the texture path (equal), per-node
// instead of per-leaf deferral (leaf phase drops to 17 lanes), an 8-wide compressed node with 8-bit boxes (profiles/r01_bvh8_*: more instructions per ray),
// sorting the BSDF samples of a pixel by lobe before sampling (one routine per chunk instead of two at 16 lanes: +1.7 %).
__device__ __forceinline__ void trace_queue(const EnvParams &p, BlockQueue &q, const int warp, const int lane)
{
    unsigned lt;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt));
    int pend = 0;
    int my = -1;
    int node = 0, sp = 0, sb = 0;                // stack = entries [sb, sp): the owner pops at the top, idle lanes are handed the bottom
    int stack[QSTACK];                           // up to 3 pushes per visit (1.5 per binary level of the LBVH walk) + one scratch slot
    RayQ r; r.ax = r.ay = r.az = 1.0f; r.bx = r.by = r.bz = 0.0f; r.nx = r.ny = r.nz = 0x7410u; r.fx = r.fy = r.fz = 0x7432u;
    const BvhView b = p.bvh;
    uint2 *pl = q.pl[warp];
    int seg = warp, exhausted = 0;           // segment being drained, number of segments found empty so far

    auto leaf_batch = [&](int n) {
        // intersect the last n (<= 32) pending (ray, leaf run) pairs, one per lane
        __syncwarp();
        const int base = pend - n;
        if (lane < n) {
            const uint2 ent = pl[base + lane];
            const int e = (int)ent.x;
            if (!(q.tex[e] >> 31)) {
                const int code = (int)ent.y;             // leaf run: (first triangle << 3) | (count - 1)
                const int start = code >> 3, cnt = (code & 7) + 1;
                const int ps = e / SEG;
                const f3 o = F3(q.ro[ps][0], q.ro[ps][1], q.ro[ps][2]);
                const f3 d = F3(q.dx[e], q.dy[e], q.dz[e]);
                bool hit = false;
                for (int k = 0; k < cnt && !hit; ++k) {
                    const float4 *t = b.tris + 3 * (size_t)(start + k);
                    const float4 t0 = __ldg(t), t1 = __ldg(t + 1), t2 = __ldg(t + 2);
                    float tt, uu, vv;
                    hit = mt_hit(o, d, F3(t0.x, t0.y, t0.z), F3(t1.x, t1.y, t1.z), F3(t2.x, t2.y, t2.z), MCS_TMAX, tt, uu, vv);
                }
                if (hit) atomicOr(&q.tex[e], 0x80000000u);
            }
        }
        pend = base;
        __syncwarp();
    };

    while (true) {
        // ---- refill idle lanes: own segment first, then steal ----
        unsigned idle = __ballot_sync(0xFFFFFFFFu, my < 0);
        while (idle && exhausted < NW) {
            const int need = __popc(idle);
            int base = 0;
            if (lane == 0) base = atomicAdd(&q.seg_head[seg], need);
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            const int avail = q.seg_cnt[seg] - base;
            if (avail <= 0) { seg = seg + 1 == NW ? 0 : seg + 1; ++exhausted; continue; }
            const int take = avail < need ? avail : need;
            const int rank = __popc(idle & lt);
            if (my < 0 && rank < take) {
                const int idx = seg * SEG + base + rank;
                my = idx;
                r = rayq_fetch(b.qgrid, q.rog[seg], q.dx[idx], q.dy[idx], q.dz[idx]);
                node = 0; sp = 0; sb = 0;
            }
            if (take < need) { seg = seg + 1 == NW ? 0 : seg + 1; ++exhausted; }
            idle = __ballot_sync(0xFFFFFFFFu, my < 0);
        }
        // ---- drain: nothing left to fetch.  The last rays of a batch are the long walks, and a warp used to finish them at a handful of
        // lanes (22.9 / 32 lanes on average over the whole kernel, profiles/r02_envshade_ab.json).  An any-hit walk is a set of
        // independent subtrees, so idle lanes take the BOTTOM stack entry (the largest pending subtree) of busy lanes and walk it for
        // the same ray: the k-th idle lane pairs with the k-th lane that has something to give.  The verdict is the ray's occluded
        // bit, set by whichever lane finds a hit -- the result cannot depend on who walks what.
        if (exhausted >= NW && idle) {
            const unsigned donors = __ballot_sync(0xFFFFFFFFu, my >= 0 && sp > sb);
            if (donors) {
                const int npair = min(__popc(idle), __popc(donors));
                // k-th donor -> k-th idle lane through the tail of the pending list (free here: pend < LEAF_BATCH at the loop top)
                uint2 *xch = pl + (PCAP - 32);
                const int kd = __popc(donors & lt), ki = __popc(idle & lt);
                if (my >= 0 && sp > sb && kd < npair) { xch[kd] = make_uint2((unsigned)my, (unsigned)stack[sb]); ++sb; }
                __syncwarp();
                if (my < 0 && ki < npair) {
                    const uint2 g = xch[ki];
                    my = (int)g.x; node = (int)g.y; sp = 0; sb = 0;
                    const int ps = my / SEG;
                    r = rayq_fetch(b.qgrid, q.rog[ps], q.dx[my], q.dy[my], q.dz[my]);
                }
                __syncwarp();
            }
        }
        int nact = __popc(__ballot_sync(0xFFFFFFFFu, my >= 0));
        if (nact == 0) {
            if (pend == 0) break;
            leaf_batch(pend < 32 ? pend : 32);        // final flush (nothing left to fetch, no walker left)
            continue;
        }
        // while draining, come back here after every node step that leaves lanes idle, so that they can be handed subtrees
        const int thresh = exhausted < NW ? REFILL_BELOW : SPLIT_BELOW;
        do {
            const int cur = my;
            unsigned lmask = 0u;
            int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
            if (my >= 0) {
                const uint4 *n = b.nodesq4 + 4 * (size_t)node;
                const uint4 k0 = __ldg(n), k1 = __ldg(n + 1), k2 = __ldg(n + 2), k3 = __ldg(n + 3);
                const bool h0 = qslab(k0, r), h1 = qslab(k1, r), h2 = qslab(k2, r), h3 = qslab(k3, r);
                const unsigned hm = (h0 ? 1u : 0u) | (h1 ? 2u : 0u) | (h2 ? 4u : 0u) | (h3 ? 8u : 0u);
                const unsigned lb = k0.w >> 28;                       // which of the four children are leaf runs (bvh.cu:k_emit_nodesq)
                c0 = (int)(k0.w & 0x0FFFFFFFu); c1 = (int)k1.w; c2 = (int)k2.w; c3 = (int)k3.w;
                lmask = hm & lb;
                const unsigned im = hm & ~lb;
                // internal children hit: push them all with UNCONDITIONAL stores and a conditional stack-pointer bump (a slot above
                // sp is scratch), continue with the last one straight from its register (its slot is released again); nothing hit ->
                // pop.  any-hit: the visiting order does not change the result.
                stack[sp] = c0; sp += (int)(im & 1u);
                stack[sp] = c1; sp += (int)((im >> 1) & 1u);
                stack[sp] = c2; sp += (int)((im >> 2) & 1u);
                stack[sp] = c3; sp += (int)(im >> 3);
                if (im) { node = (im & 8u) ? c3 : ((im & 4u) ? c2 : ((im & 2u) ? c1 : c0)); --sp; }
                else if (sp > sb) node = stack[--sp];
                else my = -1;                               // walk finished; verdict comes from the occluded bit
            }
            // defer the leaf tests: one (ray, leaf run) pair per leaf child hit, one ballot round per pair of the busiest lane
            for (unsigned mL = __ballot_sync(0xFFFFFFFFu, lmask != 0u); mL; mL = __ballot_sync(0xFFFFFFFFu, lmask != 0u)) {
                if (lmask) {
                    const unsigned low = lmask & (0u - lmask);
                    const int code = (low & 3u) ? ((low & 1u) ? c0 : c1) : ((low & 4u) ? c2 : c3);
                    pl[pend + __popc(mL & lt)] = make_uint2((unsigned)cur, (unsigned)code);
                    lmask ^= low;
                }
                pend += __popc(mL);      // (one entry per LANE -- node << 4 | leaf mask -- with the child words re-read in the batch: measured +4.3 %)
            }
            nact = __popc(__ballot_sync(0xFFFFFFFFu, my >= 0));
        } while (pend < LEAF_BATCH && nact >= thresh);
        while (pend >= LEAF_BATCH) leaf_batch(32);
        // occluded bits of this warp's rays only change inside leaf_batch (a ray is walked and leaf-tested by one warp):
        // poll here instead of once per node step
        if (my >= 0 && (q.tex[my] >> 31)) my = -1;
    }
    __syncwarp();
}

// MODE 0: forward, 1: backward, 2: forward + per-ray records
template <int MODE>
__global__ void __launch_bounds__(NW * 32, 32 / NW) env_shade_kernel(const EnvParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    BlockQueue &q = *reinterpret_cast<BlockQueue *>(smem_raw);
    BlockQueueRec *qr = MODE == 2 ? reinterpret_cast<BlockQueueRec *>(smem_raw + sizeof(BlockQueue)) : nullptr;

    const int64_t npix = (int64_t)p.B * p.H * p.W;
    const unsigned int nchunks = (unsigned int)((npix + 31) / 32);
    const int S = p.S, items = 2 * S;
    const float sample_frac = (xf(1.0f) / xf((float)(unsigned)(p.N * p.N))).v;
    const bool diffuse_only = (p.bsdf == 1u || p.bsdf == 2u);
    const bool trace_needed = p.shadow_scale != 0.0f;
    const float v_occluded = 1.0f - p.shadow_scale;          // V of an occluded ray (kernel.cu:420)
    const int nsub = (items + SEG - 1) / SEG;                // queue fills per pixel (1 for N <= 8)
    const int qb = warp * SEG;

    if (threadIdx.x == 0) { q.ring_head = 0; q.ring_tail = 0; q.more_chunks = 1; }
    __syncthreads();

    while (true) {
        // ---- collect active pixels: two warps claim 32-pixel chunks until a full batch is waiting ----
        while (true) {
            const int have = q.ring_tail - q.ring_head;
            const int more = q.more_chunks;
            __syncthreads();
            if (have >= NW || !more) break;
            if (warp < 2) {
                unsigned int chunk = 0;
                if (lane == 0) chunk = atomicAdd(p.chunk_counter, 1u);
                chunk = __shfl_sync(0xFFFFFFFFu, chunk, 0);
                if (chunk >= nchunks) { if (lane == 0) q.more_chunks = 0; }
                else {
                    const int64_t mypix = (int64_t)chunk * 32 + lane;
                    const bool mine = mypix < npix;
                    float mval = 0.0f;
                    if (mine) {
                        const int mx = (int)(mypix % p.W); const int64_t t = mypix / p.W;
                        mval = p.mask.ld1((int)(t / p.H), (int)(t % p.H), mx);
                    }
                    const bool act = mine && mval > 0.0f;
                    const unsigned am = __ballot_sync(0xFFFFFFFFu, act);
                    if (mine && !act) {
                        // masked pixel: outputs are zero (the reference returns early on zero-initialised tensors, kernel.cu:478)
                        if (MODE != 1) {
                            float *d = p.diff + mypix * 3, *s = p.spec + mypix * 3;
                            d[0] = d[1] = d[2] = 0.0f; s[0] = s[1] = s[2] = 0.0f;
                            if (p.hit_out) for (int k = 0; k < p.hit_words; ++k) p.hit_out[(size_t)mypix * p.hit_words + k] = 0u;
                            if (p.rec_count) p.rec_count[mypix] = 0u;
                        } else pixel_grad_zero(p, mypix);
                    }
                    int base = 0;
                    if (lane == 0 && am) base = atomicAdd(&q.ring_tail, __popc(am));
                    base = __shfl_sync(0xFFFFFFFFu, base, 0);
                    if (act) q.pixring[(base + __popc(am & ((1u << lane) - 1u))) & (PIXRING - 1)] = (int)mypix;
                }
            }
            __syncthreads();
        }
        const int have = q.ring_tail - q.ring_head;
        if (have <= 0) break;
        const int nb = have < NW ? have : NW;                 // pixels in this batch (one per warp)
        const bool has_px = warp < nb;
        const int64_t mypx = has_px ? (int64_t)q.pixring[(q.ring_head + warp) & (PIXRING - 1)] : 0;
        __syncthreads();
        if (threadIdx.x == 0) q.ring_head += nb;

        // accumulators live across queue fills when one pixel needs several (items > SEG)
        f3 accD = F3(0.0f), accS = F3(0.0f);
        f3 g_kd = F3(0.0f), g_ks = F3(0.0f), g_nrm = F3(0.0f), g_wo = F3(0.0f);
        int rec_off = 0;

        for (int sub = 0; sub < nsub; ++sub) {
            const int w0 = sub * SEG, w1 = min(items, w0 + SEG);
            // ================= phase G =================
            int qn = 0;
            if (has_px) {
                const PixelIn px = load_pixel(p, mypx);
                PixelFrame f;
                make_frame(px, f);
                if (lane < 3) {
                    const float ro_l = lane == 0 ? px.ro.x : (lane == 1 ? px.ro.y : px.ro.z);
                    q.rog[warp][lane] = __fsub_rn(__ldg(p.bvh.qgrid + lane), ro_l);
                    q.ro[warp][lane] = lane == 0 ? px.ro.x : (lane == 1 ? px.ro.y : px.ro.z);
                    q.wo[warp][lane] = lane == 0 ? f.wo.x.v : (lane == 1 ? f.wo.y.v : f.wo.z.v);
                }
                gen_segment<MODE>(p, q, qr, px, f, warp, w0, w1, qn, lane);
            }
            if (lane == 0) { q.seg_cnt[warp] = qn; q.seg_head[warp] = 0; q.pixid[warp] = (int)mypx; }
            __syncthreads();
            // ================= phase T =================
            const bool replay = MODE == 1 && p.hit_in != nullptr;
            if (replay) {
                // backward with the forward pass's visibility record: no traversal at all
                if (has_px) {
                    if (lane < SEG / 32) {
                        const int wi_ = w0 / 32 + lane;
                        q.hitw[warp][lane] = wi_ < p.hit_words ? __ldg(p.hit_in + (size_t)mypx * p.hit_words + wi_) : 0u;
                    }
                    __syncwarp();
                    for (int e = lane; e < qn; e += 32) {
                        const int it = q.qitem[qb + e];
                        if ((q.hitw[warp][it >> 5] >> (it & 31)) & 1u) q.tex[qb + e] |= 0x80000000u;
                    }
                }
            } else if (trace_needed) trace_queue(p, q, warp, lane);      // sets tex bit 31 of occluded rays
            __syncthreads();
            if (MODE != 1 && p.hit_out != nullptr && has_px) {
                if (lane < SEG / 32) q.hitw[warp][lane] = 0u;
                __syncwarp();
                for (int e = lane; e < qn; e += 32)
                    if (q.tex[qb + e] >> 31) { const int it = q.qitem[qb + e]; atomicOr(&q.hitw[warp][it >> 5], 1u << (it & 31)); }
                __syncwarp();
                if (lane < SEG / 32) {
                    const int wi_ = w0 / 32 + lane;
                    if (wi_ < p.hit_words) p.hit_out[(size_t)mypx * p.hit_words + wi_] = q.hitw[warp][lane];
                }
            }
            // ================= phase E =================
            if (has_px) {
                if (MODE == 2) {
                    for (int e = lane; e < qn; e += 32) {
                        const size_t rec = (size_t)mypx * items + qr->slot[qb + e];
                        p.rec_vis[rec] = trace_needed ? (uint8_t)(1u - (q.tex[qb + e] >> 31)) : (uint8_t)2;
                    }
                }
                // dense list of entries with V != 0 (deterministic order)
                int vn = 0;
                for (int e0 = 0; e0 < qn; e0 += 32) {
                    const int e = e0 + lane;
                    const bool keep = e < qn && (!(q.tex[qb + e] >> 31) || v_occluded != 0.0f);
                    const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
                    if (keep) q.vlist[qb + vn + __popc(m & ((1u << lane) - 1u))] = (uint16_t)(qb + e);
                    vn += __popc(m);
                }
                __syncwarp();
                if (MODE != 1 && p.rec_count != nullptr) {
                    // ray record for the backward pass: exactly the rays evaluated below, in evaluation order
                    float *rr = p.rec_rays + (size_t)mypx * 5 * p.rec_slots;
                    for (int k = lane; k < vn; k += 32) {
                        const int e = q.vlist[qb + k];
                        rec_store(rr, p.rec_slots, rec_off + k, F3(q.dx[e], q.dy[e], q.dz[e]), q.mis[e], q.tex[e]);
                    }
                    rec_off += vn;
                    if (sub == nsub - 1 && lane == 0) p.rec_count[mypx] = (uint32_t)rec_off;
                }
                const PixelIn px = load_pixel(p, mypx);
                const f3 wo_f = F3(q.wo[warp][0], q.wo[warp][1], q.wo[warp][2]);
                f3 dgrad = F3(0.0f), sgrad = F3(0.0f);
                if (MODE == 1) { dgrad = p.diff_grad.ld3(px.iz, px.iy, px.ix); sgrad = p.spec_grad.ld3(px.iz, px.iy, px.ix); }

                for (int k = lane; k < vn; k += 32) {
                    const int e = q.vlist[qb + k];
                    const f3 wi = F3(q.dx[e], q.dy[e], q.dz[e]);
                    const uint32_t tex = q.tex[e];
                    const float wgt = ((tex >> 31) ? v_occluded : 1.0f) * q.mis[e] * sample_frac;
                    int tx, ty;
                    tex_unpack(tex, tx, ty);
                    if (MODE != 1) {
                        float diffv; f3 specv;
                        const f3 light_col = ray_eval(p, diffuse_only, px.kd, px.ks, wo_f, px.nrm, wi, tx, ty, diffv, specv);
                        accD += light_col * (diffv * wgt);
                        accS += specv * light_col * wgt;
                    } else ray_adjoint(p, diffuse_only, px.kd, px.ks, wo_f, px.nrm, dgrad, sgrad, wi, tx, ty, wgt, g_kd, g_ks, g_nrm, g_wo);
                }

                // ---- warp reduction, single writer per pixel (kernel.cu:442-456, 533-541) ----
                if (sub == nsub - 1) {
                    if (MODE != 1) {
                        float r0 = warp_sum(accD.x), r1 = warp_sum(accD.y), r2 = warp_sum(accD.z);
                        float r3 = warp_sum(accS.x), r4 = warp_sum(accS.y), r5 = warp_sum(accS.z);
                        if (lane == 0) {
                            float *d = p.diff + px.pix * 3, *s = p.spec + px.pix * 3;
                            d[0] = r0; d[1] = r1; d[2] = r2; s[0] = r3; s[1] = r4; s[2] = r5;
                        }
                    } else pixel_grad_write(p, px.pix, lane, px.pos, px.view, g_kd, g_ks, g_nrm, g_wo);
                }
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Backward from the forward pass's RAY RECORD: no sampling, no traversal -- per pixel the warp walks the recorded rays
// (direction, MIS weight, env texel, occluded flag) in the order the forward pass evaluated them and runs the adjoint BSDF
// + env-map gradient scatter (process_sample's backward branch, kernel.cu:422-457).  One warp per pixel, plain grid.
// ---------------------------------------------------------------------------------------------
struct ReplayParams {
    TView pos, nrm, view, kd, ks, diff_grad, spec_grad;
    const float *light; int l_s1, l_s2, l_s3; int Hl, Wl;
    const uint32_t *rec_count; const float *rec_rays; int rec_slots;
    int B, H, W;
    uint32_t bsdf; float shadow_scale, sample_frac;
    float *pos_grad, *nrm_grad, *kd_grad, *ks_grad, *light_grad;
};

__global__ void __launch_bounds__(256, REPLAY_MINB) env_shade_replay_kernel(const ReplayParams p)
{
    const int lane = threadIdx.x & 31;
    const int64_t npix = (int64_t)p.B * p.H * p.W;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const bool diffuse_only = (p.bsdf == 1u || p.bsdf == 2u);
    const float v_occluded = 1.0f - p.shadow_scale;
    for (int64_t chunk = warp_global; chunk * 32 < npix; chunk += nwarps) {
        const int64_t mypix = chunk * 32 + lane;
        const uint32_t mycnt = mypix < npix ? __ldg(p.rec_count + mypix) : 0u;
        unsigned rem = __ballot_sync(0xFFFFFFFFu, mycnt != 0u);
        if (mypix < npix && mycnt == 0u) pixel_grad_zero(p, mypix);
        while (rem) {
            const int src = __ffs(rem) - 1;
            rem &= rem - 1;
            const int64_t pix = chunk * 32 + src;
            const int cnt = (int)__shfl_sync(0xFFFFFFFFu, mycnt, src);
            const int ix = (int)(pix % p.W); const int64_t tt = pix / p.W; const int iy = (int)(tt % p.H), iz = (int)(tt / p.H);
            const f3 pos = p.pos.ld3(iz, iy, ix), nrm = p.nrm.ld3(iz, iy, ix), view = p.view.ld3(iz, iy, ix), kd = p.kd.ld3(iz, iy, ix), ks = p.ks.ld3(iz, iy, ix);
            const f3 dgrad = p.diff_grad.ld3(iz, iy, ix), sgrad = p.spec_grad.ld3(iz, iy, ix);
            const f3 wo_f = safe_normalize(view - pos);
            const float *rr = p.rec_rays + (size_t)pix * 5 * p.rec_slots;
            f3 g_kd = F3(0.0f), g_ks = F3(0.0f), g_nrm = F3(0.0f), g_wo = F3(0.0f);
            for (int k = lane; k < cnt; k += 32) {
                f3 wi; float mis; uint32_t tex;
                rec_load(rr, p.rec_slots, k, wi, mis, tex);
                const float wgt = ((tex >> 31) ? v_occluded : 1.0f) * mis * p.sample_frac;
                int tx, ty;
                tex_unpack(tex, tx, ty);
                ray_adjoint(p, diffuse_only, kd, ks, wo_f, nrm, dgrad, sgrad, wi, tx, ty, wgt, g_kd, g_ks, g_nrm, g_wo);
            }
            pixel_grad_write(p, pix, lane, pos, view, g_kd, g_ks, g_nrm, g_wo);
        }
    }
}

// LCG jump-ahead table: entry k = (mul, add) with  state_after_k_steps = state * mul + add  (kernel.cu:33 is one step).  Built on the
// device in one launch (thread k composes k steps by binary exponentiation of the affine map), cached per n_samples_x in the
// context: no host copy, no host synchronisation, capturable in a CUDA graph, and alternating n_samples_x between calls
// (training N=8 / validation N=32 style, train.py:303-305) does not rebuild anything.
__global__ void k_skip_table(uint2 *__restrict__ tab, int n)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    uint32_t m = 1u, a = 0u;                       // identity
    uint32_t bm = 747796405u, ba = 2891336453u;    // one step
    for (uint32_t e = (uint32_t)k; e; e >>= 1) {
        if (e & 1u) { a = a * bm + ba; m = m * bm; }            // apply `b` after the steps composed so far
        ba = ba * bm + ba; bm = bm * bm;                        // b <- b o b
    }
    tab[k] = make_uint2(m, a);
}

static int ensure_skip_table(mcs_ctx *c, int N, cudaStream_t s, const uint2 **out)
{
    for (int i = 0; i < c->n_skip; ++i)
        if (c->skip_N[i] == N) { *out = (const uint2 *)c->lcg_skip[i].p; return 0; }
    const int slot = c->n_skip < MCS_SKIP_TABLES ? c->n_skip : (c->skip_evict++ % MCS_SKIP_TABLES);
    const int n = 5 * N * N + 3;
    if (int e = mcs_buf_reserve(c->lcg_skip[slot], sizeof(uint2) * (size_t)n + 16, s)) return e;
    k_skip_table<<<(n + 255) / 256, 256, 0, s>>>((uint2 *)c->lcg_skip[slot].p, n);
    MCS_LAUNCH_CHECK();
    c->skip_N[slot] = N;
    if (c->n_skip < MCS_SKIP_TABLES) ++c->n_skip;
    *out = (const uint2 *)c->lcg_skip[slot].p;
    return 0;
}

static int cdf_iters(int size)
{
    // 4-ary search: each step shrinks the candidate interval [lo, hi] (span s -> at most s/4 + 1); run until it is a single index
    int steps = 0;
    for (int span = size - 1; span > 0; span = span / 4) ++steps;
    return steps + 1;
}

static int fill_params(mcs_ctx *ctx, EnvParams &p,
                       const mcs_tensor *mask, const mcs_tensor *ro, const mcs_tensor *gb_pos, const mcs_tensor *gb_normal,
                       const mcs_tensor *gb_view_pos, const mcs_tensor *gb_kd, const mcs_tensor *gb_ks,
                       const mcs_tensor *light, const mcs_tensor *pdf, const mcs_tensor *rows, const mcs_tensor *cols,
                       const mcs_tensor *perms, uint32_t bsdf, uint32_t n_samples_x, uint32_t rnd_seed, const uint32_t *seed_offset_dev, float shadow_scale, int32_t batch_offset,
                       cudaStream_t s)
{
    MCS_REQUIRE(ctx != nullptr, "env_shade: null context");
    MCS_REQUIRE(ctx->T > 0, "env_shade: no acceleration structure built (call optix_build_bvh first)");
    const mcs_tensor *all[] = {mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms};
    for (const mcs_tensor *t : all) MCS_REQUIRE(view_ok(t), "env_shade: null / empty tensor argument");
    MCS_REQUIRE(bsdf <= 2u, "env_shade: BSDF must be 0 ('pbr'), 1 ('diffuse') or 2 ('white')");
    MCS_REQUIRE(n_samples_x >= 1u && n_samples_x <= 64u, "env_shade: n_samples_x must be in [1, 64]");
    p.B = ro->sizes[0]; p.H = ro->sizes[1]; p.W = ro->sizes[2];
    MCS_REQUIRE(ro->sizes[3] == 3, "env_shade: ro must be [B,H,W,3]");
    MCS_REQUIRE((int64_t)p.B * p.H * p.W < (1ll << 31) / 3, "env_shade: launch too large for 32-bit indexing");
    const mcs_tensor *gb[] = {mask, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks};
    const char *gbn[] = {"mask", "gb_pos", "gb_normal", "gb_view_pos", "gb_kd", "gb_ks"};
    for (int i = 0; i < 6; ++i) {
        for (int d = 0; d < 3; ++d)
            MCS_REQUIRE(gb[i]->sizes[d] == ro->sizes[d] || gb[i]->sizes[d] == 1, "env_shade: %s dim %d = %d is not broadcastable to %d", gbn[i], d,
                        gb[i]->sizes[d], ro->sizes[d]);
        MCS_REQUIRE(gb[i]->sizes[3] == (i == 0 ? 1 : 3) || gb[i]->sizes[3] == 1, "env_shade: %s has a bad channel count %d", gbn[i], gb[i]->sizes[3]);
    }
    p.mask = make_view(mask); p.ro = make_view(ro); p.pos = make_view(gb_pos); p.nrm = make_view(gb_normal);
    p.view = make_view(gb_view_pos); p.kd = make_view(gb_kd); p.ks = make_view(gb_ks);
    p.Hl = light->sizes[1]; p.Wl = light->sizes[2];
    MCS_REQUIRE(light->sizes[3] == 3 && p.Hl >= 2 && p.Wl >= 2, "env_shade: light must be [Hl>=2, Wl>=2, 3]");
    MCS_REQUIRE(p.Hl < 32768 && p.Wl < 65536, "env_shade: light probe too large");
    MCS_REQUIRE(pdf->sizes[1] == p.Hl && pdf->sizes[2] == p.Wl && cols->sizes[1] == p.Hl && cols->sizes[2] == p.Wl && rows->sizes[1] == p.Hl,
                "env_shade: pdf / rows / cols do not match the light probe resolution");
    p.light = (const float *)light->ptr; p.l_s1 = light->strides[1]; p.l_s2 = light->strides[2]; p.l_s3 = light->strides[3];
    p.pdf = (const float *)pdf->ptr; p.p_s1 = pdf->strides[1]; p.p_s2 = pdf->strides[2];
    p.rows = (const float *)rows->ptr; p.r_s = rows->strides[1];
    p.cols = (const float *)cols->ptr; p.c_s1 = cols->strides[1]; p.c_s2 = cols->strides[2];
    p.N = (int)n_samples_x; p.S = p.N * p.N;
    p.hit_words = (2 * p.S + 31) / 32;
    MCS_REQUIRE(perms->sizes[3] == p.S && perms->sizes[1] >= 1, "env_shade: perms must be [P, n_samples_x^2]");
    p.perms = (const int32_t *)perms->ptr; p.pm_s1 = perms->strides[1]; p.pm_s3 = perms->strides[3]; p.n_perms = (uint32_t)perms->sizes[1];
    p.m_rows = cdf_iters(p.Hl); p.m_cols = cdf_iters(p.Wl);
    p.bsdf = bsdf; p.seed = rnd_seed; p.seed_dev = seed_offset_dev; p.batch_offset = batch_offset; p.shadow_scale = shadow_scale;
    p.bvh = BvhView{(const float4 *)ctx->nodes.p, (const float4 *)ctx->tris.p, (const float *)ctx->qgrid.p, (const uint4 *)ctx->nodesq4.p};
    if (int e = ensure_skip_table(ctx, p.N, s, &p.skip)) return e;
    // work-claim counter of the persistent grid: one slot of a small ring PER LAUNCH, so launches of the same context that are in
    // flight on different streams never share a counter
    if (int e = mcs_buf_reserve(ctx->counters, MCS_COUNTER_RING * 64, s)) return e;
    p.chunk_counter = (unsigned int *)((char *)ctx->counters.p + 64 * (size_t)(ctx->counter_next++ % MCS_COUNTER_RING));
    MCS_CUDA(cudaMemsetAsync(p.chunk_counter, 0, sizeof(unsigned int), s));
    return 0;
}

template <int MODE>
static int launch_env(const EnvParams &p, cudaStream_t s)
{
    int dev = 0, sms = 0, per_sm = 0;
    MCS_CUDA(cudaGetDevice(&dev));
    MCS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const size_t smem = sizeof(BlockQueue) + (MODE == 2 ? sizeof(BlockQueueRec) : 0);
    MCS_CUDA(cudaFuncSetAttribute(env_shade_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // Shared memory and L1 share 256 KB per SM and the carve-out comes in steps (..., 100, 132, 164, 196, 228 KB): ask for exactly what
    // 32 / NW resident CTAs need, so that everything else stays L1 for the BVH nodes, triangles and probe tables (36 KB per CTA => the
    // 164 KB step, 92 KB of L1).
    {
        const size_t need = (size_t)(32 / NW) * (smem + 1024);
        int pct = (int)((need * 100 + 228 * 1024 - 1) / (228 * 1024));
        MCS_CUDA(cudaFuncSetAttribute(env_shade_kernel<MODE>, cudaFuncAttributePreferredSharedMemoryCarveout, pct > 100 ? 100 : pct));
    }
    MCS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, env_shade_kernel<MODE>, NW * 32, smem));
    if (per_sm < 1) per_sm = 1;
    const int64_t npix = (int64_t)p.B * p.H * p.W;
    int64_t want = (npix + 32 * NW - 1) / (32 * NW);
    int grid = (int)(want < (int64_t)sms * per_sm ? want : (int64_t)sms * per_sm);
    if (grid < 1) grid = 1;
    env_shade_kernel<MODE><<<grid, NW * 32, smem, s>>>(p);
    MCS_LAUNCH_CHECK();
    return 0;
}

}  // namespace

extern "C" {

int mcs_env_shade_fwd(mcs_ctx *ctx,
                      const mcs_tensor *mask, const mcs_tensor *ro, const mcs_tensor *gb_pos, const mcs_tensor *gb_normal,
                      const mcs_tensor *gb_view_pos, const mcs_tensor *gb_kd, const mcs_tensor *gb_ks,
                      const mcs_tensor *light, const mcs_tensor *pdf, const mcs_tensor *rows, const mcs_tensor *cols,
                      const mcs_tensor *perms,
                      uint32_t bsdf, uint32_t n_samples_x, uint32_t rnd_seed, const uint32_t *seed_offset_dev, float shadow_scale, int32_t batch_offset,
                      float *diff, float *spec, uint32_t *hit_record, uint32_t *rec_count, float *rec_rays, int32_t rec_slots, mcs_stream stream)
{
    EnvParams p{};
    cudaStream_t s = (cudaStream_t)stream;
    if (int e = fill_params(ctx, p, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms, bsdf, n_samples_x, rnd_seed,
                            seed_offset_dev, shadow_scale, batch_offset, s)) return e;
    MCS_REQUIRE(diff && spec, "env_shade_fwd: null output pointer");
    p.diff = diff; p.spec = spec; p.hit_out = hit_record;
    MCS_REQUIRE((rec_count == nullptr) == (rec_rays == nullptr), "env_shade_fwd: rec_count and rec_rays go together");
    MCS_REQUIRE(rec_count == nullptr || rec_slots >= 2 * p.S, "env_shade_fwd: rec_slots must be >= 2 * n_samples_x^2");
    p.rec_count = rec_count; p.rec_rays = rec_rays; p.rec_slots = rec_slots;
    return launch_env<0>(p, s);
}

int mcs_env_shade_records(mcs_ctx *ctx,
                          const mcs_tensor *mask, const mcs_tensor *ro, const mcs_tensor *gb_pos, const mcs_tensor *gb_normal,
                          const mcs_tensor *gb_view_pos, const mcs_tensor *gb_kd, const mcs_tensor *gb_ks,
                          const mcs_tensor *light, const mcs_tensor *pdf, const mcs_tensor *rows, const mcs_tensor *cols,
                          const mcs_tensor *perms,
                          uint32_t bsdf, uint32_t n_samples_x, uint32_t rnd_seed, const uint32_t *seed_offset_dev, float shadow_scale, int32_t batch_offset,
                          float *diff, float *spec, int32_t *rec_texel, uint8_t *rec_vis, mcs_stream stream)
{
    EnvParams p{};
    cudaStream_t s = (cudaStream_t)stream;
    if (int e = fill_params(ctx, p, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms, bsdf, n_samples_x, rnd_seed,
                            seed_offset_dev, shadow_scale, batch_offset, s)) return e;
    MCS_REQUIRE(diff && spec && rec_texel && rec_vis, "env_shade_records: null output pointer");
    p.diff = diff; p.spec = spec; p.rec_texel = rec_texel; p.rec_vis = rec_vis;
    return launch_env<2>(p, s);
}

int mcs_env_shade_bwd(mcs_ctx *ctx,
                      const mcs_tensor *mask, const mcs_tensor *ro, const mcs_tensor *gb_pos, const mcs_tensor *gb_normal,
                      const mcs_tensor *gb_view_pos, const mcs_tensor *gb_kd, const mcs_tensor *gb_ks,
                      const mcs_tensor *light, const mcs_tensor *pdf, const mcs_tensor *rows, const mcs_tensor *cols,
                      const mcs_tensor *perms,
                      uint32_t bsdf, uint32_t n_samples_x, uint32_t rnd_seed, const uint32_t *seed_offset_dev, float shadow_scale, int32_t batch_offset,
                      const mcs_tensor *diff_grad, const mcs_tensor *spec_grad,
                      float *gb_pos_grad, float *gb_normal_grad, float *gb_kd_grad, float *gb_ks_grad, float *light_grad,
                      const uint32_t *hit_record, mcs_stream stream)
{
    EnvParams p{};
    cudaStream_t s = (cudaStream_t)stream;
    if (int e = fill_params(ctx, p, mask, ro, gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, pdf, rows, cols, perms, bsdf, n_samples_x, rnd_seed,
                            seed_offset_dev, shadow_scale, batch_offset, s)) return e;
    MCS_REQUIRE(view_ok(diff_grad) && view_ok(spec_grad), "env_shade_bwd: null / empty upstream gradient");
    MCS_REQUIRE(gb_pos_grad && gb_normal_grad && gb_kd_grad && gb_ks_grad && light_grad, "env_shade_bwd: null output pointer");
    for (int d = 0; d < 3; ++d)
        MCS_REQUIRE(diff_grad->sizes[d] == ro->sizes[d] && spec_grad->sizes[d] == ro->sizes[d], "env_shade_bwd: upstream gradient shape mismatch");
    p.diff_grad = make_view(diff_grad); p.spec_grad = make_view(spec_grad);
    p.pos_grad = gb_pos_grad; p.nrm_grad = gb_normal_grad; p.kd_grad = gb_kd_grad; p.ks_grad = gb_ks_grad; p.light_grad = light_grad;
    p.hit_in = hit_record;
    MCS_CUDA(cudaMemsetAsync(light_grad, 0, sizeof(float) * 3 * (size_t)p.Hl * p.Wl, s));
    return launch_env<1>(p, s);
}

int mcs_env_shade_bwd_replay(const mcs_tensor *gb_pos, const mcs_tensor *gb_normal, const mcs_tensor *gb_view_pos, const mcs_tensor *gb_kd,
                             const mcs_tensor *gb_ks, const mcs_tensor *light, uint32_t bsdf, uint32_t n_samples_x, float shadow_scale,
                             const mcs_tensor *diff_grad, const mcs_tensor *spec_grad, const uint32_t *rec_count, const float *rec_rays, int32_t rec_slots,
                             float *gb_pos_grad, float *gb_normal_grad, float *gb_kd_grad, float *gb_ks_grad, float *light_grad, mcs_stream stream)
{
    cudaStream_t s = (cudaStream_t)stream;
    const mcs_tensor *all[] = {gb_pos, gb_normal, gb_view_pos, gb_kd, gb_ks, light, diff_grad, spec_grad};
    for (const mcs_tensor *t : all) MCS_REQUIRE(view_ok(t), "env_shade_bwd_replay: null / empty tensor argument");
    MCS_REQUIRE(rec_count && rec_rays && rec_slots > 0, "env_shade_bwd_replay: missing ray record");
    MCS_REQUIRE(gb_pos_grad && gb_normal_grad && gb_kd_grad && gb_ks_grad && light_grad, "env_shade_bwd_replay: null output pointer");
    MCS_REQUIRE(bsdf <= 2u && n_samples_x >= 1u, "env_shade_bwd_replay: bad bsdf / n_samples_x");
    ReplayParams p{};
    p.B = diff_grad->sizes[0]; p.H = diff_grad->sizes[1]; p.W = diff_grad->sizes[2];
    p.pos = make_view(gb_pos); p.nrm = make_view(gb_normal); p.view = make_view(gb_view_pos); p.kd = make_view(gb_kd); p.ks = make_view(gb_ks);
    p.diff_grad = make_view(diff_grad); p.spec_grad = make_view(spec_grad);
    p.Hl = light->sizes[1]; p.Wl = light->sizes[2];
    p.light = (const float *)light->ptr; p.l_s1 = light->strides[1]; p.l_s2 = light->strides[2]; p.l_s3 = light->strides[3];
    p.rec_count = rec_count; p.rec_rays = rec_rays; p.rec_slots = rec_slots;
    p.bsdf = bsdf; p.shadow_scale = shadow_scale;
    p.sample_frac = 1.0f / (float)(n_samples_x * n_samples_x);
    p.pos_grad = gb_pos_grad; p.nrm_grad = gb_normal_grad; p.kd_grad = gb_kd_grad; p.ks_grad = gb_ks_grad; p.light_grad = light_grad;
    MCS_CUDA(cudaMemsetAsync(light_grad, 0, sizeof(float) * 3 * (size_t)p.Hl * p.Wl, s));
    int dev = 0, sms = 0;
    MCS_CUDA(cudaGetDevice(&dev));
    MCS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t npix = (int64_t)p.B * p.H * p.W;
    int64_t want = (npix + 255) / 256;
    int grid = (int)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);
    if (grid < 1) grid = 1;
    env_shade_replay_kernel<<<grid, 256, 0, s>>>(p);
    MCS_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
