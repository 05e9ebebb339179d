// denoise.cu -- cross-bilateral (SVGF-style) denoiser, forward and transposed backward, for sm_100a.
// Replaces bilateral_denoiser_fwd_kernel / _bwd_kernel, render/optixutils/c_src/denoising.cu:14-130
// (8x8 blocks, every tap re-fetched from global memory with 2 expf + powf(.,128) + sqrtf per tap).
//
// B200 design (compute-bound: (2r+1)^2 = 529 taps/px at sigma = 2, only 48 B/px of compulsory HBM
// traffic, SURVEY.md section 8d):
//   * one CTA = 32x16 output pixels, the (32+2r)x(16+2r) halo tile of guides (normal, depth,
//     depth-gradient) and signals staged ONCE in shared memory: by the TMA unit as AoS tiles when the operands are contiguous
//     (bilateral_tma_kernel below: the path render.shade()'s fused tail and bench.py take), else by plain loads as SoA planes
//     (bilateral_kernel: strided channel slices; conflict-free: a warp reads 32 consecutive floats of a plane row);
//     both kernels then run the same filter, bilateral_core, which reads the tile through a per-layout accessor
//     (PlaneTile / AosTile), so the two paths give bit-identical results;
//   * each thread produces two vertically adjacent outputs so every tap value read from shared
//     memory is used twice (halves LDS traffic, the co-limiter next to the FP32/MUFU pipes);
//   * the spatial gaussian exponent is one FMA on a running tap offset; gaussian and depth term are merged into ONE
//     ex2.approx (exp(a)*exp(b) = exp2((a+b)*log2 e)); 1/max(dz*dist, eps) = min(inv_dz * rsqrt(dist^2), 1/eps) with the
//     guarded 1/dz staged per pixel; pow(x,128) is 7 squarings -- 2 MUFU and no table look-up per tap;
//   * out-of-image taps are stored as zero normals => clamp(dot, 1e-4, 1)^128 underflows to exactly
//     0, which reproduces the reference's `continue` without a branch;
//   * the diffuse and specular signals, which render.py:120-121 filters with identical guides, can
//     share one pass (NSIG = 2): weights are computed once.
#include "common.cuh"
#include <cuda.h>          // CUtensorMap + the cuTensorMapEncodeTiled prototype (resolved at run time through cudaGetDriverEntryPoint: no libcuda link)

namespace {

constexpr int TILE_W = 32;
constexpr int TILE_H = 16;
constexpr float FLT_EPS_ = 0.0001f;      // denoising.cu:12
constexpr float LOG2E = 1.4426950408889634f;

struct BilateralParams {
    TView nrm, zdz;
    TView sig[2];          // fwd: col ; bwd: out_grad (first 3 channels used)
    float *out[2];         // fwd: [B,H,W,4] ; bwd: [B,H,W,3]
    int B, H, W;
    int r;
    float neg_inv_2var_log2e;   // -log2(e) / (2 sigma^2)
};

// MUFU approximations without the range-handling wrappers of exp2f / __fdividef (their operands are bounded here: exponents
// <= 0, where a flushed denormal weight is indistinguishable from the reference's 1e-38; reciprocal arguments >= 1e-4)
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rsqrt_approx(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// 1 / max(dz * dist, 1e-4) = min(inv_dz * rsqrt(dist^2), 1e4) with inv_dz = dz > 0 ? 1/dz : +inf  (dist = 0 -> inf -> 1e4 as well)
__device__ __forceinline__ float guarded_inv(float dz) { return dz > 0.0f ? 1.0f / dz : INFINITY; }

__device__ __forceinline__ float pow128(float x)
{
    x *= x; x *= x; x *= x; x *= x; x *= x; x *= x; x *= x;
    return x;
}

// ---------------------------------------------------------------------------------------------
// The filter after staging, shared by both kernels.  Tile is the staged halo tile's accessor:
//   r                 filter radius the tile was staged for;
//   centre(lx, ly)    tile index of output (lx, ly) of the CTA;
//   row(lx, ty)       tile index of tile row ty at the first tap column of output column lx's window;
//   normal(i)         tap normal;
//   centre_depth(i)   (depth, guarded 1/dz) of a centre pixel;
//   tap_depth(i)      (depth, guarded 1/dz) of a tap; the forward pass weighs with the centre's dz and gets 0 for the second;
//   signal(s, i)      signal s (colour or upstream gradient, 3 channels).
// Params supplies neg_inv_2var_log2e, out[], H and W.
// ---------------------------------------------------------------------------------------------
template <int NSIG, bool BWD, class Tile, class Params>
__device__ __forceinline__ void bilateral_core(const Tile &t, const Params &p)
{
    const int r = t.r;
    const int b = blockIdx.z;
    // two vertically adjacent outputs per thread: rows 2*ty and 2*ty+1 of the tile
    const int lx = threadIdx.x, lyA = 2 * threadIdx.y;
    f3 cn[2]; float cz[2], cdz[2];
#pragma unroll
    for (int o = 0; o < 2; ++o) {
        const int ci = t.centre(lx, lyA + o);
        cn[o] = t.normal(ci);
        const float2 c = t.centre_depth(ci);
        cz[o] = c.x; cdz[o] = c.y;      // cdz = guarded 1/dz of the centre
    }
    float acc[2][NSIG][3]; float accw[2] = {0.0f, 0.0f};
#pragma unroll
    for (int o = 0; o < 2; ++o)
#pragma unroll
        for (int s = 0; s < NSIG; ++s) acc[o][s][0] = acc[o][s][1] = acc[o][s][2] = 0.0f;

    const float k2 = p.neg_inv_2var_log2e;
    for (int rr = 0; rr <= 2 * r + 1; ++rr) {
        // tap row rr of the tile serves output A at vertical offset rr - r and output B at rr - r - 1; a row outside an output's
        // window gets exponent -inf (weight exactly 0)
        const float fyA = (float)(rr - r), fyB = (float)(rr - r - 1);
        const float fy2[2] = {fyA * fyA, fyB * fyB};
        const float gy[2] = {rr <= 2 * r ? fy2[0] * k2 : -INFINITY, rr >= 1 ? fy2[1] * k2 : -INFINITY};
        const int rowoff = t.row(lx, lyA + rr);
        float fx = (float)(-r);
        for (int cx = 0; cx <= 2 * r; ++cx, fx += 1.0f) {
            const int i = rowoff + cx;
            const float fx2 = fx * fx;
            const f3 tn = t.normal(i);
            const float2 td = t.tap_depth(i);
            const float tz = td.x, tinv = td.y;
            float sg[NSIG][3];
#pragma unroll
            for (int s = 0; s < NSIG; ++s) {
                const f3 v = t.signal(s, i);
                sg[s][0] = v.x; sg[s][1] = v.y; sg[s][2] = v.z;
            }
#pragma unroll
            for (int o = 0; o < 2; ++o) {
                const float wn = pow128(fminf(fmaxf(dot(tn, cn[o]), FLT_EPS_), 1.0f));
                // fwd: centre's dz (denoising.cu:59); bwd: tap's dz (denoising.cu:118)
                const float inv_den = fminf((BWD ? tinv : cdz[o]) * rsqrt_approx(fx2 + fy2[o]), 1.0f / FLT_EPS_);
                const float e = fmaf(fx2, k2, gy[o]) - LOG2E * (fabsf(tz - cz[o]) * inv_den);
                const float w = wn * ex2_approx(e);
#pragma unroll
                for (int s = 0; s < NSIG; ++s) {
                    acc[o][s][0] = fmaf(sg[s][0], w, acc[o][s][0]);
                    acc[o][s][1] = fmaf(sg[s][1], w, acc[o][s][1]);
                    acc[o][s][2] = fmaf(sg[s][2], w, acc[o][s][2]);
                }
                accw[o] += w;
            }
        }
    }

    const int gx = blockIdx.x * TILE_W + lx;
#pragma unroll
    for (int o = 0; o < 2; ++o) {
        const int gy = blockIdx.y * TILE_H + lyA + o;
        if (gx < p.W && gy < p.H) {
            const int64_t px = ((int64_t)b * p.H + gy) * p.W + gx;
#pragma unroll
            for (int s = 0; s < NSIG; ++s) {
                if (!BWD) reinterpret_cast<float4 *>(p.out[s])[px] = make_float4(acc[o][s][0], acc[o][s][1], acc[o][s][2], fmaxf(accw[o], 0.0001f));
                else { float *d = p.out[s] + px * 3; d[0] = acc[o][s][0]; d[1] = acc[o][s][1]; d[2] = acc[o][s][2]; }
            }
        }
    }
}

// SoA planes of pitch TILE_W + 2r; the 1/dz plane already holds the guarded reciprocal.
template <bool BWD>
struct PlaneTile {
    const float *nx, *ny, *nz, *z, *inv_dz, *sig;      // sig: NSIG * 3 planes
    int plane, pitch, r;
    __device__ __forceinline__ int centre(int lx, int ly) const { return lx + r + (ly + r) * pitch; }
    __device__ __forceinline__ int row(int lx, int ty) const { return ty * pitch + lx; }
    __device__ __forceinline__ f3 normal(int i) const { return F3(nx[i], ny[i], nz[i]); }
    __device__ __forceinline__ float2 centre_depth(int i) const { return make_float2(z[i], inv_dz[i]); }
    __device__ __forceinline__ float2 tap_depth(int i) const { return make_float2(z[i], BWD ? inv_dz[i] : 0.0f); }
    __device__ __forceinline__ f3 signal(int s, int i) const { return F3(sig[(3 * s + 0) * plane + i], sig[(3 * s + 1) * plane + i], sig[(3 * s + 2) * plane + i]); }
};

template <int NSIG, bool BWD>
__global__ void __launch_bounds__(256) bilateral_kernel(BilateralParams p)
{
    extern __shared__ float smem[];
    const int r = p.r;
    const int tw = TILE_W + 2 * r, th = TILE_H + 2 * r;
    const int plane = tw * th;
    float *s_nx = smem, *s_ny = s_nx + plane, *s_nz = s_ny + plane, *s_z = s_nz + plane, *s_dz = s_z + plane;
    float *s_sig = s_dz + plane;                       // NSIG * 3 planes

    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * TILE_W - r, y0 = blockIdx.y * TILE_H - r;

    for (int i = tid; i < plane; i += 256) {
        int ty = i / tw, tx = i - ty * tw;
        int gy = y0 + ty, gx = x0 + tx;
        bool in = gy >= 0 && gx >= 0 && gy < p.H && gx < p.W;
        f3 n = F3(0.0f); float z = 0.0f, dz = 0.0f;
        if (in) {
            n = p.nrm.ld3(b, gy, gx);
            const float *q = p.zdz.p + p.zdz.off(b, gy, gx);
            z = __ldg(q); dz = __ldg(q + p.zdz.s3);
        }
        s_nx[i] = n.x; s_ny[i] = n.y; s_nz[i] = n.z; s_z[i] = z; s_dz[i] = guarded_inv(dz);     // plane holds 1/dz (guarded)
#pragma unroll
        for (int s = 0; s < NSIG; ++s) {
            f3 c = F3(0.0f);
            if (in) c = p.sig[s].ld3(b, gy, gx);
            s_sig[(3 * s + 0) * plane + i] = c.x; s_sig[(3 * s + 1) * plane + i] = c.y; s_sig[(3 * s + 2) * plane + i] = c.z;
        }
    }
    __syncthreads();
    bilateral_core<NSIG, BWD>(PlaneTile<BWD>{s_nx, s_ny, s_nz, s_z, s_dz, s_sig, plane, tw, r}, p);
}

// ---------------------------------------------------------------------------------------------
// Halo tile staged by the TMA unit (north_star: "the bilateral denoiser is a TMA-staged tiled kernel").
// Applies when the signals and the normals are contiguous [B,H,W,3] fp32 and zdz contiguous [B,H,W,2] with 16-byte aligned bases and
// W % 4 == 0 -- the layout render.shade()'s fused tail (ou.denoise_and_combine) and bench.py hand over; strided channel slices of an
// 8-channel tensor (the reference's BilateralDenoiser.forward) have 12-byte pixel pitches that a tensor map cannot describe and
// take bilateral_kernel.  Each operand is a 3-D tensor (W * C floats, H, B); ONE thread issues one `cp.async.bulk.tensor.3d` (SASS
// UTMALDG) per operand for the box (TWP * C, TILE_H + 2r, 1) at (x0 * C, y0, b) with x0 = tile origin - (r rounded up to 4 pixels) so that
// the box starts on a 16-byte boundary, completion counted in bytes on an mbarrier.
// Out-of-image coordinates -- negative ones included -- are ZERO-FILLED by the copy engine: a zero normal makes the tap weight
// underflow to exactly 0, which is the reference's `continue` (denoising.cu:43), so the staging loop's bounds checks, index
// arithmetic and strided loads disappear.  Tiles stay AoS in shared memory: lane x reads word 3 x + c (stride 3: conflict-free);
// the backward pass reads (depth, depth gradient) pairs with one 64-bit load after dz has been replaced by its guarded reciprocal
// in place, and its [B,H,W,4] upstream gradients with one 128-bit shared load per tap and signal.
// The filter itself is bilateral_core, the one bilateral_kernel runs, read through AosTile.
// ---------------------------------------------------------------------------------------------
struct BilateralTmaParams {
    float *out[2];
    int B, H, W, r, twp;
    int rl;                  // left halo of the staged tile = r rounded up to a multiple of 4 pixels: the box must START on a 16-byte boundary
                             // in global memory (a start at -r pixels x 12 bytes raised "illegal instruction" on the B200; measured)
    float neg_inv_2var_log2e;
};

// AoS tiles of pitch twp pixels with a left halo of rl >= r pixels: normals (stride 3), (z, dz) pairs (stride 2; backward: dz already
// replaced by its guarded reciprocal), signals (stride 3 forward, 4 backward), and in the forward a de-interleaved depth plane z.
template <bool BWD>
struct AosTile {
    const float *n, *zd, *z, *sig;
    int ns, pitch, r, rl;
    __device__ __forceinline__ int centre(int lx, int ly) const { return (ly + r) * pitch + lx + rl; }
    __device__ __forceinline__ int row(int lx, int ty) const { return ty * pitch + lx + (rl - r); }
    __device__ __forceinline__ f3 normal(int i) const { return F3(n[3 * i], n[3 * i + 1], n[3 * i + 2]); }
    __device__ __forceinline__ float2 centre_depth(int i) const { return make_float2(zd[2 * i], BWD ? zd[2 * i + 1] : guarded_inv(zd[2 * i + 1])); }
    __device__ __forceinline__ float2 tap_depth(int i) const { return BWD ? reinterpret_cast<const float2 *>(zd)[i] : make_float2(z[i], 0.0f); }
    __device__ __forceinline__ f3 signal(int s, int i) const
    {
        if (BWD) {      // one 128-bit shared load per signal (16-byte pixels: conflict-free)
            const float4 g4 = reinterpret_cast<const float4 *>(sig + s * ns)[i];
            return F3(g4.x, g4.y, g4.z);
        }
        return F3(sig[s * ns + 3 * i], sig[s * ns + 3 * i + 1], sig[s * ns + 3 * i + 2]);
    }
};

__device__ __forceinline__ uint32_t dn_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, int c0, int c1, int c2, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dn_smem_u32(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(dn_smem_u32(bar))
                 : "memory");
}

template <int NSIG, bool BWD>
__global__ void __launch_bounds__(256) bilateral_tma_kernel(const __grid_constant__ CUtensorMap m_nrm, const __grid_constant__ CUtensorMap m_zdz,
                                                                const __grid_constant__ CUtensorMap m_sigA, const __grid_constant__ CUtensorMap m_sigB,
                                                                BilateralTmaParams p)
{
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t bar;
    const int r = p.r, twp = p.twp, th = TILE_H + 2 * r;
    constexpr int CS = BWD ? 4 : 3;                 // forward: colour [.,3]; backward: out_grad [.,4] (weight channel unused, denoising.cu:122)
    const int n3 = (twp * 3 * th + 31) & ~31, n2 = (twp * 2 * th + 31) & ~31;    // 128-byte aligned sections
    const int ns = (twp * CS * th + 31) & ~31;
    float *s_n = smem, *s_zd = s_n + n3, *s_sig = s_zd + n2, *s_z = s_sig + NSIG * ns;     // s_z: forward only (depth plane)
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * TILE_W - p.rl, y0 = blockIdx.y * TILE_H - r;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(dn_smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t bytes = (uint32_t)(sizeof(float) * (size_t)twp * th * (3 + 2 + CS * NSIG));
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(dn_smem_u32(&bar)), "r"(bytes) : "memory");
        tma_load_3d(s_n, &m_nrm, x0 * 3, y0, b, &bar);
        tma_load_3d(s_zd, &m_zdz, x0 * 2, y0, b, &bar);
        tma_load_3d(s_sig, &m_sigA, x0 * CS, y0, b, &bar);
        if (NSIG == 2) tma_load_3d(s_sig + ns, &m_sigB, x0 * CS, y0, b, &bar);
    }
    __syncthreads();
    asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}" ::"r"(dn_smem_u32(&bar)) : "memory");
    // (z, dz) -> (z, guarded 1/dz) in place; the tap loop reads the pair with one 64-bit shared load (8-byte pixels: conflict-free)
    // the forward pass only needs the tap's depth: a de-interleaved plane (one 32-bit load; measured 1.41 vs 1.50 ms against the pair load)
    for (int i = tid; i < twp * th; i += 256) {
        if (BWD) s_zd[2 * i + 1] = guarded_inv(s_zd[2 * i + 1]);
        else s_z[i] = s_zd[2 * i];
    }
    __syncthreads();
    bilateral_core<NSIG, BWD>(AosTile<BWD>{s_n, s_zd, s_z, s_sig, ns, twp, r, p.rl}, p);
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                    const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_tiled_fn tma_encoder()
{
    static encode_tiled_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (encode_tiled_fn)ptr;
    }
    return fn;
}

// contiguous [B,H,W,C] fp32, 16-byte aligned base and row pitch
static bool tma_ok(const mcs_tensor *t, int C)
{
    return t->sizes[3] == C && t->strides[3] == 1 && t->strides[2] == C && t->strides[1] == C * t->sizes[2] && t->strides[0] == C * t->sizes[2] * t->sizes[1] &&
           ((uintptr_t)t->ptr % 16 == 0) && ((size_t)t->sizes[2] * C * sizeof(float)) % 16 == 0;
}

static bool tma_encode(CUtensorMap *m, const mcs_tensor *t, int C, int twp, int th)
{
    const cuuint64_t dims[3] = {(cuuint64_t)t->sizes[2] * C, (cuuint64_t)t->sizes[1], (cuuint64_t)t->sizes[0]};
    const cuuint64_t strides[2] = {(cuuint64_t)t->sizes[2] * C * sizeof(float), (cuuint64_t)t->sizes[2] * C * sizeof(float) * t->sizes[1]};
    const cuuint32_t box[3] = {(cuuint32_t)(twp * C), (cuuint32_t)th, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return tma_encoder()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void *>(t->ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct FilterGeometry {
    int r;                      // denoising.cu:28 filter_rad
    float neg_inv_2var_log2e;   // -log2(e) / (2 sigma^2)
};

static FilterGeometry filter_geometry(float sigma) { return {2 * (int)ceilf(sigma * 2.5f) + 1, -LOG2E / (2.0f * sigma * sigma)}; }

// returns 0 = launched, 1 = not applicable (caller takes the plain kernel), 2 = CUDA error (message set)
template <int NSIG, bool BWD>
static int launch_bilateral_tma(const mcs_tensor *nrm, const mcs_tensor *zdz, const mcs_tensor *const (&sig)[NSIG], float *const (&out)[NSIG], float sigma,
                                cudaStream_t stream)
{
    constexpr int CS = BWD ? 4 : 3;
    if (tma_encoder() == nullptr) return 1;
    if (!(tma_ok(nrm, 3) && tma_ok(zdz, 2) && tma_ok(sig[0], CS) && tma_ok(sig[NSIG - 1], CS))) return 1;
    const FilterGeometry g = filter_geometry(sigma);
    BilateralTmaParams p{};
    p.r = g.r;
    p.neg_inv_2var_log2e = g.neg_inv_2var_log2e;
    p.B = nrm->sizes[0]; p.H = nrm->sizes[1]; p.W = nrm->sizes[2];
    p.rl = (p.r + 3) & ~3;
    const int th = TILE_H + 2 * p.r;
    p.twp = (TILE_W + p.rl + p.r + 3) & ~3;
    if (p.twp * CS > 256 || th > 256) return 1;                                  // tensor-map box extents are limited to 256 elements
    for (int s = 0; s < NSIG; ++s) p.out[s] = out[s];
    const size_t n3 = ((size_t)p.twp * 3 * th + 31) & ~(size_t)31, n2 = ((size_t)p.twp * 2 * th + 31) & ~(size_t)31, n1 = ((size_t)p.twp * th + 31) & ~(size_t)31;
    const size_t ns = ((size_t)p.twp * CS * th + 31) & ~(size_t)31;
    const size_t smem = sizeof(float) * (n3 + n2 + NSIG * ns + (BWD ? 0 : n1));
    if (smem > 227 * 1024) return 1;
    CUtensorMap mn, mz, ma, mb;      // one signal: m_sigB is never read, encode it from the first signal
    if (!tma_encode(&mn, nrm, 3, p.twp, th) || !tma_encode(&mz, zdz, 2, p.twp, th) || !tma_encode(&ma, sig[0], CS, p.twp, th) ||
        !tma_encode(&mb, sig[NSIG - 1], CS, p.twp, th))
        return 1;
    auto kern = bilateral_tma_kernel<NSIG, BWD>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { mcs_set_error("bilateral (TMA): cudaFuncSetAttribute failed"); return 2; }
    dim3 grid((p.W + TILE_W - 1) / TILE_W, (p.H + TILE_H - 1) / TILE_H, p.B), block(32, 8, 1);
    kern<<<grid, block, smem, stream>>>(mn, mz, ma, mb, p);
    if (cudaGetLastError() != cudaSuccess) { mcs_set_error("bilateral (TMA): launch failed"); return 2; }
    return 0;
}

template <int NSIG, bool BWD>
static int launch_bilateral(const mcs_tensor *nrm, const mcs_tensor *zdz, const mcs_tensor *const (&sig)[NSIG], float *const (&out)[NSIG], float sigma,
                            cudaStream_t stream)
{
    const FilterGeometry g = filter_geometry(sigma);
    BilateralParams p{};
    p.nrm = make_view(nrm); p.zdz = make_view(zdz);
    for (int s = 0; s < NSIG; ++s) { p.sig[s] = make_view(sig[s]); p.out[s] = out[s]; }
    p.B = nrm->sizes[0]; p.H = nrm->sizes[1]; p.W = nrm->sizes[2];
    p.r = g.r;
    p.neg_inv_2var_log2e = g.neg_inv_2var_log2e;
    int tw = TILE_W + 2 * p.r, th = TILE_H + 2 * p.r;
    size_t smem = sizeof(float) * ((size_t)(5 + 3 * NSIG) * tw * th);
    MCS_REQUIRE(smem <= 227 * 1024, "bilateral: sigma %.3f needs a %zu-byte tile (> 227 KB shared memory)", sigma, smem);
    auto kern = bilateral_kernel<NSIG, BWD>;
    MCS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((p.W + TILE_W - 1) / TILE_W, (p.H + TILE_H - 1) / TILE_H, p.B), block(32, 8, 1);
    kern<<<grid, block, smem, stream>>>(p);
    MCS_LAUNCH_CHECK();
    return 0;
}

static int check_guides(const mcs_tensor *nrm, const mcs_tensor *zdz, const mcs_tensor *sig, int sig_c, const char *sig_name)
{
    MCS_REQUIRE(view_ok(nrm) && view_ok(zdz) && view_ok(sig), "bilateral: null / empty tensor argument");
    MCS_REQUIRE(nrm->sizes[3] == 3, "bilateral: nrm must have 3 channels");
    MCS_REQUIRE(zdz->sizes[3] == 2, "bilateral: zdz must have 2 channels");
    MCS_REQUIRE(sig->sizes[3] == sig_c, "bilateral: %s must have %d channels", sig_name, sig_c);
    for (int d = 0; d < 3; ++d)
        MCS_REQUIRE(nrm->sizes[d] == sig->sizes[d] && zdz->sizes[d] == sig->sizes[d], "bilateral: shape mismatch in dim %d", d);
    return 0;
}

// Every entry point: validate, then the TMA-staged kernel if the operands allow it, else the plain one.
template <int NSIG, bool BWD>
static int bilateral(const mcs_tensor *nrm, const mcs_tensor *zdz, const mcs_tensor *const (&sig)[NSIG], const char *const (&sig_name)[NSIG],
                     float *const (&out)[NSIG], float sigma, mcs_stream stream)
{
    for (int s = 0; s < NSIG; ++s)
        if (int e = check_guides(nrm, zdz, sig[s], BWD ? 4 : 3, sig_name[s])) return e;
    MCS_REQUIRE(sigma > 0.0f, "bilateral: sigma must be > 0");
    const int t = launch_bilateral_tma<NSIG, BWD>(nrm, zdz, sig, out, sigma, (cudaStream_t)stream);
    if (t != 1) return t;
    return launch_bilateral<NSIG, BWD>(nrm, zdz, sig, out, sigma, (cudaStream_t)stream);
}

}  // namespace

extern "C" {

int mcs_bilateral_fwd(const mcs_tensor *col, const mcs_tensor *nrm, const mcs_tensor *zdz, float sigma, float *out, mcs_stream stream)
{
    return bilateral<1, false>(nrm, zdz, {col}, {"col"}, {out}, sigma, stream);
}

int mcs_bilateral_bwd(const mcs_tensor *nrm, const mcs_tensor *zdz, float sigma, const mcs_tensor *out_grad, float *col_grad, mcs_stream stream)
{
    return bilateral<1, true>(nrm, zdz, {out_grad}, {"out_grad"}, {col_grad}, sigma, stream);
}

int mcs_bilateral_fwd2(const mcs_tensor *colA, const mcs_tensor *colB, const mcs_tensor *nrm, const mcs_tensor *zdz, float sigma,
                       float *outA, float *outB, mcs_stream stream)
{
    return bilateral<2, false>(nrm, zdz, {colA, colB}, {"colA", "colB"}, {outA, outB}, sigma, stream);
}

int mcs_bilateral_bwd2(const mcs_tensor *nrm, const mcs_tensor *zdz, float sigma, const mcs_tensor *out_gradA, const mcs_tensor *out_gradB,
                       float *col_gradA, float *col_gradB, mcs_stream stream)
{
    return bilateral<2, true>(nrm, zdz, {out_gradA, out_gradB}, {"out_gradA", "out_gradB"}, {col_gradA, col_gradB}, sigma, stream);
}

}  // extern "C"
