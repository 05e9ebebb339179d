// elementwise.cu -- B200 kernels for the renderutils streaming ops:
//   lambert / frostbite_diffuse / fresnel_shlick / ndf_ggx / lambda_ggx / masking_smith /
//   pbr_specular / pbr_bsdf / prepare_shading_normal, forward and backward.
// Replaces render/renderutils/c_src/bsdf.cu:382-707, normal.cu:95-178 and their launchers in
// render/renderutils/c_src/torch_bindings.cpp (8x8 blocks, one scalar-load pixel per thread).
//
// These ops are pure HBM streaming (84 B/px fwd, 156 B/px bwd for pbr_bsdf, SURVEY.md section 8d).
// Design: each thread owns FOUR consecutive pixels so that every contiguous [.,3] fp32 operand is
// moved with three 128-bit loads/stores (48 B per thread, 1536 B per warp-instruction group, fully
// coalesced), broadcast operands (e.g. view_pos [B,1,1,3]) fall back to strided scalar loads that
// hit L1; grid = enough 256-thread CTAs to cover the pixels (>= several waves over 148 SMs at
// 512x512), no shared memory, no divergence except the BSDF's own branches.
// A cp.async.bulk + mbarrier pipeline that staged the contiguous operands in shared memory was measured on B200 and was slower on
// every op (pbr_bsdf 16x512^2 fwd 0.107 vs 0.094 ms, bwd 0.309 vs 0.213 ms; shade tail fwd 0.033 vs 0.031 ms): these ops are
// instruction-issue / dependency bound (385-860 instructions per pixel at 94-139 registers), and the stages cost occupancy.  It was
// removed; the evidence is in profiles/r02_ew_tma_ab.json.
#include "bsdf.cuh"

namespace {

struct Grid { int N, H, W; int64_t npx; };

struct TIn {
    TView v;
    int fast;      // contiguous, full grid, 16B aligned -> vector path
};

struct Px4 {
    int64_t p0;
    int cnt;
};

__device__ __forceinline__ void px_decode(const Grid &g, int64_t p, int &n, int &h, int &w)
{
    w = (int)(p % g.W);
    int64_t t = p / g.W;
    h = (int)(t % g.H);
    n = (int)(t / g.H);
}

// FULL = all four pixels valid: every loop bound and array index is a compile-time constant, so the pixel
// registers never spill to local memory (the ragged tail is a separate, rarely executed instantiation).
template <int C, bool FULL>
__device__ __forceinline__ void ew_load(const TIn &t, const Grid &g, const Px4 &q, float (&out)[4][C])
{
    if (FULL && t.fast) {
        const float4 *src = reinterpret_cast<const float4 *>(t.v.p + q.p0 * C);
        float buf[4 * C];
#pragma unroll
        for (int i = 0; i < C; ++i) {
            float4 x = __ldg(src + i);
            buf[4 * i + 0] = x.x; buf[4 * i + 1] = x.y; buf[4 * i + 2] = x.z; buf[4 * i + 3] = x.w;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int c = 0; c < C; ++c) out[k][c] = buf[k * C + c];
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (FULL || k < q.cnt) {
                int n, h, w;
                px_decode(g, q.p0 + k, n, h, w);
                const float *src = t.v.p + t.v.off(n, h, w);
#pragma unroll
                for (int c = 0; c < C; ++c) out[k][c] = __ldg(src + (t.v.n3 == 1 ? 0 : c * t.v.s3));
            } else {
#pragma unroll
                for (int c = 0; c < C; ++c) out[k][c] = 0.0f;
            }
        }
    }
}

template <int C, bool FULL>
__device__ __forceinline__ void ew_store(float *dst, const Px4 &q, const float (&v)[4][C])
{
    if (FULL) {
        float buf[4 * C];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int c = 0; c < C; ++c) buf[k * C + c] = v[k][c];
        float4 *d = reinterpret_cast<float4 *>(dst + q.p0 * C);
#pragma unroll
        for (int i = 0; i < C; ++i) d[i] = make_float4(buf[4 * i], buf[4 * i + 1], buf[4 * i + 2], buf[4 * i + 3]);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k < q.cnt) {
#pragma unroll
                for (int c = 0; c < C; ++c) dst[(q.p0 + k) * C + c] = v[k][c];
            }
    }
}

__device__ __forceinline__ f3 to3(const float (&a)[3]) { return F3(a[0], a[1], a[2]); }
__device__ __forceinline__ void from3(float (&a)[3], f3 v) { a[0] = v.x; a[1] = v.y; a[2] = v.z; }

constexpr int EW_MINB = 2;     // caps the heaviest op (pbr_bsdf backward, 139 regs) at 128 so two CTAs fit: 0.32 -> 0.21 ms at 16x512x512
template <class Op>
__global__ void __launch_bounds__(256, EW_MINB) ew_kernel(Op op, Grid g)
{
    int64_t q4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    Px4 q;
    q.p0 = q4 * 4;
    if (q.p0 >= g.npx) return;
    int64_t rem = g.npx - q.p0;
    q.cnt = rem >= 4 ? 4 : (int)rem;
    if (q.cnt == 4) op.template run<true>(g, q);
    else op.template run<false>(g, q);
}

// ---------------------------------------------------------------------------------------------
// Ops
// ---------------------------------------------------------------------------------------------
struct LambertFwd {
    TIn nrm, wi; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], o[4][1];
        ew_load<3, FULL>(nrm, g, q, a); ew_load<3, FULL>(wi, g, q, b);
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k][0] = fwd_lambert(to3(a[k]), to3(b[k]));
        ew_store<1, FULL>(out, q, o);
    }
};
struct LambertBwd {
    TIn nrm, wi, dout; float *d_nrm, *d_wi;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], d[4][1], ga[4][3], gb[4][3];
        ew_load<3, FULL>(nrm, g, q, a); ew_load<3, FULL>(wi, g, q, b); ew_load<1, FULL>(dout, g, q, d);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f3 x = F3(0.0f), y = F3(0.0f);
            bwd_lambert(to3(a[k]), to3(b[k]), x, y, d[k][0]);
            from3(ga[k], x); from3(gb[k], y);
        }
        ew_store<3, FULL>(d_nrm, q, ga); ew_store<3, FULL>(d_wi, q, gb);
    }
};
struct FrostbiteFwd {
    TIn nrm, wi, wo, lr; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], l[4][1], o[4][1];
        ew_load<3, FULL>(nrm, g, q, a); ew_load<3, FULL>(wi, g, q, b); ew_load<3, FULL>(wo, g, q, c); ew_load<1, FULL>(lr, g, q, l);
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k][0] = fwd_frostbite(to3(a[k]), to3(b[k]), to3(c[k]), l[k][0]);
        ew_store<1, FULL>(out, q, o);
    }
};
struct FrostbiteBwd {
    TIn nrm, wi, wo, lr, dout; float *d_nrm, *d_wi, *d_wo, *d_lr;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], l[4][1], d[4][1], ga[4][3], gb[4][3], gc[4][3], gl[4][1];
        ew_load<3, FULL>(nrm, g, q, a); ew_load<3, FULL>(wi, g, q, b); ew_load<3, FULL>(wo, g, q, c); ew_load<1, FULL>(lr, g, q, l); ew_load<1, FULL>(dout, g, q, d);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f3 x = F3(0.0f), y = F3(0.0f), z = F3(0.0f); float dl = 0.0f;
            bwd_frostbite(to3(a[k]), to3(b[k]), to3(c[k]), l[k][0], x, y, z, dl, d[k][0]);
            from3(ga[k], x); from3(gb[k], y); from3(gc[k], z); gl[k][0] = dl;
        }
        ew_store<3, FULL>(d_nrm, q, ga); ew_store<3, FULL>(d_wi, q, gb); ew_store<3, FULL>(d_wo, q, gc); ew_store<1, FULL>(d_lr, q, gl);
    }
};
struct FresnelFwd {
    TIn f0, f90, c; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], cc[4][1], o[4][3];
        ew_load<3, FULL>(f0, g, q, a); ew_load<3, FULL>(f90, g, q, b); ew_load<1, FULL>(c, g, q, cc);
#pragma unroll
        for (int k = 0; k < 4; ++k) from3(o[k], fwd_fresnel3(to3(a[k]), to3(b[k]), cc[k][0]));
        ew_store<3, FULL>(out, q, o);
    }
};
struct FresnelBwd {
    TIn f0, f90, c, dout; float *d_f0, *d_f90, *d_c;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], cc[4][1], d[4][3], ga[4][3], gb[4][3], gc[4][1];
        ew_load<3, FULL>(f0, g, q, a); ew_load<3, FULL>(f90, g, q, b); ew_load<1, FULL>(c, g, q, cc); ew_load<3, FULL>(dout, g, q, d);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f3 x = F3(0.0f), y = F3(0.0f); float z = 0.0f;
            bwd_fresnel3(to3(a[k]), to3(b[k]), cc[k][0], x, y, z, to3(d[k]));
            from3(ga[k], x); from3(gb[k], y); gc[k][0] = z;
        }
        ew_store<3, FULL>(d_f0, q, ga); ew_store<3, FULL>(d_f90, q, gb); ew_store<1, FULL>(d_c, q, gc);
    }
};
template <int WHICH>   // 0 ndf, 1 lambda
struct Ggx2Fwd {
    TIn a2, c; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][1], b[4][1], o[4][1];
        ew_load<1, FULL>(a2, g, q, a); ew_load<1, FULL>(c, g, q, b);
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k][0] = WHICH == 0 ? fwd_ndf_ggx(a[k][0], b[k][0]) : fwd_lambda_ggx(a[k][0], b[k][0]);
        ew_store<1, FULL>(out, q, o);
    }
};
template <int WHICH>
struct Ggx2Bwd {
    TIn a2, c, dout; float *d_a2, *d_c;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][1], b[4][1], d[4][1], ga[4][1], gb[4][1];
        ew_load<1, FULL>(a2, g, q, a); ew_load<1, FULL>(c, g, q, b); ew_load<1, FULL>(dout, g, q, d);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float x = 0.0f, y = 0.0f;
            if (WHICH == 0) bwd_ndf_ggx(a[k][0], b[k][0], x, y, d[k][0]);
            else bwd_lambda_ggx(a[k][0], b[k][0], x, y, d[k][0]);
            ga[k][0] = x; gb[k][0] = y;
        }
        ew_store<1, FULL>(d_a2, q, ga); ew_store<1, FULL>(d_c, q, gb);
    }
};
struct MaskingFwd {
    TIn a2, ci, co; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][1], b[4][1], c[4][1], o[4][1];
        ew_load<1, FULL>(a2, g, q, a); ew_load<1, FULL>(ci, g, q, b); ew_load<1, FULL>(co, g, q, c);
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k][0] = fwd_masking_smith(a[k][0], b[k][0], c[k][0]);
        ew_store<1, FULL>(out, q, o);
    }
};
struct MaskingBwd {
    TIn a2, ci, co, dout; float *d_a2, *d_ci, *d_co;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][1], b[4][1], c[4][1], d[4][1], ga[4][1], gb[4][1], gc[4][1];
        ew_load<1, FULL>(a2, g, q, a); ew_load<1, FULL>(ci, g, q, b); ew_load<1, FULL>(co, g, q, c); ew_load<1, FULL>(dout, g, q, d);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float x = 0.0f, y = 0.0f, z = 0.0f;
            bwd_masking_smith(a[k][0], b[k][0], c[k][0], x, y, z, d[k][0]);
            ga[k][0] = x; gb[k][0] = y; gc[k][0] = z;
        }
        ew_store<1, FULL>(d_a2, q, ga); ew_store<1, FULL>(d_ci, q, gb); ew_store<1, FULL>(d_co, q, gc);
    }
};
struct SpecFwd {
    TIn col, nrm, wo, wi, alpha; float min_roughness; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], d[4][3], al[4][1], o[4][3];
        ew_load<3, FULL>(col, g, q, a); ew_load<3, FULL>(nrm, g, q, b); ew_load<3, FULL>(wo, g, q, c); ew_load<3, FULL>(wi, g, q, d); ew_load<1, FULL>(alpha, g, q, al);
#pragma unroll
        for (int k = 0; k < 4; ++k) from3(o[k], fwd_pbr_specular(to3(a[k]), to3(b[k]), to3(c[k]), to3(d[k]), al[k][0], min_roughness));
        ew_store<3, FULL>(out, q, o);
    }
};
struct SpecBwd {
    TIn col, nrm, wo, wi, alpha, dout; float min_roughness; float *d_col, *d_nrm, *d_wo, *d_wi, *d_alpha;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], d[4][3], al[4][1], go[4][3];
        ew_load<3, FULL>(col, g, q, a); ew_load<3, FULL>(nrm, g, q, b); ew_load<3, FULL>(wo, g, q, c); ew_load<3, FULL>(wi, g, q, d); ew_load<1, FULL>(alpha, g, q, al);
        ew_load<3, FULL>(dout, g, q, go);
        float ga[4][3], gb[4][3], gc[4][3], gd[4][3], gal[4][1];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f3 x = F3(0.0f), y = F3(0.0f), z = F3(0.0f), w = F3(0.0f); float da = 0.0f;
            bwd_pbr_specular(to3(a[k]), to3(b[k]), to3(c[k]), to3(d[k]), al[k][0], min_roughness, x, y, z, w, da, to3(go[k]));
            from3(ga[k], x); from3(gb[k], y); from3(gc[k], z); from3(gd[k], w); gal[k][0] = da;
        }
        ew_store<3, FULL>(d_col, q, ga); ew_store<3, FULL>(d_nrm, q, gb); ew_store<3, FULL>(d_wo, q, gc); ew_store<3, FULL>(d_wi, q, gd); ew_store<1, FULL>(d_alpha, q, gal);
    }
};
struct PbrFwd {
    TIn kd, arm, pos, nrm, view, light; float min_roughness; int bsdf; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], d[4][3], e[4][3], f[4][3], o[4][3];
        ew_load<3, FULL>(kd, g, q, a); ew_load<3, FULL>(arm, g, q, b); ew_load<3, FULL>(pos, g, q, c);
        ew_load<3, FULL>(nrm, g, q, d); ew_load<3, FULL>(view, g, q, e); ew_load<3, FULL>(light, g, q, f);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            from3(o[k], ru_fwd_pbr_bsdf(to3(a[k]), to3(b[k]), to3(c[k]), to3(d[k]), to3(e[k]), to3(f[k]), min_roughness, bsdf));
        ew_store<3, FULL>(out, q, o);
    }
};
struct PbrBwd {
    TIn kd, arm, pos, nrm, view, light, dout; float min_roughness; int bsdf;
    float *d_kd, *d_arm, *d_pos, *d_nrm, *d_view, *d_light;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], d[4][3], e[4][3], f[4][3], go[4][3];
        ew_load<3, FULL>(kd, g, q, a); ew_load<3, FULL>(arm, g, q, b); ew_load<3, FULL>(pos, g, q, c);
        ew_load<3, FULL>(nrm, g, q, d); ew_load<3, FULL>(view, g, q, e); ew_load<3, FULL>(light, g, q, f); ew_load<3, FULL>(dout, g, q, go);
        float ga[4][3], gb[4][3], gc[4][3], gd[4][3], ge[4][3], gf[4][3];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f3 x0 = F3(0.0f), x1 = F3(0.0f), x2 = F3(0.0f), x3 = F3(0.0f), x4 = F3(0.0f), x5 = F3(0.0f);
            ru_bwd_pbr_bsdf(to3(a[k]), to3(b[k]), to3(c[k]), to3(d[k]), to3(e[k]), to3(f[k]), min_roughness, bsdf,
                            x0, x1, x2, x3, x4, x5, to3(go[k]));
            from3(ga[k], x0); from3(gb[k], x1); from3(gc[k], x2); from3(gd[k], x3); from3(ge[k], x4); from3(gf[k], x5);
        }
        ew_store<3, FULL>(d_kd, q, ga); ew_store<3, FULL>(d_arm, q, gb); ew_store<3, FULL>(d_pos, q, gc);
        ew_store<3, FULL>(d_nrm, q, gd); ew_store<3, FULL>(d_view, q, ge); ew_store<3, FULL>(d_light, q, gf);
    }
};
struct PsnFwd {
    TIn pos, view, pn, sn, st, gn; int two_sided, opengl; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], d[4][3], e[4][3], f[4][3], o[4][3];
        ew_load<3, FULL>(pos, g, q, a); ew_load<3, FULL>(view, g, q, b); ew_load<3, FULL>(pn, g, q, c);
        ew_load<3, FULL>(sn, g, q, d); ew_load<3, FULL>(st, g, q, e); ew_load<3, FULL>(gn, g, q, f);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f3 smooth_nrm = safe_normalize(to3(d[k])), smooth_tng = safe_normalize(to3(e[k]));
            f3 view_vec = safe_normalize(to3(b[k]) - to3(a[k]));
            f3 geom = to3(f[k]);
            f3 sh = fwd_perturb_normal(to3(c[k]), smooth_nrm, smooth_tng, opengl != 0);
            f3 res = (two_sided && dot(view_vec, geom) < 0.0f) ? fwd_bend_normal(view_vec, -sh, -geom) : fwd_bend_normal(view_vec, sh, geom);
            from3(o[k], res);
        }
        ew_store<3, FULL>(out, q, o);
    }
};
struct PsnBwd {
    TIn pos, view, pn, sn, st, gn, dout; int two_sided, opengl;
    float *d_pos, *d_view, *d_pn, *d_sn, *d_st, *d_gn;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float a[4][3], b[4][3], c[4][3], d[4][3], e[4][3], f[4][3], go[4][3];
        ew_load<3, FULL>(pos, g, q, a); ew_load<3, FULL>(view, g, q, b); ew_load<3, FULL>(pn, g, q, c);
        ew_load<3, FULL>(sn, g, q, d); ew_load<3, FULL>(st, g, q, e); ew_load<3, FULL>(gn, g, q, f); ew_load<3, FULL>(dout, g, q, go);
        float ga[4][3], gb[4][3], gc[4][3], gd[4][3], ge[4][3], gf[4][3];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f3 _sn = to3(d[k]), _st = to3(e[k]);
            f3 smooth_nrm = safe_normalize(_sn), smooth_tng = safe_normalize(_st);
            f3 _vv = to3(b[k]) - to3(a[k]);
            f3 view_vec = safe_normalize(_vv);
            f3 geom = to3(f[k]), p = to3(c[k]);
            f3 sh = fwd_perturb_normal(p, smooth_nrm, smooth_tng, opengl != 0);
            f3 d_vv = F3(0.0f), d_sh = F3(0.0f), d_geom = F3(0.0f);
            if (two_sided && dot(view_vec, geom) < 0.0f) {
                bwd_bend_normal(view_vec, -sh, -geom, d_vv, d_sh, d_geom, to3(go[k]));
                d_sh = -d_sh; d_geom = -d_geom;
            } else bwd_bend_normal(view_vec, sh, geom, d_vv, d_sh, d_geom, to3(go[k]));
            f3 dp = F3(0.0f), dsn = F3(0.0f), dst = F3(0.0f);
            bwd_perturb_normal(p, smooth_nrm, smooth_tng, dp, dsn, dst, d_sh, opengl != 0);
            f3 d__vv = F3(0.0f), d__sn = F3(0.0f), d__st = F3(0.0f);
            bwd_safe_normalize(_vv, d__vv, d_vv);
            bwd_safe_normalize(_sn, d__sn, dsn);
            bwd_safe_normalize(_st, d__st, dst);
            from3(ga[k], -d__vv); from3(gb[k], d__vv); from3(gc[k], dp); from3(gd[k], d__sn); from3(ge[k], d__st); from3(gf[k], d_geom);
        }
        ew_store<3, FULL>(d_pos, q, ga); ew_store<3, FULL>(d_view, q, gb); ew_store<3, FULL>(d_pn, q, gc);
        ew_store<3, FULL>(d_sn, q, gd); ew_store<3, FULL>(d_st, q, ge); ew_store<3, FULL>(d_gn, q, gf);
    }
};

// ---------------------------------------------------------------------------------------------
// Host-side launch plumbing
// ---------------------------------------------------------------------------------------------
// Tail of render.shade(), render/render.py:119-131 (row f3): normalise the two denoiser outputs (rgb weighted sum, weight) and recombine
// the demodulated signals:  shaded = (A.rgb / A.w) * kd * (1 - ks.z) + B.rgb / B.w   ('pbr');   shaded = (A.rgb / A.w) * kd   ('diffuse' / 'white').
// One launch instead of ~8 torch element-wise kernels forward and ~14 backward.
struct CombineFwd {
    TIn a4, b4, kd, ks; int pbr; float *out;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float A[4][4], B[4][4], d[4][3], s[4][3], o[4][3];
        ew_load<4, FULL>(a4, g, q, A); ew_load<3, FULL>(kd, g, q, d);
        if (pbr) { ew_load<4, FULL>(b4, g, q, B); ew_load<3, FULL>(ks, g, q, s); }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float ia = 1.0f / A[k][3], m = pbr ? 1.0f - s[k][2] : 1.0f, ib = pbr ? 1.0f / B[k][3] : 0.0f;
#pragma unroll
            for (int c = 0; c < 3; ++c) o[k][c] = A[k][c] * ia * d[k][c] * m + (pbr ? B[k][c] * ib : 0.0f);
        }
        ew_store<3, FULL>(out, q, o);
    }
};
struct CombineBwd {
    TIn a4, b4, kd, ks, dout; int pbr; float *d_a4, *d_b4, *d_kd, *d_ks;
    template <bool FULL> __device__ void run(const Grid &g, const Px4 &q) const
    {
        float A[4][4], B[4][4], d[4][3], s[4][3], go[4][3], gA[4][4], gB[4][4], gd[4][3], gs[4][3];
        ew_load<4, FULL>(a4, g, q, A); ew_load<3, FULL>(kd, g, q, d); ew_load<3, FULL>(dout, g, q, go);
        if (pbr) { ew_load<4, FULL>(b4, g, q, B); ew_load<3, FULL>(ks, g, q, s); }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float ia = 1.0f / A[k][3], m = pbr ? 1.0f - s[k][2] : 1.0f, ib = pbr ? 1.0f / B[k][3] : 0.0f;
            float gaw = 0.0f, gbw = 0.0f, gm = 0.0f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float da = A[k][c] * ia;                       // demodulated diffuse
                gA[k][c] = go[k][c] * d[k][c] * m * ia;
                gaw -= go[k][c] * d[k][c] * m * da * ia;
                gd[k][c] = go[k][c] * da * m;
                gm += go[k][c] * da * d[k][c];
                gB[k][c] = pbr ? go[k][c] * ib : 0.0f;
                gbw -= pbr ? go[k][c] * B[k][c] * ib * ib : 0.0f;
            }
            gA[k][3] = gaw; gB[k][3] = gbw;
            gs[k][0] = 0.0f; gs[k][1] = 0.0f; gs[k][2] = pbr ? -gm : 0.0f;
        }
        ew_store<4, FULL>(d_a4, q, gA); ew_store<3, FULL>(d_kd, q, gd);
        if (pbr) { ew_store<4, FULL>(d_b4, q, gB); ew_store<3, FULL>(d_ks, q, gs); }
    }
};

struct GridBuilder {
    Grid g{1, 1, 1, 0};
    bool ok = true;
    void add(const mcs_tensor *t)
    {
        if (!view_ok(t)) { ok = false; return; }
        g.N = t->sizes[0] > g.N ? t->sizes[0] : g.N;      // update_grid, torch_bindings.cpp:87-101
        g.H = t->sizes[1] > g.H ? t->sizes[1] : g.H;
        g.W = t->sizes[2] > g.W ? t->sizes[2] : g.W;
    }
    void finish() { g.npx = (int64_t)g.N * g.H * g.W; }
};

static bool mk_in(const mcs_tensor *t, const Grid &g, int C, TIn &out, const char *name)
{
    if (!(t->sizes[3] == C || t->sizes[3] == 1)) { mcs_set_error("%s must have %d channels (got %d)", name, C, t->sizes[3]); return false; }
    for (int d = 0; d < 3; ++d) {
        int full = d == 0 ? g.N : (d == 1 ? g.H : g.W);
        if (!(t->sizes[d] == full || t->sizes[d] == 1)) { mcs_set_error("%s: dim %d = %d not broadcastable to %d", name, d, t->sizes[d], full); return false; }
    }
    out.v = make_view(t);
    bool contig = t->sizes[0] == g.N && t->sizes[1] == g.H && t->sizes[2] == g.W && t->sizes[3] == C &&
                  (C == 1 || t->strides[3] == 1) && t->strides[2] == C && t->strides[1] == C * g.W && t->strides[0] == C * g.W * g.H;
    out.fast = contig && ((uintptr_t)t->ptr % 16 == 0);
    return true;
}

template <class Op>
static int launch(const Op &op, const Grid &g, cudaStream_t s)
{
    if (g.npx == 0) return 0;
    int64_t nthreads = (g.npx + 3) / 4;
    int block = 256;
    int64_t nblocks = (nthreads + block - 1) / block;
    MCS_REQUIRE(nblocks < (1ll << 31), "elementwise grid too large");
    ew_kernel<Op><<<(unsigned)nblocks, block, 0, s>>>(op, g);
    MCS_LAUNCH_CHECK();
    return 0;
}

#define IN(field, tensor, C) if (!mk_in(tensor, gb.g, C, op.field, #tensor)) return 1
#define GRID(...) GridBuilder gb; { const mcs_tensor *ts_[] = {__VA_ARGS__}; for (auto t_ : ts_) gb.add(t_); } \
    MCS_REQUIRE(gb.ok, "%s: null / empty tensor argument", __func__); gb.finish()

}  // namespace

extern "C" {

int mcs_lambert_fwd(const mcs_tensor *nrm, const mcs_tensor *wi, float *out, mcs_stream s)
{
    GRID(nrm, wi); LambertFwd op; IN(nrm, nrm, 3); IN(wi, wi, 3); op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_lambert_bwd(const mcs_tensor *nrm, const mcs_tensor *wi, const mcs_tensor *d_out, float *d_nrm, float *d_wi, mcs_stream s)
{
    GRID(nrm, wi, d_out); LambertBwd op; IN(nrm, nrm, 3); IN(wi, wi, 3); IN(dout, d_out, 1); op.d_nrm = d_nrm; op.d_wi = d_wi;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_frostbite_fwd(const mcs_tensor *nrm, const mcs_tensor *wi, const mcs_tensor *wo, const mcs_tensor *lin_rough, float *out, mcs_stream s)
{
    GRID(nrm, wi, wo, lin_rough); FrostbiteFwd op; IN(nrm, nrm, 3); IN(wi, wi, 3); IN(wo, wo, 3); IN(lr, lin_rough, 1); op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_frostbite_bwd(const mcs_tensor *nrm, const mcs_tensor *wi, const mcs_tensor *wo, const mcs_tensor *lin_rough, const mcs_tensor *d_out,
                      float *d_nrm, float *d_wi, float *d_wo, float *d_lin_rough, mcs_stream s)
{
    GRID(nrm, wi, wo, lin_rough, d_out); FrostbiteBwd op; IN(nrm, nrm, 3); IN(wi, wi, 3); IN(wo, wo, 3); IN(lr, lin_rough, 1); IN(dout, d_out, 1);
    op.d_nrm = d_nrm; op.d_wi = d_wi; op.d_wo = d_wo; op.d_lr = d_lin_rough;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_fresnel_shlick_fwd(const mcs_tensor *f0, const mcs_tensor *f90, const mcs_tensor *cos_theta, float *out, mcs_stream s)
{
    GRID(f0, f90, cos_theta); FresnelFwd op; IN(f0, f0, 3); IN(f90, f90, 3); IN(c, cos_theta, 1); op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_fresnel_shlick_bwd(const mcs_tensor *f0, const mcs_tensor *f90, const mcs_tensor *cos_theta, const mcs_tensor *d_out,
                           float *d_f0, float *d_f90, float *d_cos, mcs_stream s)
{
    GRID(f0, f90, cos_theta, d_out); FresnelBwd op; IN(f0, f0, 3); IN(f90, f90, 3); IN(c, cos_theta, 1); IN(dout, d_out, 3);
    op.d_f0 = d_f0; op.d_f90 = d_f90; op.d_c = d_cos;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_ndf_ggx_fwd(const mcs_tensor *alpha_sqr, const mcs_tensor *cos_theta, float *out, mcs_stream s)
{
    GRID(alpha_sqr, cos_theta); Ggx2Fwd<0> op; IN(a2, alpha_sqr, 1); IN(c, cos_theta, 1); op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_ndf_ggx_bwd(const mcs_tensor *alpha_sqr, const mcs_tensor *cos_theta, const mcs_tensor *d_out, float *d_alpha_sqr, float *d_cos, mcs_stream s)
{
    GRID(alpha_sqr, cos_theta, d_out); Ggx2Bwd<0> op; IN(a2, alpha_sqr, 1); IN(c, cos_theta, 1); IN(dout, d_out, 1); op.d_a2 = d_alpha_sqr; op.d_c = d_cos;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_lambda_ggx_fwd(const mcs_tensor *alpha_sqr, const mcs_tensor *cos_theta, float *out, mcs_stream s)
{
    GRID(alpha_sqr, cos_theta); Ggx2Fwd<1> op; IN(a2, alpha_sqr, 1); IN(c, cos_theta, 1); op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_lambda_ggx_bwd(const mcs_tensor *alpha_sqr, const mcs_tensor *cos_theta, const mcs_tensor *d_out, float *d_alpha_sqr, float *d_cos, mcs_stream s)
{
    GRID(alpha_sqr, cos_theta, d_out); Ggx2Bwd<1> op; IN(a2, alpha_sqr, 1); IN(c, cos_theta, 1); IN(dout, d_out, 1); op.d_a2 = d_alpha_sqr; op.d_c = d_cos;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_masking_smith_fwd(const mcs_tensor *alpha_sqr, const mcs_tensor *cos_i, const mcs_tensor *cos_o, float *out, mcs_stream s)
{
    GRID(alpha_sqr, cos_i, cos_o); MaskingFwd op; IN(a2, alpha_sqr, 1); IN(ci, cos_i, 1); IN(co, cos_o, 1); op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_masking_smith_bwd(const mcs_tensor *alpha_sqr, const mcs_tensor *cos_i, const mcs_tensor *cos_o, const mcs_tensor *d_out,
                          float *d_alpha_sqr, float *d_cos_i, float *d_cos_o, mcs_stream s)
{
    GRID(alpha_sqr, cos_i, cos_o, d_out); MaskingBwd op; IN(a2, alpha_sqr, 1); IN(ci, cos_i, 1); IN(co, cos_o, 1); IN(dout, d_out, 1);
    op.d_a2 = d_alpha_sqr; op.d_ci = d_cos_i; op.d_co = d_cos_o;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_pbr_specular_fwd(const mcs_tensor *col, const mcs_tensor *nrm, const mcs_tensor *wo, const mcs_tensor *wi, const mcs_tensor *alpha,
                         float min_roughness, float *out, mcs_stream s)
{
    GRID(col, nrm, wo, wi, alpha); SpecFwd op; IN(col, col, 3); IN(nrm, nrm, 3); IN(wo, wo, 3); IN(wi, wi, 3); IN(alpha, alpha, 1);
    op.min_roughness = min_roughness; op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_pbr_specular_bwd(const mcs_tensor *col, const mcs_tensor *nrm, const mcs_tensor *wo, const mcs_tensor *wi, const mcs_tensor *alpha,
                         float min_roughness, const mcs_tensor *d_out,
                         float *d_col, float *d_nrm, float *d_wo, float *d_wi, float *d_alpha, mcs_stream s)
{
    GRID(col, nrm, wo, wi, alpha, d_out); SpecBwd op; IN(col, col, 3); IN(nrm, nrm, 3); IN(wo, wo, 3); IN(wi, wi, 3); IN(alpha, alpha, 1); IN(dout, d_out, 3);
    op.min_roughness = min_roughness; op.d_col = d_col; op.d_nrm = d_nrm; op.d_wo = d_wo; op.d_wi = d_wi; op.d_alpha = d_alpha;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_pbr_bsdf_fwd(const mcs_tensor *kd, const mcs_tensor *arm, const mcs_tensor *pos, const mcs_tensor *nrm, const mcs_tensor *view_pos,
                     const mcs_tensor *light_pos, float min_roughness, int32_t bsdf, float *out, mcs_stream s)
{
    GRID(kd, arm, pos, nrm, view_pos, light_pos); PbrFwd op;
    IN(kd, kd, 3); IN(arm, arm, 3); IN(pos, pos, 3); IN(nrm, nrm, 3); IN(view, view_pos, 3); IN(light, light_pos, 3);
    op.min_roughness = min_roughness; op.bsdf = bsdf; op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_pbr_bsdf_bwd(const mcs_tensor *kd, const mcs_tensor *arm, const mcs_tensor *pos, const mcs_tensor *nrm, const mcs_tensor *view_pos,
                     const mcs_tensor *light_pos, float min_roughness, int32_t bsdf, const mcs_tensor *d_out,
                     float *d_kd, float *d_arm, float *d_pos, float *d_nrm, float *d_view_pos, float *d_light_pos, mcs_stream s)
{
    GRID(kd, arm, pos, nrm, view_pos, light_pos, d_out); PbrBwd op;
    IN(kd, kd, 3); IN(arm, arm, 3); IN(pos, pos, 3); IN(nrm, nrm, 3); IN(view, view_pos, 3); IN(light, light_pos, 3); IN(dout, d_out, 3);
    op.min_roughness = min_roughness; op.bsdf = bsdf;
    op.d_kd = d_kd; op.d_arm = d_arm; op.d_pos = d_pos; op.d_nrm = d_nrm; op.d_view = d_view_pos; op.d_light = d_light_pos;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_prepare_shading_normal_fwd(const mcs_tensor *pos, const mcs_tensor *view_pos, const mcs_tensor *perturbed_nrm, const mcs_tensor *smooth_nrm,
                                   const mcs_tensor *smooth_tng, const mcs_tensor *geom_nrm, int32_t two_sided_shading, int32_t opengl,
                                   float *out, mcs_stream s)
{
    GRID(pos, view_pos, perturbed_nrm, smooth_nrm, smooth_tng, geom_nrm); PsnFwd op;
    IN(pos, pos, 3); IN(view, view_pos, 3); IN(pn, perturbed_nrm, 3); IN(sn, smooth_nrm, 3); IN(st, smooth_tng, 3); IN(gn, geom_nrm, 3);
    op.two_sided = two_sided_shading; op.opengl = opengl; op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_prepare_shading_normal_bwd(const mcs_tensor *pos, const mcs_tensor *view_pos, const mcs_tensor *perturbed_nrm, const mcs_tensor *smooth_nrm,
                                   const mcs_tensor *smooth_tng, const mcs_tensor *geom_nrm, int32_t two_sided_shading, int32_t opengl,
                                   const mcs_tensor *d_out,
                                   float *d_pos, float *d_view_pos, float *d_perturbed_nrm, float *d_smooth_nrm, float *d_smooth_tng, float *d_geom_nrm,
                                   mcs_stream s)
{
    GRID(pos, view_pos, perturbed_nrm, smooth_nrm, smooth_tng, geom_nrm, d_out); PsnBwd op;
    IN(pos, pos, 3); IN(view, view_pos, 3); IN(pn, perturbed_nrm, 3); IN(sn, smooth_nrm, 3); IN(st, smooth_tng, 3); IN(gn, geom_nrm, 3); IN(dout, d_out, 3);
    op.two_sided = two_sided_shading; op.opengl = opengl;
    op.d_pos = d_pos; op.d_view = d_view_pos; op.d_pn = d_perturbed_nrm; op.d_sn = d_smooth_nrm; op.d_st = d_smooth_tng; op.d_gn = d_geom_nrm;
    return launch(op, gb.g, (cudaStream_t)s);
}

int mcs_shade_combine_fwd(const mcs_tensor *a4, const mcs_tensor *b4, const mcs_tensor *kd, const mcs_tensor *ks, int32_t pbr, float *out, mcs_stream s)
{
    GRID(a4, b4, kd, ks); CombineFwd op; IN(a4, a4, 4); IN(b4, b4, 4); IN(kd, kd, 3); IN(ks, ks, 3); op.pbr = pbr; op.out = out;
    return launch(op, gb.g, (cudaStream_t)s);
}
int mcs_shade_combine_bwd(const mcs_tensor *a4, const mcs_tensor *b4, const mcs_tensor *kd, const mcs_tensor *ks, int32_t pbr, const mcs_tensor *d_out,
                          float *d_a4, float *d_b4, float *d_kd, float *d_ks, mcs_stream s)
{
    GRID(a4, b4, kd, ks, d_out); CombineBwd op; IN(a4, a4, 4); IN(b4, b4, 4); IN(kd, kd, 3); IN(ks, ks, 3); IN(dout, d_out, 3); op.pbr = pbr;
    op.d_a4 = d_a4; op.d_b4 = d_b4; op.d_kd = d_kd; op.d_ks = d_ks;
    return launch(op, gb.g, (cudaStream_t)s);
}

}  // extern "C"
