// dfb_math.h -- per-voxel / per-point arithmetic shared by every kernel.
//
// Two tiers (DESIGN.md "Exactness"):
//   * fast tier  : fp32 closed-form DQB warp + projection, used only to CLASSIFY a voxel
//                  (certainly-not-updated / certainly-clamped / uncertain) with explicit error margins;
//   * exact tier : a literal re-statement of the reference's numpy arithmetic -- same operation order,
//                  same float32/float64 roundings (numpy>=2 promotion) -- written with explicit
//                  round-to-nearest intrinsics so the compiler can neither fuse nor reorder it.
//
// The header is also compilable by a host C++ compiler (DFB_HD expands to nothing, the rounding
// intrinsics to plain IEEE operations; build with -ffp-contract=off) so that tests can exercise the
// very same per-voxel functions on the CPU box that has no GPU (tests/hostshim/).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define DFB_HD __host__ __device__ __forceinline__
#define DFB_HDN inline __host__ __device__
#else
#define DFB_HD inline
#define DFB_HDN inline
#endif

#if !defined(__CUDACC__)
struct float4 { float x, y, z, w; };
#endif

namespace dfb {

// ---------------------------------------------------------------------------------------------
// explicit-rounding scalar ops (no FMA contraction, no reassociation)
// ---------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
DFB_HD float fmul(float a, float b) { return __fmul_rn(a, b); }
DFB_HD float fadd(float a, float b) { return __fadd_rn(a, b); }
DFB_HD float fsub(float a, float b) { return __fsub_rn(a, b); }
DFB_HD float fdiv(float a, float b) { return __fdiv_rn(a, b); }
DFB_HD float fsqrt(float a) { return __fsqrt_rn(a); }
DFB_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
DFB_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
DFB_HD double dsub(double a, double b) { return __dsub_rn(a, b); }
DFB_HD double ddiv(double a, double b) { return __ddiv_rn(a, b); }
DFB_HD double dsqrt(double a) { return __dsqrt_rn(a); }
DFB_HD double drint(double a) { return rint(a); }
#else
DFB_HD float fmul(float a, float b) { volatile float r = a * b; return r; }
DFB_HD float fadd(float a, float b) { volatile float r = a + b; return r; }
DFB_HD float fsub(float a, float b) { volatile float r = a - b; return r; }
DFB_HD float fdiv(float a, float b) { volatile float r = a / b; return r; }
DFB_HD float fsqrt(float a) { volatile float r = sqrtf(a); return r; }
DFB_HD double dmul(double a, double b) { volatile double r = a * b; return r; }
DFB_HD double dadd(double a, double b) { volatile double r = a + b; return r; }
DFB_HD double dsub(double a, double b) { volatile double r = a - b; return r; }
DFB_HD double ddiv(double a, double b) { volatile double r = a / b; return r; }
DFB_HD double dsqrt(double a) { volatile double r = sqrt(a); return r; }
DFB_HD double drint(double a) { return nearbyint(a); }
#endif

struct OpsF {
    typedef float T;
    static DFB_HD T mul(T a, T b) { return fmul(a, b); }
    static DFB_HD T add(T a, T b) { return fadd(a, b); }
    static DFB_HD T sub(T a, T b) { return fsub(a, b); }
};
struct OpsD {
    typedef double T;
    static DFB_HD T mul(T a, T b) { return dmul(a, b); }
    static DFB_HD T add(T a, T b) { return dadd(a, b); }
    static DFB_HD T sub(T a, T b) { return dsub(a, b); }
};

// core/util.py:263-269  quaternion_multiply(quaternion1, quaternion0), expressions evaluated in the
// promoted input dtype (Ops::T), left to right, then widened to float64.
template <class Ops>
DFB_HD void qmul_ref(const typename Ops::T* q1, const typename Ops::T* q0, double* out) {
    typedef typename Ops::T T;
    const T w0 = q0[0], x0 = q0[1], y0 = q0[2], z0 = q0[3];
    const T w1 = q1[0], x1 = q1[1], y1 = q1[2], z1 = q1[3];
    out[0] = (double)Ops::add(Ops::sub(Ops::sub(Ops::mul(-x1, x0), Ops::mul(y1, y0)), Ops::mul(z1, z0)), Ops::mul(w1, w0));
    out[1] = (double)Ops::add(Ops::sub(Ops::add(Ops::mul(x1, w0), Ops::mul(y1, z0)), Ops::mul(z1, y0)), Ops::mul(w1, x0));
    out[2] = (double)Ops::add(Ops::add(Ops::add(Ops::mul(-x1, z0), Ops::mul(y1, w0)), Ops::mul(z1, x0)), Ops::mul(w1, y0));
    out[3] = (double)Ops::add(Ops::add(Ops::sub(Ops::mul(x1, y0), Ops::mul(y1, x0)), Ops::mul(z1, w0)), Ops::mul(w1, z0));
}

// core/util.py:68-72  dqb_warp(dq, pos).  `dq_is_f32`: dq is a float32 array in the reference, so
// dual_quaternion_multiply(dq, vq) multiplies float32 by float32 (vq is float32 by construction, Q3).
// pos is rounded to float32 first (Q3).  out = dual part [5:8] of dq * vq * conj(dq).
DFB_HDN void dqb_warp_ref(const double* dq, bool dq_is_f32, const double* pos, double* out) {
    const float vr[4] = {1.f, 0.f, 0.f, 0.f};
    const float vd[4] = {0.f, (float)pos[0], (float)pos[1], (float)pos[2]};
    double qr[4], qd[4], t0[4], t1[4];
    if (dq_is_f32) {
        const float r[4] = {(float)dq[0], (float)dq[1], (float)dq[2], (float)dq[3]};
        const float d[4] = {(float)dq[4], (float)dq[5], (float)dq[6], (float)dq[7]};
        qmul_ref<OpsF>(r, vr, qr);
        qmul_ref<OpsF>(r, vd, t0);
        qmul_ref<OpsF>(d, vr, t1);
    } else {
        const double vrd[4] = {1.0, 0.0, 0.0, 0.0};
        const double vdd[4] = {0.0, (double)vd[1], (double)vd[2], (double)vd[3]};
        qmul_ref<OpsD>(dq, vrd, qr);
        qmul_ref<OpsD>(dq, vdd, t0);
        qmul_ref<OpsD>(dq + 4, vrd, t1);
    }
    for (int i = 0; i < 4; ++i) qd[i] = dadd(t0[i], t1[i]);
    // dual_quaternion_conjugate (core/util.py:299-304): [w,-x,-y,-z,-dw,dx,dy,dz] as float64
    const double cr[4] = {dq[0], -dq[1], -dq[2], -dq[3]};
    const double cd[4] = {-dq[4], dq[5], dq[6], dq[7]};
    qmul_ref<OpsD>(qr, cd, t0);
    qmul_ref<OpsD>(qd, cr, t1);
    out[0] = dadd(t0[1], t1[1]);
    out[1] = dadd(t0[2], t1[2]);
    out[2] = dadd(t0[3], t1[3]);
}

// Closed form of dqb_warp for a float64 dq (possibly non-unit): the dual part of dq * (1 + eps p) * conj(dq) is
//   (w^2 - |v|^2) p + 2 (v.p) v + 2 w (v x p) + 2 (w dv - dw v + v x dv).
// Same value as the literal product chain of dqb_warp_ref up to float64 rounding order (<= 1e-15 relative; checked
// against the oracle by the tests); about a third of its operations.  The float32 rounding of the point (Q3) is kept.
DFB_HDN void dqb_warp_closed(const double* q, const double* pos, double* out) {
    const double p[3] = {(double)(float)pos[0], (double)(float)pos[1], (double)(float)pos[2]};
    const double w = q[0], x = q[1], y = q[2], z = q[3], dw = q[4], dx = q[5], dy = q[6], dz = q[7];
    const double s = w * w - (x * x + y * y + z * z);
    const double vp = x * p[0] + y * p[1] + z * p[2];
    const double cx = y * p[2] - z * p[1], cy = z * p[0] - x * p[2], cz = x * p[1] - y * p[0];
    out[0] = s * p[0] + 2.0 * (vp * x + w * cx + (w * dx - dw * x + (y * dz - z * dy)));
    out[1] = s * p[1] + 2.0 * (vp * y + w * cy + (w * dy - dw * y + (z * dx - x * dz)));
    out[2] = s * p[2] + 2.0 * (vp * z + w * cz + (w * dz - dw * z + (x * dy - y * dx)));
}

// core/util.py:74-76  dqb_warp_normal: real part only, promoted to float64 by np.append.
DFB_HDN void dqb_warp_normal_ref(const double* dq, const double* n, double* out) {
    const double rq[8] = {dq[0], dq[1], dq[2], dq[3], 0.0, 0.0, 0.0, 0.0};
    dqb_warp_ref(rq, false, n, out);
}

// la.norm(a - b) for float32 3-vectors: float32 subtraction, cblas_sdot (float32 products summed in a
// double, rounded to float32 -- OpenBLAS x86-64 tail loop, see oracle/dq.py:norm3_like_la), float32 sqrt.
DFB_HD float norm3_f32_ref(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = fsub(ax, bx), dy = fsub(ay, by), dz = fsub(az, bz);
    const double s = dadd(dadd((double)fmul(dx, dx), (double)fmul(dy, dy)), (double)fmul(dz, dz));
    return fsqrt((float)s);
}

// core/fusion.py:527-551 dq_blend (dmax=None) for a float32 point and float32 node data.
// ids: k node indices; node_pos [n][3], node_dq [n][8], node_w [n] (float32 storage of dg_w).
// Also returns the Q4 mean node distance (core/fusion.py:180-183) when wi_out != nullptr.
// rec (optional): the packed node records [n][3] float4 = (pos.xyz, coef), dq[0..3], dq[4..7] -- the same float32 values as
// node_pos / node_dq, fetched with three 16-byte loads per node instead of eleven scalar ones (the exact pass of the a3 path).
template <int KT = 0>   // KT > 0: compile-time neighbour count (loop unrolled: the k exp() chains overlap)
DFB_HDN void dq_blend_ref(const float* p, const int* ids, int k_rt, const float* node_pos, const float* node_dq,
                          const float* node_w, double* se3, float* wi_out, double* n2_out = nullptr, const float4* rec = nullptr) {
    double b[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    float wi = 0.f;
    const int k = KT > 0 ? KT : k_rt;
    double wts[KT > 0 ? KT : 1];
    if (KT > 0) {
#pragma unroll
        for (int i = 0; i < (KT > 0 ? KT : 1); ++i) {
            float nx, ny, nz;
            if (rec) { const float4 r0 = rec[3 * (size_t)ids[i]]; nx = r0.x; ny = r0.y; nz = r0.z; }
            else { const float* np_ = node_pos + 3 * (size_t)ids[i]; nx = np_[0]; ny = np_[1]; nz = np_[2]; }
            const float nrm = norm3_f32_ref(p[0], p[1], p[2], nx, ny, nz);
            const float q = fdiv(nrm, fmul(2.0f, node_w[ids[i]]));
            wts[i] = exp((double)fmul(-1.0f, fmul(q, q)));
        }
    }
#pragma unroll
    for (int i = 0; i < k; ++i) {
        const int id = ids[i];
        float npx = 0.f, npy = 0.f, npz = 0.f;
        if (!(KT > 0) || wi_out) {
            if (rec) { const float4 r0 = rec[3 * (size_t)id]; npx = r0.x; npy = r0.y; npz = r0.z; }
            else { const float* np_ = node_pos + 3 * (size_t)id; npx = np_[0]; npy = np_[1]; npz = np_[2]; }
        }
        double w;
        if (KT > 0) {
            w = wts[KT > 0 ? i : 0];
        } else {
            const float nrm = norm3_f32_ref(p[0], p[1], p[2], npx, npy, npz);
            const float two_w = fmul(2.0f, node_w[id]);
            const float q = fdiv(nrm, two_w);
            const float arg = fmul(-1.0f, fmul(q, q));
            w = exp((double)arg);
        }
        const float wf = (float)w;  // `w * dg_dq`: python float is weak -> product in float32
        float dqi[8];
        if (rec) {
            const float4 r1 = rec[3 * (size_t)id + 1], r2 = rec[3 * (size_t)id + 2];
            dqi[0] = r1.x; dqi[1] = r1.y; dqi[2] = r1.z; dqi[3] = r1.w; dqi[4] = r2.x; dqi[5] = r2.y; dqi[6] = r2.z; dqi[7] = r2.w;
        } else {
            const float* dq_ = node_dq + 8 * (size_t)id;
            for (int c = 0; c < 8; ++c) dqi[c] = dq_[c];
        }
        for (int c = 0; c < 8; ++c) b[c] = dadd(b[c], (double)fmul(wf, dqi[c]));
        if (wi_out) {
            // la.norm(node - pos)/len(locations), accumulated in float32 starting from python 0
            const float nrm2 = norm3_f32_ref(npx, npy, npz, p[0], p[1], p[2]);
            const float term = fdiv(nrm2, (float)k);
            wi = (i == 0) ? term : fadd(wi, term);
        }
    }
    if (wi_out) *wi_out = wi;
    double s = 0.0;
    for (int c = 0; c < 8; ++c) s = dadd(s, dmul(b[c], b[c]));
    if (n2_out) {
        // caller applies the closed form W(b,p)/|b|^2 (== W(b/|b|, p), W being quadratic in the dq): one division instead
        // of a square root and eight; same value up to float64 rounding order
        *n2_out = s;
        if (s == 0.0) {
            se3[0] = 1.0;
            for (int c = 1; c < 8; ++c) se3[c] = 0.0;
            *n2_out = 1.0;
        } else {
            for (int c = 0; c < 8; ++c) se3[c] = b[c];
        }
        return;
    }
    const double nrm8 = dsqrt(s);
    if (nrm8 == 0.0) {
        se3[0] = 1.0;
        for (int c = 1; c < 8; ++c) se3[c] = 0.0;
        return;
    }
    for (int c = 0; c < 8; ++c) se3[c] = ddiv(b[c], nrm8);
}

// core/fusion.py:502-520 warp(pos, dqs, locations, normal, m_lw) for a float32 point.
template <int KT = 0>
DFB_HDN void warp_ref(const float* p, const float* nrm_in, const int* ids, int k, const float* node_pos,
                      const float* node_dq, const float* node_w, const double* lw, bool has_lw, bool lw_is_f32,
                      double* out_p, double* out_n, float* wi_out, bool closed_form = false, const float4* rec = nullptr) {
    double pd[3] = {(double)p[0], (double)p[1], (double)p[2]};
    double se3[8];
    if (k > 0) {
        if (closed_form && !(nrm_in && out_n)) {
            double n2;
            dq_blend_ref<KT>(p, ids, k, node_pos, node_dq, node_w, se3, wi_out, &n2, rec);
            dqb_warp_closed(se3, pd, out_p);
            const double inv = 1.0 / n2;
            out_p[0] *= inv; out_p[1] *= inv; out_p[2] *= inv;
        } else {
            dq_blend_ref<KT>(p, ids, k, node_pos, node_dq, node_w, se3, wi_out, nullptr, rec);
            if (closed_form) dqb_warp_closed(se3, pd, out_p);
            else dqb_warp_ref(se3, false, pd, out_p);
        }
    } else {
        out_p[0] = pd[0]; out_p[1] = pd[1]; out_p[2] = pd[2];
    }
    if (has_lw) {
        double t[3] = {out_p[0], out_p[1], out_p[2]};
        if (closed_form && !lw_is_f32) dqb_warp_closed(lw, t, out_p);   // a float32 lw multiplies in float32: literal path
        else dqb_warp_ref(lw, lw_is_f32, t, out_p);
    }
    if (nrm_in && out_n) {
        double nd[3] = {(double)nrm_in[0], (double)nrm_in[1], (double)nrm_in[2]};
        if (k > 0) dqb_warp_normal_ref(se3, nd, out_n);
        else { out_n[0] = nd[0]; out_n[1] = nd[1]; out_n[2] = nd[2]; }
        if (has_lw) {
            double t[3] = {out_n[0], out_n[1], out_n[2]};
            dqb_warp_normal_ref(lw, t, out_n);
        }
    }
}

// 3-term dot product as numpy's matmul evaluates a 3x3 @ 3 / 3x4 @ 4 product row (left to right).
DFB_HD double dot3_ref(const double* r, double a, double b, double c) {
    return dadd(dadd(dmul(r[0], a), dmul(r[1], b)), dmul(r[2], c));
}
DFB_HD double dot4_ref(const double* r, double a, double b, double c, double d) {
    return dadd(dadd(dadd(dmul(r[0], a), dmul(r[1], b)), dmul(r[2], c)), dmul(r[3], d));
}

// fast-tier transcendental / reciprocal: raw MUFU ops on the device (2 ulp; the error margins have > 30 ulp head-room)
DFB_HD float fast_exp2(float x) {
#if defined(__CUDA_ARCH__)
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
#else
    return exp2f(x);
#endif
}
DFB_HD float fast_rcp(float x) {
#if defined(__CUDA_ARCH__)
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
#else
    return 1.0f / x;
#endif
}

// fp32 clamped update of FusionDM.fuseDepths: v' = (scale*v*w + tdist)/(scale*(w+1)); w' = min(w+1, wmax)
// The quotient uses the MUFU reciprocal (<= 1 ulp): |v'| <= tdist, so the result is within 3 ulp = 4e-7 tdist of the
// float64 value the reference stores, against the 1e-5 tdist budget.
// BOTH tiers evaluate a clamped update with this function (the exact tier once its float64 decision is "tl >= tdist"), so a
// voxel gets the same bits whichever tier resolves it -- slabs / brick grids of any decomposition concatenate to the
// single-volume result bit for bit (SURVEY 8e).
DFB_HD void clamp_update(float& v, float& w, float tdist, float wmax, float scale) {
    // explicit roundings: the compiler must not contract / reassociate this differently at its two call sites
#if defined(__CUDA_ARCH__)
    v = __fmul_rn(__fmaf_rn(__fmul_rn(scale, v), w, tdist), fast_rcp(__fmul_rn(scale, __fadd_rn(1.0f, w))));
#else
    v = fmul(fmaf(fmul(scale, v), w, tdist), fast_rcp(fmul(scale, fadd(1.0f, w))));
#endif
    w = fminf(fadd(1.0f, w), wmax);
}

// Per-voxel body of FusionDM.fuseDepths from project_to_pixel on (core/fusion_dm.py:194-210,
// core/util.py:312-320).  v,w: running float64 state (in/out).  Returns bit0 = updated, bit1 = in frustum.
DFB_HDN int project_fuse_ref(const double* lpos, const float* depth, int rows, int cols, const double* K,
                             const double* Kinv, double tdist, double scale, double wmax, double* v, double* w) {
    const double p0 = dot3_ref(K, lpos[0], lpos[1], lpos[2]);
    const double p1 = dot3_ref(K + 3, lpos[0], lpos[1], lpos[2]);
    const double p2 = dot3_ref(K + 6, lpos[0], lpos[1], lpos[2]);
    if (p2 == 0.0) return 0;
    const double u = ddiv(p0, p2), vv = ddiv(p1, p2);
    if (!(u >= 0.0 && u < (double)(cols - 1) && vv >= 0.0 && vv < (double)(rows - 1))) return 0;
    const long ui = (long)drint(u), vi = (long)drint(vv);
    const double z = -1.0 * (double)depth[(size_t)vi * cols + ui];
    if (!(z > 0.0)) return 2;
    const double c2 = dot3_ref(Kinv + 6, dmul(z, u), dmul(z, vv), dmul(z, 1.0));
    const double tl = dsub(c2, lpos[2]);
    if (!(tl > -1.0 * tdist)) return 2;
    if (!(tl < tdist)) {
        // min(tdist, tl) = tdist: the clamped running average, evaluated exactly like the fast tier does (see clamp_update)
        float vf = (float)*v, wf = (float)*w;
        clamp_update(vf, wf, (float)tdist, (float)wmax, (float)scale);
        *v = (double)vf;
        *w = (double)wf;
        return 3;
    }
    const double m = tl;  // python min(tdist, tl)
    const double wt = *w;
    *v = ddiv(dadd(dmul(dmul(scale, *v), wt), dmul(m, 1.0)), dmul(scale, dadd(1.0, wt)));
    const double s = dadd(1.0, wt);
    *w = (wmax < s) ? wmax : s;  // python min(wi + wi_t, wmax)
    return 3;
}

// Projective data association of one warped canonical point w / normal m (float64, from warp_ref) against n_views depth maps
// (SURVEY 8f rank 1; the contract is oracle/assoc.py).  Per view v, in ascending order: camera frame l = E_v [w,1], ln = R_v m
// (w, m when E == nullptr); front-facing ln.l < 0; projection as project_fuse_ref plus a one-pixel border ring; the centre depth
// and its four 4-neighbours valid (> 0) and within max_distance of it; live point c = Kinv [z u, z v, z] at the integer pixel,
// live normal g = (P(u+1) - P(u-1)) x (P(v+1) - P(v-1)) turned to face the camera; gates |l - c|^2 <= max_distance^2 and
// ln.g >= min_normal_dot |ln| |g|; cost |ln.(l - c)|, smallest cost wins (strict <: ties keep the lower view).
// Returns the view (-1: none); cost_out = cost (+inf: none), corr_out = R_v^T (c - t_v) (0: none).
// depth[v]: [rows][cols] float32, negative depth, 0 = no data.  E: [n_views][12] row-major 3x4 or nullptr.
DFB_HDN int assoc_projective_ref(const double* w, const double* m, const float* const* depth, int n_views, int rows, int cols,
                                 const double* K, const double* Kinv, const double* E, double max_distance, double min_normal_dot,
                                 double* cost_out, double* corr_out) {
    int best = -1;
    double best_cost = INFINITY, bc[3] = {0.0, 0.0, 0.0};
    const double md2 = dmul(max_distance, max_distance);
    for (int v = 0; v < n_views; ++v) {
        const double* Ev = E ? E + 12 * v : nullptr;
        double l[3], ln[3];
        for (int r = 0; r < 3; ++r) {
            l[r] = Ev ? dot4_ref(Ev + 4 * r, w[0], w[1], w[2], 1.0) : w[r];
            ln[r] = Ev ? dot3_ref(Ev + 4 * r, m[0], m[1], m[2]) : m[r];
        }
        if (!(dot3_ref(ln, l[0], l[1], l[2]) < 0.0)) continue;
        const double p0 = dot3_ref(K, l[0], l[1], l[2]);
        const double p1 = dot3_ref(K + 3, l[0], l[1], l[2]);
        const double p2 = dot3_ref(K + 6, l[0], l[1], l[2]);
        if (p2 == 0.0) continue;
        const double u = ddiv(p0, p2), vv = ddiv(p1, p2);
        if (!(u >= 0.0 && u < (double)(cols - 1) && vv >= 0.0 && vv < (double)(rows - 1))) continue;
        const long ui = (long)drint(u), vi = (long)drint(vv);
        if (ui < 1 || ui > cols - 2 || vi < 1 || vi > rows - 2) continue;
        const float* D = depth[v];
        // centre, u-1, u+1, v-1, v+1
        const long pu[5] = {ui, ui - 1, ui + 1, ui, ui};
        const long pv[5] = {vi, vi, vi, vi - 1, vi + 1};
        double z[5];
        bool ok = true;
        for (int j = 0; j < 5 && ok; ++j) {
            z[j] = -1.0 * (double)D[(size_t)pv[j] * cols + pu[j]];
            ok = z[j] > 0.0 && (j == 0 || fabs(dsub(z[j], z[0])) <= max_distance);
        }
        if (!ok) continue;
        double P[5][3];
        for (int j = 0; j < 5; ++j) {
            const double a = dmul(z[j], (double)pu[j]), b = dmul(z[j], (double)pv[j]), c2 = dmul(z[j], 1.0);
            for (int r = 0; r < 3; ++r) P[j][r] = dot3_ref(Kinv + 3 * r, a, b, c2);
        }
        const double* c = P[0];
        const double du[3] = {dsub(P[2][0], P[1][0]), dsub(P[2][1], P[1][1]), dsub(P[2][2], P[1][2])};
        const double dv[3] = {dsub(P[4][0], P[3][0]), dsub(P[4][1], P[3][1]), dsub(P[4][2], P[3][2])};
        double g[3] = {dsub(dmul(du[1], dv[2]), dmul(du[2], dv[1])), dsub(dmul(du[2], dv[0]), dmul(du[0], dv[2])),
                       dsub(dmul(du[0], dv[1]), dmul(du[1], dv[0]))};
        const double gc = dot3_ref(g, c[0], c[1], c[2]);
        if (gc == 0.0) continue;
        if (gc > 0.0) { g[0] = -g[0]; g[1] = -g[1]; g[2] = -g[2]; }
        const double d[3] = {dsub(l[0], c[0]), dsub(l[1], c[1]), dsub(l[2], c[2])};
        if (!(dot3_ref(d, d[0], d[1], d[2]) <= md2)) continue;
        const double nl = dsqrt(dot3_ref(ln, ln[0], ln[1], ln[2])), ng = dsqrt(dot3_ref(g, g[0], g[1], g[2]));
        if (!(dot3_ref(ln, g[0], g[1], g[2]) >= dmul(dmul(min_normal_dot, nl), ng))) continue;
        const double cost = fabs(dot3_ref(ln, d[0], d[1], d[2]));
        if (!(cost < best_cost)) continue;
        best = v;
        best_cost = cost;
        if (Ev) {
            const double e[3] = {dsub(c[0], Ev[3]), dsub(c[1], Ev[7]), dsub(c[2], Ev[11])};
            for (int j = 0; j < 3; ++j) bc[j] = dadd(dadd(dmul(Ev[j], e[0]), dmul(Ev[4 + j], e[1])), dmul(Ev[8 + j], e[2]));
        } else {
            bc[0] = c[0]; bc[1] = c[1]; bc[2] = c[2];
        }
    }
    *cost_out = best_cost;
    corr_out[0] = bc[0]; corr_out[1] = bc[1]; corr_out[2] = bc[2];
    return best;
}

// core/util.py:102-137 interpolate_tsdf on a float32 live volume; returns false for "None".
DFB_HDN bool interpolate_tsdf_ref(const double* pos, const float* t, int rx, int ry, int rz, double* out) {
    const double mn = fmin(fmin(pos[0], pos[1]), pos[2]);
    if (!(mn >= 0.0) || pos[0] > rx - 1 || pos[1] > ry - 1 || pos[2] > rz - 1) return false;
    if (!(pos[0] == pos[0] && pos[1] == pos[1] && pos[2] == pos[2])) return false;
    const double fx = floor(pos[0]), fy = floor(pos[1]), fz = floor(pos[2]);
    const long x0 = (long)fx, y0 = (long)fy, z0 = (long)fz;
    const long x1 = (long)ceil(pos[0]), y1 = (long)ceil(pos[1]), z1 = (long)ceil(pos[2]);
    const double xd = dsub(pos[0], fx), yd = dsub(pos[1], fy), zd = dsub(pos[2], fz);
#define DFB_T(a, b, c) ((double)t[((size_t)(a) * ry + (size_t)(b)) * rz + (size_t)(c)])
    const double c000 = DFB_T(x0, y0, z0), c100 = DFB_T(x1, y0, z0), c001 = DFB_T(x0, y1, z0), c101 = DFB_T(x1, y1, z0);
    const double c010 = DFB_T(x0, y0, z1), c110 = DFB_T(x1, y0, z1), c011 = DFB_T(x0, y1, z1), c111 = DFB_T(x1, y1, z1);
#undef DFB_T
    const double ix = dsub(1.0, xd), iy = dsub(1.0, yd), iz = dsub(1.0, zd);
    const double c00 = dadd(dmul(c000, ix), dmul(c100, xd));
    const double c01 = dadd(dmul(c001, ix), dmul(c101, xd));
    const double c10 = dadd(dmul(c010, ix), dmul(c110, xd));
    const double c11 = dadd(dmul(c011, ix), dmul(c111, xd));
    const double c0 = dadd(dmul(c00, iy), dmul(c10, yd));  // Q1: y/z weights swapped, as in the reference
    const double c1 = dadd(dmul(c01, iy), dmul(c11, yd));
    *out = dadd(dmul(c0, iz), dmul(c1, zd));
    return true;
}

// Fusion.updateTSDF value update (core/fusion.py:180-190); k==0: FusionDM.updateTSDF (:310-313).
// wi: Q4 float32 mean node distance (ignored for k==0).  Returns true (mask) when updated.
DFB_HD bool volume_fuse_ref(bool valid, double tl, float wi_f, int k, double tdist, double wmax, double* v, double* w) {
    if (!valid || !(tl > -1.0 * tdist)) return false;
    if (k == 0) {
        const double wt = *w;
        const double m = (tl < tdist) ? tl : tdist;
        *v = ddiv(dadd(dmul(*v, wt), dmul(m, 1.0)), dadd(1.0, wt));
        const double s = dadd(1.0, wt);
        *w = (wmax < s) ? wmax : s;
        return true;
    }
    const double wi = (double)wi_f;
    const double wt = (*w == 0.0) ? wi : *w;
    // `min(tdist, tl) * wi`: tdist is a python float (weak) -> float32 product when clamped
    const double term = (tl < tdist) ? dmul(tl, wi) : (double)fmul((float)tdist, wi_f);
    *v = ddiv(dadd(dmul(*v, wt), term), dadd(wi, wt));
    const double s = dadd(wi, wt);
    *w = (wmax < s) ? wmax : s;
    return true;
}

// ---------------------------------------------------------------------------------------------
// fast tier (fp32)
// ---------------------------------------------------------------------------------------------
struct Affine34 {  // row-major 3x4, fp32
    float m[12];
};

// closed form of dq * [1,0,0,0,0,p] * conj(dq) for a NON-unit dq (Q2): out = Q(b,p) (caller divides by |b|^2)
DFB_HD void dq_apply_unnormalised(const float* b, float px, float py, float pz, float* o) {
    const float w = b[0], x = b[1], y = b[2], z = b[3], dw = b[4], dx = b[5], dy = b[6], dz = b[7];
    const float vv = x * x + y * y + z * z;
    const float s = w * w - vv;
    const float vp = x * px + y * py + z * pz;
    const float cx = y * pz - z * py, cy = z * px - x * pz, cz = x * py - y * px;
    const float tx = w * dx - dw * x + (y * dz - z * dy);
    const float ty = w * dy - dw * y + (z * dx - x * dz);
    const float tz = w * dz - dw * z + (x * dy - y * dx);
    o[0] = s * px + 2.f * (vp * x + w * cx + tx);
    o[1] = s * py + 2.f * (vp * y + w * cy + ty);
    o[2] = s * pz + 2.f * (vp * z + w * cz + tz);
}

// dq (double, possibly non-unit) -> the affine map p -> dqb_warp(dq, p)
inline void dq_to_affine(const double* q, double* A /*12*/) {
    const double w = q[0], x = q[1], y = q[2], z = q[3], dw = q[4], dx = q[5], dy = q[6], dz = q[7];
    const double s = w * w - (x * x + y * y + z * z);
    // rotation-like part: s*I + 2 v v^T + 2 w [v]x
    A[0] = s + 2 * x * x;        A[1] = 2 * (x * y - w * z);  A[2] = 2 * (x * z + w * y);
    A[4] = 2 * (x * y + w * z);  A[5] = s + 2 * y * y;        A[6] = 2 * (y * z - w * x);
    A[8] = 2 * (x * z - w * y);  A[9] = 2 * (y * z + w * x);  A[10] = s + 2 * z * z;
    A[3] = 2 * (w * dx - dw * x + (y * dz - z * dy));
    A[7] = 2 * (w * dy - dw * y + (z * dx - x * dz));
    A[11] = 2 * (w * dz - dw * z + (x * dy - y * dx));
}

}  // namespace dfb
