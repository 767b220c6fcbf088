// Device helpers shared by the two flavours of the fused column kernel
// (pgw_timestep.cu: per-thread cp.async flavour, pgw_column_tma.cu: TMA flavour).
#pragma once
#include <cuda.h>
#include <limits.h>

#include "pgw_common.cuh"

namespace pgw {

constexpr int kColumnThreads = 128;  // columns per CTA (= TMA box width)
#ifndef PGW_NODE_L2_AHEAD
#define PGW_NODE_L2_AHEAD 2
#endif
constexpr int kL2Ahead = PGW_NODE_L2_AHEAD;   // delta nodes pulled into L2 this many steps ahead of their use

// Raw (before, after) pair of a 2-D delta; all pairs of a column are loaded up front so
// that their DRAM latencies overlap, then blended.
struct Pair2 { float lo, hi; };
__device__ __forceinline__ Pair2 load_pair(const pgw_tslab &s, uint32_t off) {
    Pair2 r;
    r.lo = __ldg(s.lo + off);
    r.hi = __ldg(s.hi + off);      // == lo slab for an exact hit (x_new == 0)
    return r;
}
// scipy interp1d._call_linear with x = [0, x_hi]: slope * x_new + y_lo (float64)
__device__ __forceinline__ double blend_f64(const pgw_tslab &s, const Pair2 &v) {
    const double lo = (double)v.lo;
    if (s.x_new == 0.0) return lo;
    return ((double)v.hi - lo) / s.x_hi * s.x_new + lo;
}
// float32 weight of the `hi` slab; 0 for an exact hit
__device__ __forceinline__ float slab_weight(const pgw_tslab &s) {
    return (s.x_new == 0.0) ? 0.0f : (float)(s.x_new / s.x_hi);
}
__device__ __forceinline__ float blend_f32(float w, float x0, float x1) {
    return (w == 0.0f) ? x0 : fmaf(w, x1 - x0, x0);
}

__device__ __forceinline__ float fast_rcp(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float fast_lg2(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float fast_ex2(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// MUFU.RCP64H: >= 20 good bits of 1/x in one instruction
__device__ __forceinline__ double rcp64_approx(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
}

// ln(pb/pt), pb >= pt > 0, in float64 without a float64 log or divide:
// 2 atanh(s), s = (pb-pt)/(pb+pt) = 2 s (1 + s^2/3 + s^4/5 + s^6/7 + ...).
// Truncated after s^6/7 the relative error is s^8/9 < 2e-11 for s < 0.06, far below
// the 1e-9 the ps iteration needs; all adjacent ERA5 half levels below ~100 hPa
// have s < 0.05.  FAST = the host has verified s < 0.06 for every layer the
// iteration can touch, so the exact-log branch is compiled out.
struct LnConst { double c3, c5, c7; };

template <bool FAST>
__device__ __forceinline__ double ln_ratio(double pb, double pt, const LnConst &k) {
    const double d = pb - pt;
    const double sm = pb + pt;
    double r = rcp64_approx(sm);
    r = fma(r, fma(-sm, r, 1.0), r);            // one Newton step: ~1e-12 relative
    const double s = d * r;
    if (!FAST) { if (s > 0.06) return log(pb / pt); }
    const double s2 = s * s;
    double poly = fma(s2, k.c7, k.c5);
    poly = fma(s2, poly, k.c3);
    poly = fma(s2, poly, 2.0);
    return s * poly;
}

// PGW_FLAG_REF_DTYPES: ln(pb) - ln(pt) the way numpy forms it (functions.py:136-138: the difference of two float64
// logs, each within an ulp of ln p ~ 11.5, i.e. an absolute error of ~2e-15) to that same accuracy: exact
// division, series to s^10 (relative truncation error s^12/13 < 2e-16 for s < 0.06), the exact logs otherwise.
// The value is then rounded into a float32 running sum (ulp 0.0078 m2/s2), so what matters is that it sits
// within ~1e-10 m2/s2 of numpy's: a different rounding of the sum then happens once in ~1e7 levels.
__device__ __forceinline__ double ln_ratio_ref(double pb, double pt) {
    const double s = (pb - pt) / (pb + pt);
    if (!(fabs(s) < 0.06)) return log(pb) - log(pt);
    const double s2 = s * s;
    double poly = fma(s2, 2.0 / 11.0, 2.0 / 9.0);
    poly = fma(s2, poly, 2.0 / 7.0);
    poly = fma(s2, poly, 2.0 / 5.0);
    poly = fma(s2, poly, 2.0 / 3.0);
    poly = fma(s2, poly, 2.0);
    return s * poly;
}

// `zero` (== 0) that carries a data dependency on four registers: orders a following
// asynchronous operation behind the instructions that produced / read them.
__device__ __forceinline__ int reg_fence(float x0, float x1, float x2, float x3) {
    int z;
    asm volatile("{\n\t.reg .b32 t;\n\tor.b32 t, %1, %2;\n\tor.b32 t, t, %3;\n\tor.b32 t, t, %4;\n\t"
                 "and.b32 %0, t, 0;\n\t}"
                 : "=r"(z) : "r"(__float_as_int(x0)), "r"(__float_as_int(x1)), "r"(__float_as_int(x2)),
                   "r"(__float_as_int(x3)));
    return z;
}

// Saturation vapour pressure of the ERA and the PGW state (functions.py:74-105), RELHUM of
// the ERA state (:107-116) + delta, back to vapour pressure (:123); T - 273.16 is formed from
// the exact T - 273 so that T_pgw is never rounded to fp32.  `cold` (warp-uniform): every
// temperature involved is <= 250.16 K, ice only (alpha == 0 exactly).  The general form is
// branch free: both exponentials, alpha from selects (exactly 1 / 0 outside the mixed band).
// Returns the vapour pressure of the PGW state.
__device__ __forceinline__ float thermo_e_pgw(bool cold, float p, float t, float q, float dta, float dhur) {
    const float tm273 = t - 273.0f;
    const float dTe = tm273 - 0.16f, tkp = tm273 + dta, dTp = tm273 + (dta - 0.16f);
    constexpr float kCw = 17.502f * 1.4426950408889634f, kCi = 22.587f * 1.4426950408889634f;
    float es_e, es_p;
    if (cold) {
        const float de = tm273 + (273.0f + 0.7f), dp = tkp + (273.0f + 0.7f);
        const float rr = fast_rcp(de * dp);               // one reciprocal for both states
        es_e = 611.21f * fast_ex2(kCi * dTe * (rr * dp));
        es_p = 611.21f * fast_ex2(kCi * dTp * (rr * de));
    } else {
        const float dew = tm273 + (273.0f - 32.19f), dei = tm273 + (273.0f + 0.7f);
        const float dpw = tkp + (273.0f - 32.19f), dpi = tkp + (273.0f + 0.7f);
        const float pe = dew * dei, pp = dpw * dpi;
        const float rr = fast_rcp(pe * pp);               // one reciprocal for all four quotients
        const float re = rr * pp, rp = rr * pe;           // 1/pe, 1/pp
        const float ew_e = fast_ex2(kCw * dTe * (re * dei)), ei_e = fast_ex2(kCi * dTe * (re * dew));
        const float ew_p = fast_ex2(kCw * dTp * (rp * dpi)), ei_p = fast_ex2(kCi * dTp * (rp * dpw));
        const float r_e = (dTe + 23.0f) * (1.0f / 23.0f), r_p = (dTp + 23.0f) * (1.0f / 23.0f);
        const float al_e = dTe >= 0.0f ? 1.0f : (dTe <= -23.0f ? 0.0f : r_e * r_e);   // NaN stays NaN
        const float al_p = dTp >= 0.0f ? 1.0f : (dTp <= -23.0f ? 0.0f : r_p * r_p);
        es_e = 611.21f * (al_e * ew_e + (1.0f - al_e) * ei_e);
        es_p = 611.21f * (al_p * ew_p + (1.0f - al_p) * ei_p);
    }
    const float rh_pgw = fmaf(100.0f * q * p, fast_rcp((0.622f + 0.378f * q) * es_e), dhur);
    return rh_pgw * 0.01f * es_p;
}
// The same for TWO levels at once with the packed float32 pair instructions of sm_100 (FADD2 / FMUL2 / FFMA2):
// the sweep handles level pairs, whose thermodynamics are two independent, identical instruction sequences; packed,
// every add/multiply of the pair is one issue slot instead of two (MUFU and the selects stay scalar).  Same
// operations in the same order per lane as thermo_e_pgw.
__device__ __forceinline__ float2 thermo_e_pgw_x2(bool cold, float2 p, float2 t, float2 q, float2 dta, float2 dhur) {
    const auto S = [](float a) { return make_float2(a, a); };
    const float2 tm273 = __fadd2_rn(t, S(-273.0f));
    const float2 dTe = __fadd2_rn(tm273, S(-0.16f)), tkp = __fadd2_rn(tm273, dta);
    const float2 dTp = __fadd2_rn(tm273, __fadd2_rn(dta, S(-0.16f)));
    constexpr float kCw = 17.502f * 1.4426950408889634f, kCi = 22.587f * 1.4426950408889634f;
    float2 es_e, es_p;
    if (cold) {
        const float2 de = __fadd2_rn(tm273, S(273.0f + 0.7f)), dp = __fadd2_rn(tkp, S(273.0f + 0.7f));
        const float2 dd = __fmul2_rn(de, dp);
        const float2 rr = make_float2(fast_rcp(dd.x), fast_rcp(dd.y));
        const float2 ae = __fmul2_rn(__fmul2_rn(S(kCi), dTe), __fmul2_rn(rr, dp));
        const float2 ap = __fmul2_rn(__fmul2_rn(S(kCi), dTp), __fmul2_rn(rr, de));
        es_e = __fmul2_rn(S(611.21f), make_float2(fast_ex2(ae.x), fast_ex2(ae.y)));
        es_p = __fmul2_rn(S(611.21f), make_float2(fast_ex2(ap.x), fast_ex2(ap.y)));
    } else {
        const float2 dew = __fadd2_rn(tm273, S(273.0f - 32.19f)), dei = __fadd2_rn(tm273, S(273.0f + 0.7f));
        const float2 dpw = __fadd2_rn(tkp, S(273.0f - 32.19f)), dpi = __fadd2_rn(tkp, S(273.0f + 0.7f));
        const float2 pe = __fmul2_rn(dew, dei), pp = __fmul2_rn(dpw, dpi);
        const float2 pq = __fmul2_rn(pe, pp);
        const float2 rr = make_float2(fast_rcp(pq.x), fast_rcp(pq.y));
        const float2 re = __fmul2_rn(rr, pp), rp = __fmul2_rn(rr, pe);
        const float2 cwe = __fmul2_rn(S(kCw), dTe), cie = __fmul2_rn(S(kCi), dTe);
        const float2 cwp = __fmul2_rn(S(kCw), dTp), cip = __fmul2_rn(S(kCi), dTp);
        const float2 a1 = __fmul2_rn(cwe, __fmul2_rn(re, dei)), a2 = __fmul2_rn(cie, __fmul2_rn(re, dew));
        const float2 a3 = __fmul2_rn(cwp, __fmul2_rn(rp, dpi)), a4 = __fmul2_rn(cip, __fmul2_rn(rp, dpw));
        const float2 ew_e = make_float2(fast_ex2(a1.x), fast_ex2(a1.y)), ei_e = make_float2(fast_ex2(a2.x), fast_ex2(a2.y));
        const float2 ew_p = make_float2(fast_ex2(a3.x), fast_ex2(a3.y)), ei_p = make_float2(fast_ex2(a4.x), fast_ex2(a4.y));
        const float2 r_e = __fmul2_rn(__fadd2_rn(dTe, S(23.0f)), S(1.0f / 23.0f));
        const float2 r_p = __fmul2_rn(__fadd2_rn(dTp, S(23.0f)), S(1.0f / 23.0f));
        const float2 q_e = __fmul2_rn(r_e, r_e), q_p = __fmul2_rn(r_p, r_p);
        const auto sel = [](float dT, float sq) { return dT >= 0.0f ? 1.0f : (dT <= -23.0f ? 0.0f : sq); };   // NaN stays NaN
        const float2 al_e = make_float2(sel(dTe.x, q_e.x), sel(dTe.y, q_e.y));
        const float2 al_p = make_float2(sel(dTp.x, q_p.x), sel(dTp.y, q_p.y));
        const float2 one = S(1.0f);
        const float2 be = __fadd2_rn(one, make_float2(-al_e.x, -al_e.y)), bp = __fadd2_rn(one, make_float2(-al_p.x, -al_p.y));
        es_e = __fmul2_rn(S(611.21f), __ffma2_rn(al_e, ew_e, __fmul2_rn(be, ei_e)));
        es_p = __fmul2_rn(S(611.21f), __ffma2_rn(al_p, ew_p, __fmul2_rn(bp, ei_p)));
    }
    const float2 den = __fmul2_rn(__ffma2_rn(S(0.378f), q, S(0.622f)), es_e);
    const float2 rd = make_float2(fast_rcp(den.x), fast_rcp(den.y));
    const float2 rh = __ffma2_rn(__fmul2_rn(__fmul2_rn(S(100.0f), q), p), rd, dhur);
    return __fmul2_rn(__fmul2_rn(rh, S(0.01f)), es_p);
}
__device__ __forceinline__ bool is_cold(float t, float dta) { return fmaxf(t, t + dta) <= 250.0f; }   // conservative

// Saturation vapour pressure over water and ice (functions.py:74-105) of ONE state, given as T - 273: the
// general (not `cold`) form of thermo_e_pgw.  PGW_FLAG_REINTERP, whose levels are not swept in warp-uniform pairs.
__device__ __forceinline__ float es_water_ice(float tm273) {
    const float dT = tm273 - 0.16f;
    constexpr float kCw = 17.502f * 1.4426950408889634f, kCi = 22.587f * 1.4426950408889634f;
    const float dw = tm273 + (273.0f - 32.19f), di = tm273 + (273.0f + 0.7f);
    const float rr = fast_rcp(dw * di);
    const float ew = fast_ex2(kCw * dT * (rr * di)), ei = fast_ex2(kCi * dT * (rr * dw));
    const float r = (dT + 23.0f) * (1.0f / 23.0f);
    const float al = dT >= 0.0f ? 1.0f : (dT <= -23.0f ? 0.0f : r * r);              // NaN stays NaN
    return 611.21f * (al * ew + (1.0f - al) * ei);
}
// RELHUM of the ERA state (step_03_apply_to_era.py:91-94, functions.py:107-116) at p = akm + PS * bkm
__device__ __forceinline__ float rh_era_f32(float p, float t, float q) {
    return 100.0f * q * p * fast_rcp((0.622f + 0.378f * q) * es_water_ice(t - 273.0f));
}

// specific humidity from vapour pressure (functions.py:66-72), p = akm + ps * bkm
__device__ __forceinline__ float qv_from_e(float e, float ps, float2 m) {
    return 0.622f * e * fast_rcp(fmaf(-0.378f, e, fmaf(ps, m.y, m.x)));
}

// ---------------------------------------------------------------------------
// TMA / mbarrier primitives (sm_100a)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
#ifndef PGW_WAIT_HINT_NS
#define PGW_WAIT_HINT_NS 0
#endif
// Column-warp wait.  A failed try_wait costs three issue slots (SYNCS + 2 BRA) of an issue-bound kernel, so
// the poll may carry a suspend-time hint: the warp then sleeps in hardware until the phase completes or the
// time is up instead of returning after the (short) default limit.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
#if PGW_WAIT_HINT_NS > 0
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "PGW_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra PGW_DONE;\n\t"
        "bra PGW_WAIT;\n\t"
        "PGW_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)PGW_WAIT_HINT_NS) : "memory");
#else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "PGW_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra PGW_DONE;\n\t"
        "bra PGW_WAIT;\n\t"
        "PGW_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
#endif
}
// non-blocking probe of a phase (acquire): lets independent work sit between the probe and the branch on it
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
#ifndef PGW_PRODUCER_SLEEP_NS
#define PGW_PRODUCER_SLEEP_NS 64
#endif
#define PGW_STR2_(x) #x
#define PGW_STR_(x) PGW_STR2_(x)
// Producer-side wait: suspend in hardware and back off between polls so that the lone
// producer thread does not take issue slots from the column warps.
__device__ __forceinline__ void mbar_wait_backoff(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "PGW_WAITB:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra PGW_DONEB;\n\t"
        "nanosleep.u32 " PGW_STR_(PGW_PRODUCER_SLEEP_NS) ";\n\t"
        "bra PGW_WAITB;\n\t"
        "PGW_DONEB:\n\t}" ::"r"(smem_u32(bar)), "r"(parity), "r"(100000u) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (TMA store)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// NOTE: TMA tile coordinates must not be negative on sm_100a (illegal instruction).
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, int c0, int c1, const void *src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(src)) : "memory");
}
// pull a box into L2 only (no shared-memory slot needed)
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap *map, int c0, int c1) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

}  // namespace pgw

// ---- host-side pieces shared by pgw_timestep.cu and pgw_column_tma.cu
struct pgw_column_plan {
    bool ref;           // PGW_FLAG_REF_DTYPES
    bool tma;
    int lst, np;        // top level of the stash, number of parked levels
    size_t smem;
    bool fast;          // ln_ratio series valid for every layer the iteration can touch
    bool local;         // PGW_FLAG_LOCAL_PREF
    int ncand;          // PGW_FLAG_LOCAL_PREF: zg levels >= p_floor (candidate p_ref levels)
    bool reinterp;      // PGW_FLAG_REINTERP
};
// pgw_column_tma.cu
bool pgw_tma_eligible(const pgw_timestep_args *a, int lst_generic, int *lst_tma, size_t *smem);
int pgw_launch_column_tma(const pgw_timestep_args *a, const pgw_column_plan &plan, cudaStream_t st);
// Opt a kernel in to `smem` bytes of dynamic shared memory on the CURRENT device.  The attribute is per device
// and per kernel; `slot` (0..15) names the kernel variant in a per-device table of what has been configured.
int pgw_ensure_smem(const void *kernel, int slot, size_t smem, int np);
