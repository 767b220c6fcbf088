// Stand-alone operators of libpgw_b200 (sm_100a): the pieces of functions.py
// that the reference exposes individually (and that step_01 / user scripts call
// on their own), each behind the C ABI declared in include/pgw_b200.h.  The
// fused per-timestep pass (pgw_timestep.cu) does not call these; they exist so
// that `functions.py` is a drop-in name by name.
#include "pgw_common.cuh"

namespace pgw {

// ---------------------------------------------------------------------------
// interp_1d_for_timelatlon + interp_extrap_1d (functions.py:479-580).
// One thread per (time, column); lanes = adjacent columns -> coalesced level
// accesses.  The reference scans the source from index 0 for every target; the
// first source index with src >= x can only move up while targets ascend, so the
// scan resumes from the previous position and restarts from 0 when a target is
// smaller than its predecessor.  This returns exactly the index the full scan
// finds, for any (also non-monotone) input.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128)
interp_logp_kernel(const T *__restrict__ var, const T *__restrict__ src_p, const T *__restrict__ targ_p,
                   T *__restrict__ out, int nt, int ks, int kt, long long ncol, int src_1d, int p_is_log,
                   int mode, uint32_t *err) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)nt * ncol) return;
    const long long t = idx / ncol, c = idx - t * ncol;
    const T *v = var + t * ks * ncol + c;
    const T *sp = src_1d ? src_p : src_p + t * ks * ncol + c;
    const long long sstr = src_1d ? 1 : ncol;
    const T *tp = targ_p + t * kt * ncol + c;
    T *o = out + t * kt * ncol + c;
    auto lg = [&](T x) -> T { return p_is_log ? x : log(x); };

    unsigned bits = 0;
    if (lg(sp[(long long)(ks - 1) * sstr]) < lg(sp[0])) bits |= PGW_ERR_SRC_NOT_ASCENDING;   // :500-501
    if (lg(tp[(long long)(kt - 1) * ncol]) < lg(tp[0])) bits |= PGW_ERR_TARG_NOT_ASCENDING;  // :502-503
    if (bits) { atomicOr(err, bits); return; }

    int si = 0;                     // candidate: first index with src >= x
    T sx = lg(sp[0]);               // ln p of node si
    T sx_prev = sx;                 // ln p of node si-1 (valid when si > 0)
    T x_prev = T(0);
    bool have_prev = false;
    for (int ti = 0; ti < kt; ++ti) {
        const T x = lg(tp[(long long)ti * ncol]);
        if (have_prev && !(x >= x_prev)) { si = 0; sx = lg(sp[0]); }
        x_prev = x; have_prev = true;
        while (si < ks && !(sx >= x)) {         // NaN nodes are skipped like the reference's 'pass'
            ++si;
            sx_prev = sx;
            if (si < ks) sx = lg(sp[(long long)si * sstr]);
        }
        int i1, i2;
        bool extrap = false;
        if (si == 0 && sx > x) {                 // :530-538
            extrap = true;
            if (mode == PGW_EXTRAP_LINEAR) { i1 = 0; i2 = 1; } else { i1 = 0; i2 = 0; }
        } else if (si < ks && sx == x) {         // :540-543
            i1 = i2 = si;
        } else if (si < ks) {                    // :545-548
            i1 = si - 1; i2 = si;
        } else {                                 // :554-561
            extrap = true;
            if (mode == PGW_EXTRAP_LINEAR) { i1 = ks - 2; i2 = ks - 1; } else { i1 = i2 = ks - 1; }
        }
        T y;
        if (extrap && mode == PGW_EXTRAP_OFF) { bits |= PGW_ERR_EXTRAP_OFF; y = T(0); }
        else if (extrap && mode == PGW_EXTRAP_NAN) y = T(NAN);
        else if (i1 == i2) y = v[(long long)i1 * ncol];
        else {
            T x1, x2;
            if (i2 == si && si > 0 && si < ks) { x1 = sx_prev; x2 = sx; }
            else { x1 = lg(sp[(long long)i1 * sstr]); x2 = lg(sp[(long long)i2 * sstr]); }
            const T y1 = v[(long long)i1 * ncol], y2 = v[(long long)i2 * ncol];
            y = y1 + (x - x1) * (y2 - y1) / (x2 - x1);      // :575-578
        }
        o[(long long)ti * ncol] = y;
    }
    if (bits) atomicOr(err, bits);
}

// ---------------------------------------------------------------------------
// humidity conversions (functions.py:58-125)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void q2rh_kernel(const T *__restrict__ hus, const T *__restrict__ pa, const T *__restrict__ ta,
                            T *__restrict__ hur, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const T q = hus[i], p = pa[i];
        const T e = q * p / (T(0.622) + T(0.378) * q);
        hur[i] = e / esat_generic<T>(ta[i]) * T(100);
    }
}

template <typename T>
__global__ void rh2q_kernel(const T *__restrict__ hur, const T *__restrict__ pa, const T *__restrict__ ta,
                            T *__restrict__ hus, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const T e = hur[i] / T(100) * esat_generic<T>(ta[i]);
        hus[i] = T(0.622) * e / (pa[i] - (T(1) - T(0.622)) * e);
    }
}

// ---------------------------------------------------------------------------
// integ_geopot (functions.py:128-189): per column, float64 arithmetic.
// Pass 1 finds the half level with the smallest non-negative p_hl - p_ref
// (first occurrence, like argmin); pass 2 integrates from the surface up to it.
// ---------------------------------------------------------------------------
// T: type of the pressures, zgs and p_ref; TS: type of ta and hus -- Rd * Tv is formed in TS like in
// the reference (rd_tv in pgw_common.cuh), everything else in float64.
template <typename T, typename TS>
__global__ void __launch_bounds__(128)
integ_geopot_kernel(const T *__restrict__ pa_hl, const T *__restrict__ zgs, const TS *__restrict__ ta,
                    const TS *__restrict__ hus, const T *__restrict__ p_ref_field, double p_ref_scalar,
                    double *__restrict__ phi_ref, int nlev, long long ncol, uint32_t *err) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncol) return;
    const double p_ref = p_ref_field ? (double)p_ref_field[c] : p_ref_scalar;
    int hstar = -1;
    double best = INFINITY;
    for (int h = 0; h <= nlev; ++h) {
        double p = (double)pa_hl[(long long)h * ncol + c];
        if (!(p > 0.0)) p = 0.0001;                               // :135
        const double d = p - p_ref;
        if (d >= 0.0 && d < best) { best = d; hstar = h; }
    }
    if (hstar < 0) { atomicOr(err, PGW_ERR_PREF_BELOW_SFC); phi_ref[c] = NAN; return; }   // :162-165
    double phi = (double)zgs[c];
    double p_lo = (double)pa_hl[(long long)nlev * ncol + c];
    if (!(p_lo > 0.0)) p_lo = 0.0001;
    double ln_lo = log(p_lo);
    for (int l = nlev - 1; l >= hstar; --l) {                     // :147-152
        double p_up = (double)pa_hl[(long long)l * ncol + c];
        if (!(p_up > 0.0)) p_up = 0.0001;
        const double ln_up = log(p_up);
        phi = phi + rd_tv(ta[(long long)l * ncol + c], hus[(long long)l * ncol + c]) * (ln_lo - ln_up);
        ln_lo = ln_up;
    }
    if (hstar < 1) { phi_ref[c] = NAN; return; }                  // no full level above (KeyError in xarray)
    const double rtv_star = rd_tv(ta[(long long)(hstar - 1) * ncol + c], hus[(long long)(hstar - 1) * ncol + c]);
    phi_ref[c] = phi - rtv_star * (log(p_ref) - ln_lo);           // :174-179
}

// ---------------------------------------------------------------------------
// integrate_tos (functions.py:1145-1186)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void integrate_tos_kernel(const T *__restrict__ tos, const T *__restrict__ ts,
                                     const T *__restrict__ land, const T *__restrict__ ice,
                                     T *__restrict__ out, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const T ic = ice[i], to = tos[i], t = ts[i];
        T r = t;
        if (!isnan(ic) && !isnan(to)) {
            T fr = ic + land[i];
            fr = fr < T(0) ? T(0) : (fr > T(1) ? T(1) : fr);
            r = fr * t + (T(1) - fr) * to;
        }
        out[i] = r;
    }
}

__global__ void time_interp_kernel(const float *__restrict__ lo, const float *__restrict__ hi, double x_hi,
                                   double x_new, float *__restrict__ out, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const double a = (double)lo[i];
        out[i] = (x_new == 0.0) ? lo[i] : (float)(((double)hi[i] - a) / x_hi * x_new + a);
    }
}

__global__ void time_mean_kernel(const float *__restrict__ series, int ntime, float *__restrict__ out,
                                 long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int t = 0; t < ntime; ++t) s += (double)series[(long long)t * n + i];
        out[i] = (float)(s / (double)ntime);
    }
}

// ---------------------------------------------------------------------------
// the small humidity helpers of functions.py:58-105 as one elementwise kernel
// ---------------------------------------------------------------------------
template <typename T>
__global__ void humidity_op_kernel(int op, const T *__restrict__ x, const T *__restrict__ y,
                                   T *__restrict__ out, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        T r;
        switch (op) {
            case PGW_HUM_Q2E: r = x[i] * y[i] / (T(0.622) + T(0.378) * x[i]); break;              // :58-64
            case PGW_HUM_E2Q: r = T(0.622) * x[i] / (y[i] - (T(1) - T(0.622)) * x[i]); break;     // :66-72
            case PGW_HUM_ESAT_WATER:
                r = T(611.21) * exp(T(17.502) * (x[i] - T(273.16)) / (x[i] - T(32.19))); break;  // :74-89
            case PGW_HUM_ESAT_ICE:
                r = T(611.21) * exp(T(22.587) * (x[i] - T(273.16)) / (x[i] - T(-0.7))); break;
            default: r = esat_generic<T>(x[i]); break;                                           // :91-105
        }
        out[i] = r;
    }
}

// ---------------------------------------------------------------------------
// replace_delta_sfc applied to every column (functions.py:343-366, :396-402)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128)
replace_delta_sfc_kernel(const T *__restrict__ source_P, const T *__restrict__ ps_hist,
                         const T *__restrict__ delta, const T *__restrict__ delta_sfc,
                         T *__restrict__ out_P, T *__restrict__ out_d, int K, long long ncol, int src_1d,
                         uint32_t *err) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncol) return;
    const T *sp = src_1d ? source_P : source_P + c;
    const long long ss = src_1d ? 1 : ncol;
    const T ph = ps_hist[c], ds = delta_sfc[c];
    T pmax = -INFINITY, pmin = INFINITY;
    int sfc = -1;
    for (int k = 0; k < K; ++k) {
        const T p = sp[(long long)k * ss];
        out_P[(long long)k * ncol + c] = p;
        out_d[(long long)k * ncol + c] = delta[(long long)k * ncol + c];
        pmax = p > pmax ? p : pmax;
        pmin = p < pmin ? p : pmin;
        if (ph > p) sfc = k;                       // np.max(np.argwhere(ps_hist > source_P))
    }
    if (ph > pmax) {                               // :356-359
        out_P[(long long)(K - 1) * ncol + c] = ph;
        out_d[(long long)(K - 1) * ncol + c] = ds;
    } else if (ph < pmin || sfc < 0) {             // :360-361 and the empty argwhere of :363
        atomicOr(err, PGW_ERR_PS_HIST_RANGE);
    } else {                                       // :362-365
        for (int k = sfc; k < K; ++k) out_d[(long long)k * ncol + c] = ds;
        out_P[(long long)sfc * ncol + c] = ph;
    }
}

inline unsigned ew_grid(long long n, int block) {
    long long g = (n + block - 1) / block;
    const long long cap = 148LL * 16;          // persistent-style: 16 CTAs per SM, grid-stride loop
    return (unsigned)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace pgw

using namespace pgw;

#define PGW_REQUIRE(cond) do { if (!(cond)) return PGW_E_INVALID; } while (0)

template <typename T>
static int interp_logp_impl(const T *var, const T *src_p, const T *targ_p, T *out, int nt, int ks, int kt,
                            long long ncol, int src_1d, int p_is_log, int mode, uint32_t *err, void *stream) {
    PGW_REQUIRE(var && src_p && targ_p && out && err);
    PGW_REQUIRE(nt > 0 && ks >= 1 && kt >= 1 && ncol > 0);
    PGW_REQUIRE(mode >= PGW_EXTRAP_OFF && mode <= PGW_EXTRAP_NAN);
    PGW_REQUIRE(!(mode == PGW_EXTRAP_LINEAR && ks < 2));
    const long long total = (long long)nt * ncol;
    interp_logp_kernel<T><<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        var, src_p, targ_p, out, nt, ks, kt, ncol, src_1d, p_is_log, mode, err);
    return pgw_check_launch("interp_logp_kernel");
}

extern "C" {

int pgw_interp_logp_f64(const double *var, const double *src_p, const double *targ_p, double *out, int nt,
                        int ks, int kt, long long ncol, int src_p_is_1d, int p_is_log, int mode,
                        uint32_t *err, void *stream) {
    return interp_logp_impl<double>(var, src_p, targ_p, out, nt, ks, kt, ncol, src_p_is_1d, p_is_log, mode, err, stream);
}
int pgw_interp_logp_f32(const float *var, const float *src_p, const float *targ_p, float *out, int nt, int ks,
                        int kt, long long ncol, int src_p_is_1d, int p_is_log, int mode, uint32_t *err,
                        void *stream) {
    return interp_logp_impl<float>(var, src_p, targ_p, out, nt, ks, kt, ncol, src_p_is_1d, p_is_log, mode, err, stream);
}

#define PGW_EW3(NAME, KERNEL, T)                                                                     \
    int NAME(const T *a, const T *b, const T *c, T *o, long long n, void *stream) {                  \
        PGW_REQUIRE(a && b && c && o && n > 0);                                                      \
        KERNEL<T><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(a, b, c, o, n);                 \
        return pgw_check_launch(#KERNEL);                                                            \
    }
PGW_EW3(pgw_specific_to_relative_humidity_f32, q2rh_kernel, float)
PGW_EW3(pgw_specific_to_relative_humidity_f64, q2rh_kernel, double)
PGW_EW3(pgw_relative_to_specific_humidity_f32, rh2q_kernel, float)
PGW_EW3(pgw_relative_to_specific_humidity_f64, rh2q_kernel, double)

#define PGW_GEOPOT(NAME, T, TS)                                                                      \
    int NAME(const T *pa_hl, const T *zgs, const TS *ta, const TS *hus, const T *p_ref_field,        \
             double p_ref, double *phi_ref, int nlev, long long ncol, uint32_t *err, void *stream) { \
        PGW_REQUIRE(pa_hl && zgs && ta && hus && phi_ref && err && nlev >= 1 && ncol > 0);           \
        integ_geopot_kernel<T, TS><<<(unsigned)((ncol + 127) / 128), 128, 0, (cudaStream_t)stream>>>(\
            pa_hl, zgs, ta, hus, p_ref_field, p_ref, phi_ref, nlev, ncol, err);                      \
        return pgw_check_launch("integ_geopot_kernel");                                              \
    }
PGW_GEOPOT(pgw_integ_geopot_f32, float, float)
PGW_GEOPOT(pgw_integ_geopot_f64, double, double)
PGW_GEOPOT(pgw_integ_geopot_f64_f32, double, float)

#define PGW_TOS(NAME, T)                                                                             \
    int NAME(const T *tos, const T *ts, const T *land, const T *ice, T *out, long long n,            \
             void *stream) {                                                                         \
        PGW_REQUIRE(tos && ts && land && ice && out && n > 0);                                       \
        integrate_tos_kernel<T><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(tos, ts, land,    \
                                                                                    ice, out, n);   \
        return pgw_check_launch("integrate_tos_kernel");                                             \
    }
PGW_TOS(pgw_integrate_tos_f32, float)
PGW_TOS(pgw_integrate_tos_f64, double)

#define PGW_HUMOP(NAME, T)                                                                           \
    int NAME(int op, const T *x, const T *y, T *out, long long n, void *stream) {                    \
        PGW_REQUIRE(x && out && n > 0 && op >= PGW_HUM_Q2E && op <= PGW_HUM_ESAT_BLEND);             \
        PGW_REQUIRE(y || op >= PGW_HUM_ESAT_WATER);                                                  \
        humidity_op_kernel<T><<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(op, x, y, out, n);  \
        return pgw_check_launch("humidity_op_kernel");                                               \
    }
PGW_HUMOP(pgw_humidity_op_f32, float)
PGW_HUMOP(pgw_humidity_op_f64, double)

#define PGW_RDS(NAME, T)                                                                             \
    int NAME(const T *source_P, const T *ps_hist, const T *delta, const T *delta_sfc, T *out_P,      \
             T *out_d, int K, long long ncol, int src_p_is_1d, uint32_t *err, void *stream) {        \
        PGW_REQUIRE(source_P && ps_hist && delta && delta_sfc && out_P && out_d && err);             \
        PGW_REQUIRE(K >= 1 && ncol > 0);                                                             \
        replace_delta_sfc_kernel<T><<<(unsigned)((ncol + 127) / 128), 128, 0, (cudaStream_t)stream>>>( \
            source_P, ps_hist, delta, delta_sfc, out_P, out_d, K, ncol, src_p_is_1d, err);           \
        return pgw_check_launch("replace_delta_sfc_kernel");                                         \
    }
PGW_RDS(pgw_replace_delta_sfc_f32, float)
PGW_RDS(pgw_replace_delta_sfc_f64, double)

int pgw_time_interp_f32(const float *lo, const float *hi, double x_hi, double x_new, float *out, long long n,
                        void *stream) {
    PGW_REQUIRE(lo && hi && out && n > 0);
    PGW_REQUIRE(x_new == 0.0 || x_hi != 0.0);
    time_interp_kernel<<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(lo, hi, x_hi, x_new, out, n);
    return pgw_check_launch("time_interp_kernel");
}

// ---------------------------------------------------------------------------
// NetCDF-3 stores big-endian numbers: the file pipeline moves the raw bytes of the float32 fields
// between the file and pinned host memory and swaps them here, next to the H2D / D2H copies
// (step_03_apply_to_era.py:60, :378 -- the decode xarray does on the CPU).  In place, 16 bytes/thread.
// ---------------------------------------------------------------------------
namespace pgw {
__global__ void __launch_bounds__(256) byteswap32_kernel(uint32_t *__restrict__ data, long long n) {
    const long long n4 = n >> 2;
    uint4 *const v = reinterpret_cast<uint4 *>(data);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        uint4 x = v[i];
        x.x = __byte_perm(x.x, 0, 0x0123); x.y = __byte_perm(x.y, 0, 0x0123);
        x.z = __byte_perm(x.z, 0, 0x0123); x.w = __byte_perm(x.w, 0, 0x0123);
        v[i] = x;
    }
    for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        data[i] = __byte_perm(data[i], 0, 0x0123);
}
}  // namespace pgw

int pgw_byteswap32(void *data, long long n, void *stream) {
    PGW_REQUIRE(data && n > 0 && (reinterpret_cast<uintptr_t>(data) & 15u) == 0);
    pgw::byteswap32_kernel<<<ew_grid((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<uint32_t *>(data), n);
    return pgw_check_launch("byteswap32_kernel");
}

// ---------------------------------------------------------------------------
// One stamp of ta, hur, ua, va into the engine's node layout d4 (one float4 per pressure node and column),
// optionally swapping the byte order of big-endian NetCDF-3 records on the way.  Words are moved, never
// converted, so NaN payloads survive.  A thread packs four consecutive nodes from one 16-byte load per input
// when every input is 16-byte aligned; otherwise (and for the last n % 4 nodes) one node per word load.
// ---------------------------------------------------------------------------
namespace pgw {
__device__ __forceinline__ uint32_t maybe_swap(uint32_t x, int swap) { return swap ? __byte_perm(x, 0, 0x0123) : x; }

__global__ void __launch_bounds__(256) pack_d4_kernel(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                                                     const uint32_t *__restrict__ c, const uint32_t *__restrict__ d,
                                                     uint4 *__restrict__ out, long long n, int swap, int vec) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n4 = vec ? n >> 2 : 0;
    for (long long i = t0; i < n4; i += stride) {
        const uint4 x = reinterpret_cast<const uint4 *>(a)[i], y = reinterpret_cast<const uint4 *>(b)[i];
        const uint4 z = reinterpret_cast<const uint4 *>(c)[i], w = reinterpret_cast<const uint4 *>(d)[i];
        uint4 *o = out + 4 * i;
        o[0] = make_uint4(maybe_swap(x.x, swap), maybe_swap(y.x, swap), maybe_swap(z.x, swap), maybe_swap(w.x, swap));
        o[1] = make_uint4(maybe_swap(x.y, swap), maybe_swap(y.y, swap), maybe_swap(z.y, swap), maybe_swap(w.y, swap));
        o[2] = make_uint4(maybe_swap(x.z, swap), maybe_swap(y.z, swap), maybe_swap(z.z, swap), maybe_swap(w.z, swap));
        o[3] = make_uint4(maybe_swap(x.w, swap), maybe_swap(y.w, swap), maybe_swap(z.w, swap), maybe_swap(w.w, swap));
    }
    for (long long i = (n4 << 2) + t0; i < n; i += stride)
        out[i] = make_uint4(maybe_swap(a[i], swap), maybe_swap(b[i], swap), maybe_swap(c[i], swap),
                            maybe_swap(d[i], swap));
}
}  // namespace pgw

int pgw_pack_d4_f32(const void *ta, const void *hur, const void *ua, const void *va, void *out, long long n,
                    int swap, void *stream) {
    PGW_REQUIRE(ta && hur && ua && va && out && n > 0 && (swap == 0 || swap == 1));
    PGW_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15u) == 0);
    const uintptr_t any = reinterpret_cast<uintptr_t>(ta) | reinterpret_cast<uintptr_t>(hur) |
                          reinterpret_cast<uintptr_t>(ua) | reinterpret_cast<uintptr_t>(va);
    const int vec = (any & 15u) == 0;
    pgw::pack_d4_kernel<<<ew_grid(vec ? (n + 3) / 4 : n, 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const uint32_t *>(ta), static_cast<const uint32_t *>(hur), static_cast<const uint32_t *>(ua),
        static_cast<const uint32_t *>(va), static_cast<uint4 *>(out), n, swap, vec);
    return pgw_check_launch("pack_d4_kernel");
}

int pgw_time_mean_f32(const float *series, int ntime, float *out, long long n, void *stream) {
    PGW_REQUIRE(series && out && ntime > 0 && n > 0);
    time_mean_kernel<<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(series, ntime, out, n);
    return pgw_check_launch("time_mean_kernel");
}

}  // extern "C"
