/*
 * pgw_b200.h -- C ABI of libpgw_b200.so, the sm_100a implementation of the
 * PGW4ERA5 per-timestep path.
 *
 * Every entry point takes plain DEVICE pointers owned by the caller, sizes, a
 * CUDA stream (passed as void*) and returns 0 or a negative host-side error
 * (PGW_E_*).  Data-dependent failures that the reference reports as Python
 * ValueErrors are accumulated on the device in a sticky 32-bit error word
 * (PGW_ERR_* bits, atomicOr) that the caller reads back after the stream
 * synchronises; the Python host layer maps the bits to the reference's
 * messages.  Nothing here allocates device memory; workspaces are passed in.
 *
 * Layout: all fields are C-order with the horizontal index fastest, i.e.
 * element (level k, column c) lives at k*ncol + c, ncol = nlat*nlon, exactly
 * the (time, level, lat, lon) layout of the reference for one timestep.
 *
 * "Replaces" cites the reference (menschj/PGW4ERA5) interface each entry point
 * stands in for.
 */
#ifndef PGW_B200_H
#define PGW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGW_B200_ABI_VERSION 10  /* 6: + pgw_timestep_status, pgw_timestep_run/_finish, PGW_FLAG_REF_DTYPES, first_k,
                                       pgw_band_pack/_unpack, pgw_band_exchange, pgw_regrid_bilinear_band_f32
                                    7: + PGW_FLAG_LOCAL_PREF and its args, PGW_ERR_PREF_FLOOR, first_k[4]
                                    8: + PGW_FLAG_REINTERP (no layout change)
                                    9: + pgw_pack_d4_f32
                                   10: + pgw_regrid_pack_d4_f32, PGW_REGRID_PACK_MAX_NX_S */

/* host-side return codes */
#define PGW_OK               0
#define PGW_E_INVALID       -1   /* bad argument (null pointer, size, mode)      */
#define PGW_E_LAUNCH        -2   /* CUDA launch / runtime error                 */
#define PGW_E_SMEM          -3   /* column stash does not fit in shared memory  */

/* device-side sticky error bits */
#define PGW_ERR_SRC_NOT_ASCENDING   (1u << 0)  /* functions.py:500-501 */
#define PGW_ERR_TARG_NOT_ASCENDING  (1u << 1)  /* functions.py:502-503 */
#define PGW_ERR_EXTRAP_OFF          (1u << 2)  /* functions.py:564-566 */
#define PGW_ERR_PS_HIST_RANGE       (1u << 4)  /* functions.py:360-361,363 */
#define PGW_ERR_PREF_BELOW_SFC      (1u << 5)  /* functions.py:162-165 */
#define PGW_ERR_NO_PREF             (1u << 6)  /* step_03_apply_to_era.py:245-251 */
#define PGW_ERR_BAND_TIMEOUT        (1u << 8)  /* pgw_band_exchange: a peer's status block did not arrive */
#define PGW_ERR_PS_BOUND            (1u << 7)  /* ps left the range the column
                                                  stash was sized for: rerun
                                                  with a larger ps_bound */
#define PGW_ERR_PREF_FLOOR          (1u << 9)  /* PGW_FLAG_LOCAL_PREF: p_ref left the range the
                                                  column stash was sized for: rerun
                                                  with a lower p_floor */

/* extrapolation modes of interp_extrap_1d, functions.py:516-520 */
#define PGW_EXTRAP_OFF       0
#define PGW_EXTRAP_LINEAR    1
#define PGW_EXTRAP_CONSTANT  2
#define PGW_EXTRAP_NAN       3

/* pgw_timestep_args.flags */
#define PGW_FLAG_DIRECT  1   /* take the cp.async flavour of the column kernel, which integrates every parked
                                level in every iteration (the TMA flavour uses a polynomial in dps) */
#define PGW_FLAG_REF_DTYPES 2 /* reproduce the dtypes the reference computes in when PS and FIS are float32 in the
                                ERA5 file (every real file): delta_ps and ps_pgw are float32
                                (step_03_apply_to_era.py:186-195: zeros_like(PS), in-place +=), the half-level
                                geopotential is a float32 running sum rounded on every level (functions.py:141,
                                :147-152), -adj_factor*ps_pgw is a float32 product (step_03:302-303).  Implies
                                PGW_FLAG_DIRECT.  Without the flag the accumulation is float64, i.e. the reference
                                on a file that stores PS and FIS as double. */
#define PGW_FLAG_LOCAL_PREF 4 /* p_ref_inp = None (step_03_apply_to_era.py:219-251): the reference pressure is picked
                                per column and iteration among zg's pressure levels (determine_p_ref,
                                functions.py:583-598) and the climate term is the zg delta on that level.  Takes the
                                cp.async flavour; not combinable with PGW_FLAG_REF_DTYPES.  Reads the last block of
                                pgw_timestep_args (zg .. p_ref_out); p_ref and zg_ref are ignored, p_floor sizes the
                                column stash in place of p_ref. */
#define PGW_FLAG_REINTERP 8   /* i_reinterp = 1 (step_03_apply_to_era.py:155-173, :202-216, :330-343): no delta is
                                applied before the iteration; every iteration interpolates the ERA state (T, RELHUM)
                                linearly in ln p ('constant' extrapolation, functions.py:434-580) onto its own
                                pressures akm + ps_pgw bkm and adds the deltas there, and ta_pgw of the lowest level
                                of that iteration divides adj_ps.  The outputs are the state evaluated in the last
                                iteration: PS, and T, QV, U, V on every level at its pressures (U, V interpolated
                                after the loop).  Takes the cp.async flavour; not combinable with
                                PGW_FLAG_LOCAL_PREF or PGW_FLAG_REF_DTYPES (PGW_E_INVALID).  When N < k_spec,
                                pgw_timestep_finalize does not rewrite PS/QV from the speculative QV: it relaunches
                                the column kernel with k_spec = N read from the device result (a replay: every CTA
                                returns at once unless `rewritten` is set; its updates of maxerr, err, first_k and
                                stats repeat values already there), so the outputs equal those of a run with
                                k_spec = N bit for bit. */

#define PGW_MAX_SOIL   16
#define PGW_MAX_ITER   64

const char *pgw_version(void);
int pgw_abi_version(void);          /* PGW_B200_ABI_VERSION the library was built with */
const char *pgw_last_error(void);      /* text of the last PGW_E_LAUNCH */

/* ------------------------------------------------------------------------
 * Vertical log-pressure interpolation.
 * Replaces interp_1d_for_timelatlon(orig_array, src_p, targ_p, interp_array,
 * ntime, nlat, nlon, extrapolate), functions.py:479-508 (+ interp_extrap_1d
 * :511-580), the reference's only compiled boundary, and the np.log calls of
 * its caller interp_logp_4d, functions.py:469-475.
 *   var   [nt, ks, ncol]   values on source levels
 *   src_p [nt, ks, ncol]   source pressure, or [ks] if src_p_is_1d
 *   targ_p[nt, kt, ncol]   target pressure
 *   out   [nt, kt, ncol]
 *   p_is_log: 0 = arrays hold pressure (log taken in-kernel),
 *             1 = arrays already hold ln p (the numba signature).
 *   err   device uint32, OR-ed with PGW_ERR_{SRC,TARG}_NOT_ASCENDING /
 *         PGW_ERR_EXTRAP_OFF.
 * ---------------------------------------------------------------------- */
int pgw_interp_logp_f64(const double *var, const double *src_p, const double *targ_p,
                        double *out, int nt, int ks, int kt, long long ncol,
                        int src_p_is_1d, int p_is_log, int mode,
                        uint32_t *err, void *stream);
int pgw_interp_logp_f32(const float *var, const float *src_p, const float *targ_p,
                        float *out, int nt, int ks, int kt, long long ncol,
                        int src_p_is_1d, int p_is_log, int mode,
                        uint32_t *err, void *stream);

/* ------------------------------------------------------------------------
 * Humidity conversions (IFS saturation vapour pressure over water and ice).
 * Replace specific_to_relative_humidity(hus, pa, ta), functions.py:107-116 and
 * relative_to_specific_humidity(hur, pa, ta), functions.py:118-125.
 * Elementwise over n values.
 * ---------------------------------------------------------------------- */
int pgw_specific_to_relative_humidity_f32(const float *hus, const float *pa, const float *ta,
                                          float *hur, long long n, void *stream);
int pgw_relative_to_specific_humidity_f32(const float *hur, const float *pa, const float *ta,
                                          float *hus, long long n, void *stream);
int pgw_specific_to_relative_humidity_f64(const double *hus, const double *pa, const double *ta,
                                          double *hur, long long n, void *stream);
int pgw_relative_to_specific_humidity_f64(const double *hur, const double *pa, const double *ta,
                                          double *hus, long long n, void *stream);

/* The small helpers of the same block, elementwise over n values:
 *   PGW_HUM_Q2E         specific_humidity_to_vapor_pressure(x=hus, y=pa)      functions.py:58-64
 *   PGW_HUM_E2Q         vapor_pressure_to_specific_humidity(x=vapp, y=pa)     functions.py:66-72
 *   PGW_HUM_ESAT_WATER  saturation_vapor_pressure_water_or_ice(x=ta, water)   functions.py:74-89
 *   PGW_HUM_ESAT_ICE    saturation_vapor_pressure_water_or_ice(x=ta, ice)
 *   PGW_HUM_ESAT_BLEND  saturation_vapor_pressure_water_and_ice(x=ta)         functions.py:91-105
 * (y may be NULL for the three ESAT operations). */
#define PGW_HUM_Q2E         0
#define PGW_HUM_E2Q         1
#define PGW_HUM_ESAT_WATER  2
#define PGW_HUM_ESAT_ICE    3
#define PGW_HUM_ESAT_BLEND  4
int pgw_humidity_op_f32(int op, const float *x, const float *y, float *out, long long n, void *stream);
int pgw_humidity_op_f64(int op, const double *x, const double *y, double *out, long long n, void *stream);

/* ------------------------------------------------------------------------
 * Surface insertion into the 3-D deltas, every column.
 * Replaces replace_delta_sfc(source_P, ps_hist, delta, delta_sfc), functions.py:343-366,
 * as applied through xr.apply_ufunc(vectorize=True), functions.py:396-402.
 *   source_P [K, ncol] (or [K] if src_p_is_1d), ps_hist, delta_sfc [ncol], delta [K, ncol]
 *   out_P, out_d [K, ncol];  err: PGW_ERR_PS_HIST_RANGE (the reference's bare ValueError)
 * ---------------------------------------------------------------------- */
int pgw_replace_delta_sfc_f32(const float *source_P, const float *ps_hist, const float *delta,
                              const float *delta_sfc, float *out_P, float *out_d, int K,
                              long long ncol, int src_p_is_1d, uint32_t *err, void *stream);
int pgw_replace_delta_sfc_f64(const double *source_P, const double *ps_hist, const double *delta,
                              const double *delta_sfc, double *out_P, double *out_d, int K,
                              long long ncol, int src_p_is_1d, uint32_t *err, void *stream);

/* ------------------------------------------------------------------------
 * Hydrostatic geopotential at a reference pressure.
 * Replaces integ_geopot(pa_hl, zgs, ta, hus, level1, p_ref), functions.py:128-189.
 *   pa_hl [nlev+1, ncol] half-level pressure (index 0 = model top)
 *   zgs   [ncol] surface geopotential;  ta, hus [nlev, ncol]
 *   p_ref_field [ncol] or NULL (then the scalar p_ref is used)
 *   phi_ref [ncol] float64 output
 *   err: PGW_ERR_PREF_BELOW_SFC
 * ---------------------------------------------------------------------- */
int pgw_integ_geopot_f32(const float *pa_hl, const float *zgs, const float *ta, const float *hus,
                         const float *p_ref_field, double p_ref, double *phi_ref,
                         int nlev, long long ncol, uint32_t *err, void *stream);
int pgw_integ_geopot_f64(const double *pa_hl, const double *zgs, const double *ta, const double *hus,
                         const double *p_ref_field, double p_ref, double *phi_ref,
                         int nlev, long long ncol, uint32_t *err, void *stream);
/* float64 pressures with the float32 T and QV of an ERA5 file: like numpy in the reference, Rd * Tv is
 * then a chain of float32 products (functions.py:144, :151, :177), the sums are float64 */
int pgw_integ_geopot_f64_f32(const double *pa_hl, const double *zgs, const float *ta, const float *hus,
                             const double *p_ref_field, double p_ref, double *phi_ref,
                             int nlev, long long ncol, uint32_t *err, void *stream);

/* ------------------------------------------------------------------------
 * Land / sea-ice weighted blend of the ts and tos deltas.
 * Replaces integrate_tos(tos_field, ts_field, land_frac, ice_frac),
 * functions.py:1145-1186.  n values each.
 * ---------------------------------------------------------------------- */
int pgw_integrate_tos_f32(const float *tos, const float *ts, const float *land, const float *ice,
                          float *out, long long n, void *stream);
int pgw_integrate_tos_f64(const double *tos, const double *ts, const double *land, const double *ice,
                          double *out, long long n, void *stream);

/* ------------------------------------------------------------------------
 * Two-point linear time interpolation of a delta field (the arithmetic of
 * load_delta, functions.py:288-292 -> xarray .interp -> scipy interp1d):
 *   out = (hi - lo) / x_hi * x_new + lo      (float64 math, float32 storage)
 * and the time mean used for the deep-soil delta (step_03_apply_to_era.py:134-136).
 * ---------------------------------------------------------------------- */
int pgw_time_interp_f32(const float *lo, const float *hi, double x_hi, double x_new,
                        float *out, long long n, void *stream);
int pgw_time_mean_f32(const float *series, int ntime, float *out, long long n, void *stream);

/* ------------------------------------------------------------------------
 * The fused per-timestep pass.
 * Replaces the body of pgw_for_era5(), step_03_apply_to_era.py:60-343 with
 * a scalar or (PGW_FLAG_LOCAL_PREF, i_reinterp = 0) per-column p_ref, and i_reinterp = 0 or
 * (PGW_FLAG_REINTERP) 1: pressures (:64-88), RELHUM (:91-94),
 * sea-ice/skin/soil update (:103-146, integrate_tos), load_delta's time blend
 * (functions.py:288-292), replace_delta_sfc + vert_interp_delta
 * (functions.py:343-431) for ta,hur,ua,va, delta application (:158-173) and
 * k_spec iterations of the surface-pressure fixed point (:182-319, integ_geopot
 * and relative_to_specific_humidity inside).
 *
 * The stopping rule of the reference is field-global (:189,:308): iteration
 * stops at the first N with max|phi error| <= thresh.  The kernel therefore
 * runs exactly k_spec iterations for every column, records max|err_k| for
 * k = 1..k_spec in maxerr[k-1] (float64 bits, atomicMax) and the trajectory
 * dps_k in dps_traj, and writes PS/QV for dps_{k_spec}.  The caller then
 *   - all-reduces maxerr (MAX) over ranks in latitude-band mode,
 *   - calls pgw_timestep_finalize(), which finds N on the device and, if
 *     N < k_spec, rewrites PS/QV for dps_N (PGW_FLAG_REINTERP: replays the
 *     column kernel for k_spec = N),
 *   - reruns with a larger k_spec if maxerr[k_spec-1] > thresh.
 * ---------------------------------------------------------------------- */
typedef struct pgw_tslab {
    const float *lo;    /* field at the delta stamp before the ERA5 time      */
    const float *hi;    /* field at the stamp after (== lo for an exact hit)  */
    double x_hi;        /* (t_after  - t_before) in ns, as xarray hands scipy  */
    double x_new;       /* (t_target - t_before) in ns; 0 for an exact hit     */
} pgw_tslab;

typedef struct pgw_timestep_args {
    /* sizes */
    long long ncol;         /* nlat*nlon of this rank's band                   */
    int nlev;               /* full model levels (137)                         */
    int nplev;              /* GCM pressure levels K (<= 64)                   */
    int nsoil;              /* soil levels (<= PGW_MAX_SOIL)                   */
    int plev_descending;    /* 1: 3-D delta slabs are stored bottom-up
                               (pressure descending, CMIP6 order)              */
    int flags;              /* PGW_FLAG_*                                      */
    int reserved0;
    /* level tables, DEVICE float64 */
    const double *ak, *bk;      /* [nlev+1] */
    const double *akm, *bkm;    /* [nlev]   */
    const double *plev;         /* [nplev] in FILE order                       */
    /* HOST copies of ak, bk ([nlev+1]); used to size the shared-memory stash  */
    const double *ak_host, *bk_host;
    /* HOST copies of akm, bkm ([nlev]); optional (may be NULL): with them, and with
       ncol % 4 == 0 and 16-byte aligned 3-D fields, pgw_timestep() streams the 3-D
       fields with TMA (cp.async.bulk.tensor) instead of per-thread copies          */
    const double *akm_host, *bkm_host;
    /* ERA5 fields of one timestep, DEVICE float32 */
    const float *PS, *FIS, *FR_LAND, *FR_SEA_ICE, *T_SKIN;   /* [ncol]         */
    const float *T_SO;                                       /* [nsoil, ncol]  */
    const float *T, *QV, *U, *V;                             /* [nlev, ncol]   */
    /* climate deltas bracketing the ERA5 time */
    pgw_tslab d4;           /* ta, hur, ua, va deltas packed per node and column:
                               float4 [nplev, ncol] = {ta, hur, ua, va}, 16-byte
                               aligned (lo/hi point at float4 data)            */
    pgw_tslab tas, hurs, ps_hist, ts, tos, siconc;   /* [ncol]                 */
    pgw_tslab zg_ref;                   /* zg delta on the p_ref level, [ncol] */
    const float *ts_clim;               /* annual-mean ts delta [ncol]         */
    double soil_decay[PGW_MAX_SOIL];    /* exp(-soil1/2.8)                     */
    /* surface-pressure adjustment (settings.py:140-150) */
    double p_ref;
    double adj_factor;
    double thresh_phi_ref_max_error;
    int k_spec;             /* iterations to run (1..PGW_MAX_ITER)             */
    double ps_bound;        /* upper bound of ps used to size the column stash */
    /* outputs, DEVICE float32 (must not alias the inputs) */
    float *PS_out, *T_SKIN_out, *FR_SEA_ICE_out;   /* [ncol]                   */
    float *T_SO_out;                                /* [nsoil, ncol]            */
    float *T_out, *QV_out, *U_out, *V_out;          /* [nlev, ncol]             */
    float *dps_out;                                 /* [ncol] ps_pgw - PS       */
    /* workspace */
    float *dps_traj;        /* [k_spec, ncol]                                  */
    uint64_t *maxerr;       /* [PGW_MAX_ITER] float64 bits, zeroed by the call */
    float *stats;           /* [2]: min target p, min source p (ta/hur)        */
    uint32_t *err;          /* sticky error word                               */
    int32_t *first_k;       /* [4] or NULL: first iteration (0-based) in which PGW_ERR_PREF_BELOW_SFC /
                               PGW_ERR_PS_BOUND / PGW_ERR_NO_PREF / PGW_ERR_PREF_FLOOR fired (atomicMin;
                               INT32_MAX = never).  The kernel runs k_spec
                               iterations for every column, the reference stops after N: a condition that only
                               fires in an iteration >= N never happened in the reference. */
    uint32_t *poly_fallback; /* or NULL: number of (warp, iteration) pairs of the TMA flavour that left the range
                               of the dps polynomial and integrated all parked levels directly (diagnostic) */
    /* PGW_FLAG_LOCAL_PREF only (may be zero otherwise).  p_ref_k of iteration k is the first level of zg_plev, in
       file order, with 0.95*PS > p and 0.95*(PS + dps_k) > p, and from the second iteration on at most p_ref_{k-1}.
       The stash covers every layer that can contain a pressure >= p_floor for ps <= ps_bound; a column whose
       p_ref_k falls below p_floor sets PGW_ERR_PREF_FLOOR (rerun with a lower p_floor).  No qualifying level:
       PGW_ERR_NO_PREF and p_ref NaN. */
    pgw_tslab zg;               /* zg delta on all of zg's levels, [nzg, ncol] per time slab */
    const double *zg_plev;      /* [nzg] DEVICE, zg's pressure levels in FILE order (distinct values) */
    const double *zg_plev_host; /* [nzg] HOST copy (sizes the table of candidate levels) */
    int nzg;                    /* 1..64 */
    int reserved1;
    double p_floor;             /* lowest p_ref the column stash is sized for */
    uint8_t *pref_traj;         /* [k_spec, ncol] workspace: index of p_ref_k in zg_plev (255 = none) */
    double *p_ref_out;          /* [ncol] p_ref of the iteration the result is for (finalize rewrites it for N) */
} pgw_timestep_args;

/* bytes of dynamic shared memory the column kernel needs for these args, or
 * a negative PGW_E_* code */
long long pgw_sizeof_timestep_args(void);   /* for FFI layout checks */
long long pgw_timestep_smem_bytes(const pgw_timestep_args *a);
/* 1 if pgw_timestep() takes the TMA flavour of the column kernel for these args, 0 if the
 * per-thread cp.async flavour (odd ncol, unaligned fields, PGW_COLUMN_PATH=generic, PGW_FLAG_DIRECT,
 * PGW_FLAG_REF_DTYPES, and PGW_FLAG_LOCAL_PREF and PGW_FLAG_REINTERP on every grid: the TMA flavour handles a
 * scalar p_ref and iteration-invariant parked levels only) */
int pgw_timestep_uses_tma(const pgw_timestep_args *a);
/* The plan pgw_timestep() launches for these args: info[0] 1 for the TMA flavour, info[1] 1 if every layer the
 * iteration can touch takes the ln series (the FAST instances; 0: the exact-log ones), info[2] the top level of
 * the stash, info[3] the number of parked levels, info[4] the tensor-memory columns per CTA (0 for cp.async),
 * info[5] 1 if the TMA flavour takes its L137 instance (137 levels, 56 parked).  PGW_OK or PGW_E_INVALID. */
int pgw_timestep_plan_info(const pgw_timestep_args *a, int info[6]);
/* Resources per CTA of the TMA flavour for nplev pressure nodes, nlev levels and np parked levels (even): the
 * tensor-memory columns it allocates and the bytes of dynamic shared memory it is launched with (padded to the
 * CTA's share of the SM's tensor memory).  Host arithmetic only; PGW_E_INVALID for arguments out of range. */
int pgw_column_tma_layout(int nplev, int nlev, int np, int *tmem_cols, long long *smem_bytes);
int pgw_timestep(const pgw_timestep_args *a, void *stream);

/* device-side result of the convergence scan, written by finalize */
typedef struct pgw_timestep_result {
    int n_iter;             /* N = first k with maxerr[k-1] <= thresh, or 0    */
    int converged;          /* 1 if N found within k_spec                      */
    int rewritten;          /* 1 if PS/QV were rewritten for N < k_spec        */
    int reserved;
} pgw_timestep_result;

int pgw_timestep_finalize(const pgw_timestep_args *a, pgw_timestep_result *result_dev,
                          void *stream);

/* The status block of one timestep in flight: what the kernels report and the host reads back.  maxerr, stats,
 * err and first_k of the args must point at the members of ONE such block in device memory. */
typedef struct pgw_timestep_status {
    uint64_t maxerr[PGW_MAX_ITER];  /* max|phi error| per iteration, float64 bits                  */
    pgw_timestep_result result;     /* written by finalize                                         */
    float stats[2];                 /* min target pressure, min source pressure (functions.py:417) */
    uint32_t err;                   /* PGW_ERR_* bits                                              */
    int32_t first_k[4];             /* see pgw_timestep_args.first_k                               */
    uint32_t poly_fallback;         /* see pgw_timestep_args.poly_fallback                         */
} pgw_timestep_status;
long long pgw_sizeof_timestep_status(void);

/* One call per timestep: clears the status block, runs the column kernel and -- unless PGW_RUN_NO_FINALIZE --
 * finalize, then copies the status block to `status_host` (pinned host memory, may be NULL) on the same stream.
 * Latitude-band mode passes PGW_RUN_NO_FINALIZE, reduces the block over the bands (pgw_band_pack -> all-reduce MAX
 * -> pgw_band_unpack) and calls pgw_timestep_finish (finalize + copy). */
#define PGW_RUN_NO_FINALIZE 1
int pgw_timestep_run(const pgw_timestep_args *a, pgw_timestep_status *status_dev,
                     pgw_timestep_status *status_host, int run_flags, void *stream);
int pgw_timestep_finish(const pgw_timestep_args *a, pgw_timestep_status *status_dev,
                        pgw_timestep_status *status_host, void *stream);
/* The status block as PGW_BAND_WORDS float64 such that an element-wise MAX over the latitude bands merges it:
 * maxerr[64] | -stats[2] | one word per error bit [32] | -first_k[4]; and back.  The stopping rule of the
 * reference is field-global (step_03_apply_to_era.py:189,308), so this is the one exchange of band mode. */
#define PGW_BAND_WORDS (PGW_MAX_ITER + 2 + 32 + 4)
int pgw_band_pack(const pgw_timestep_status *status_dev, double *words_dev, void *stream);
int pgw_band_unpack(const double *words_dev, pgw_timestep_status *status_dev, void *stream);
/* The same exchange WITHOUT a collective library, as one kernel over peer memory (NVLink / NVSwitch): every rank owns
 * an inbox of PGW_BAND_PARITIES x world x PGW_BAND_SLOT float64 in memory its peers can store to (CUDA IPC / VMM
 * peer mappings, e.g. torch symmetric memory); inbox_ptrs_dev[r] is rank r's inbox as seen from this GPU.
 * The kernel packs this band's status block, stores it into slot [seq % parities][rank] of EVERY inbox, publishes it
 * with a system-scope release of the slot's flag word (= seq), waits until all `world` flags of its own inbox carry
 * seq, merges the blocks (MAX) and unpacks the result into status_dev -- launched on the stream right behind the
 * column kernel, it is the collective fused into the step: no host round trip, no second library, ~100 stores per
 * peer.  seq must increase by one per snapshot, identically on all ranks, starting at 1 on a zeroed inbox.  A peer
 * that does not deliver within timeout_s sets PGW_ERR_BAND_TIMEOUT (the kernel never spins for ever). */
#define PGW_BAND_SLOT      (PGW_BAND_WORDS + 4)   /* words per slot: the block, the flag, padding */
#define PGW_BAND_PARITIES  8
int pgw_band_exchange(pgw_timestep_status *status_dev, double *const *inbox_ptrs_dev, int rank, int world,
                      unsigned long long seq, double timeout_s, void *stream);

/* ------------------------------------------------------------------------
 * The staged per-timestep path: pgw_for_era5() run stage by stage on float64
 * device arrays with the operators above plus the small ones below.  It covers
 * i_reinterp = 1 (step_03_apply_to_era.py:202-216, :330-343) and p_ref_inp = None (:219-251), the references
 * the fused pass's PGW_FLAG_REINTERP and PGW_FLAG_LOCAL_PREF are tested against, and their combination with
 * each other or with the file dtypes, which the fused pass does not cover;
 * host orchestration: pgw4era5_b200/staged.py.
 *   pgw_surface_update        sea ice / skin / soil block, step_03:103-146
 *                             (reads only the 2-D members of the args)
 *   pgw_hybrid_pressure_f64   p[l,c] = a[l] + ps[c]*b[l], step_03:64-88,:196-199
 *   pgw_axpy_f64              out = x + alpha*y (delta application :169-172,
 *                             ps update :192-193)
 *   pgw_determine_p_ref_f64   determine_p_ref per column, functions.py:583-598;
 *                             opts in the order of the zg file; p_ref_last NULL
 *                             in the first iteration; PGW_ERR_NO_PREF if none
 *   pgw_select_plev_f64       field.sel(plev = p_ref[c]) per column, :292-295
 *   pgw_ps_adjust_f64         phi_ref_error, adj_ps and atomicMax of |error|
 *                             (float64 bits in *maxerr), step_03:286-308
 * ---------------------------------------------------------------------- */
int pgw_surface_update(const pgw_timestep_args *a, void *stream);
int pgw_hybrid_pressure_f64(const double *ps, const double *a, const double *b, double *out, int nlev,
                            long long ncol, void *stream);
int pgw_axpy_f64(const double *x, const double *y, double alpha, double *out, long long n, void *stream);
int pgw_determine_p_ref_f64(const double *p_min_era, const double *p_min_pgw, const double *opts, int nopt,
                            const double *p_ref_last, double *out, long long n, uint32_t *err, void *stream);
int pgw_select_plev_f64(const double *field, const double *plev, int K, const double *p_ref, double *out,
                        long long n, void *stream);
int pgw_ps_adjust_f64(const double *phi_pgw, const double *phi_era, const double *dphi_clim, const double *ps_pgw,
                      const double *ta_low, double adj_factor, double *adj, uint64_t *maxerr, long long n,
                      void *stream);

/* ------------------------------------------------------------------------
 * step_02: bilinear regridding and annual-cycle smoothing.
 * pgw_regrid_bilinear_f32 replaces the two scipy interp1d passes of
 * regrid_lat_lon(), functions.py:859 and :892, including the pole rows
 * (:833-842, zonal mean of the nearest row) and the periodic longitude
 * (:866-874) which are applied through index tables instead of concatenation:
 *   src [nfield, ny_s, nx_s]  ->  dst [nfield, ny_t, nx_t]
 *   j0,j1 [ny_t] source rows (-1 = south-pole row, -2 = north-pole row,
 *                i.e. the zonal mean of row 0 / ny_s-1), wy [ny_t] weight of j1
 *   i0,i1 [nx_t] source columns (already wrapped), wx [nx_t] weight of i1
 *   polemean [nfield, 2] zonal means (filled by pgw_zonal_mean_f32: the mean of
 *                the valid points of the row, skipping NaN like xarray; NaN if none)
 * pgw_smooth_harmonic_f32 replaces filter_data()/harmonic_ac_analysis(),
 * functions.py:606-740: per grid point mean + 3 harmonics of the nt-long series.
 * ---------------------------------------------------------------------- */
int pgw_zonal_mean_f32(const float *src, float *polemean, long long nfield, int ny_s, int nx_s,
                       void *stream);
int pgw_regrid_bilinear_f32(const float *src, float *dst, const float *polemean,
                            long long nfield, int ny_s, int nx_s, int ny_t, int nx_t,
                            const int *j0, const int *j1, const double *wy,
                            const int *i0, const int *i1, const double *wx,
                            void *stream);
/* The same for the band [jt_begin, jt_end) of target rows only; dst holds just those rows,
 * [nfield, jt_end - jt_begin, nx_t].  One variable split over several GPUs by target latitude (the source field
 * is replicated, the pole-row means are computed on every GPU); the tables stay those of the whole target grid. */
int pgw_regrid_bilinear_band_f32(const float *src, float *dst, const float *polemean,
                                 long long nfield, int ny_s, int nx_s, int ny_t, int nx_t,
                                 int jt_begin, int jt_end,
                                 const int *j0, const int *j1, const double *wy,
                                 const int *i0, const int *i1, const double *wx,
                                 void *stream);
int pgw_smooth_harmonic_f32(const float *series, float *out, int nt, long long npoint,
                            void *stream);

/* ------------------------------------------------------------------------
 * step_02, ocean variables (tos, siconc): NaN-ignoring Gaussian-kernel regridding from the curvilinear
 * GCM ocean grid.  Replaces nan_ignoring_interp(), functions.py:900-1060.
 * pgw_geod_to_meter_f64: the coordinate mapping of :946-973 / :1006-1022 -- lon > 180 -> lon - 360,
 *   lat_m = sign(lat) * geod.inv(lon, 0, lon, lat), lon_m = sign(lon) * geod.inv(0, lat, lon, lat),
 *   half_turn (optional) = geod.inv(0, lat, 180, lat); WGS84 geodesics (pyproj Geod.inv in the reference).
 * pgw_gauss_interp_f64: pyvista PolyData.interpolate(points, null_value=nan, radius, sharpness) of :1038-1048
 *   (vtkPointInterpolator + vtkGaussianKernel) plus the land mask FR_LAND > 0.7 -> NaN (:1031, :1055):
 *   src_lat_m ASCENDING [nsrc], src_lon_m [nsrc], src_val [nfield <= 12, nsrc] (NaN = absent for that
 *   field), dst_* [ndst], land_fr [ndst] or NULL, out [nfield, ndst].
 * ---------------------------------------------------------------------- */
int pgw_geod_to_meter_f64(const double *lat_deg, const double *lon_deg, double *lat_m, double *lon_m,
                          double *half_turn, long long n, void *stream);
int pgw_gauss_interp_f64(const double *src_lat_m, const double *src_lon_m, const double *src_val,
                         long long nsrc, int nfield, const double *dst_lat_m, const double *dst_lon_m,
                         const float *land_fr, double *out, long long ndst, double radius, double sharpness,
                         void *stream);

/* ------------------------------------------------------------------------
 * File pipeline: byte order of n 32-bit words, in place (data 16-byte aligned).
 * NetCDF-3 stores big-endian floats; replaces the decode/encode xarray performs on the CPU
 * inside open_dataset / to_netcdf (step_03_apply_to_era.py:60, :378) for the float32 fields.
 * ---------------------------------------------------------------------- */
int pgw_byteswap32(void *data, long long n, void *stream);

/* ------------------------------------------------------------------------
 * Streamed climatology: one delta stamp of ta, hur, ua, va (n = K*ncol 32-bit words each) into the
 * node layout of the column kernel, out[i] = {ta[i], hur[i], ua[i], va[i]} (out: float4[n], 16-byte
 * aligned).  swap = 1 also reverses the byte order of every word (raw NetCDF-3 records are big-endian).
 * Words are moved, not converted: NaN payloads survive.  Any n and any 4-byte alignment of the inputs;
 * 16-byte loads when all four are 16-byte aligned.
 * ---------------------------------------------------------------------- */
int pgw_pack_d4_f32(const void *ta, const void *hur, const void *ua, const void *va, void *out, long long n,
                    int swap, void *stream);

/* ------------------------------------------------------------------------
 * Climatology on the GCM grid: one delta stamp of ta, hur, ua, va regridded to the ERA5 grid and packed in one
 * pass, bit-identical to pgw_regrid_bilinear_band_f32 on each variable followed by pgw_pack_d4_f32.
 *   src [4, nlev, ny_s, nx_s] (ta, hur, ua, va), polemean [4 * nlev, 2] (pgw_zonal_mean_f32 of src),
 *   tables and target rows [jt_begin, jt_end) as for pgw_regrid_bilinear_band_f32,
 *   dst float4 [nlev, jt_end - jt_begin, nx_t] (16-byte aligned).
 * Source rows up to PGW_REGRID_PACK_MAX_NX_S columns run in the fused kernel and scratch may be NULL.  Wider
 * ones are regridded variable by variable into scratch (16-byte aligned, 4 pieces of n = nlev * (jt_end -
 * jt_begin) * nx_t floats, each rounded up to a multiple of 4) and then packed.
 * ---------------------------------------------------------------------- */
#define PGW_REGRID_PACK_MAX_NX_S 1536    /* the latitude-blended row of the four variables in 48 KB of shared memory */
int pgw_regrid_pack_d4_f32(const float *src, float *dst, const float *polemean, int nlev, int ny_s, int nx_s,
                           int ny_t, int nx_t, int jt_begin, int jt_end, const int *j0, const int *j1,
                           const double *wy, const int *i0, const int *i1, const double *wx, float *scratch,
                           void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PGW_B200_H */
