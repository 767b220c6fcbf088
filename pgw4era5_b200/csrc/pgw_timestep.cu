// The fused per-timestep column kernel of libpgw_b200 (sm_100a).
//
// One thread owns one ERA5 column; a warp is 32 adjacent longitudes, so every
// level access of a warp is one coalesced 128-byte line.  The column is swept
// bottom-up so that everything the surface-pressure iteration needs (the
// levels between the surface and p_ref) is seen first and parked in shared
// memory; after the iteration the rest of the column is streamed through
// registers with the adjusted surface pressure already known.  Each input
// element is read once and each output element written once.
//
// Reference semantics restated here (menschj/PGW4ERA5):
//   step_03_apply_to_era.py:64-94    pressures, RELHUM
//   step_03_apply_to_era.py:103-146  sea ice, skin and soil temperature
//   functions.py:288-292             two-point time interpolation of deltas
//   functions.py:343-366, 369-431    surface insertion + vertical interpolation
//   functions.py:511-580             interp_extrap_1d ('constant' mode)
//   step_03_apply_to_era.py:158-173  delta application
//   step_03_apply_to_era.py:182-319  surface-pressure fixed point
//   functions.py:118-125, 128-189    hus from RH, geopotential integration
#include "pgw_column.cuh"

#include <cuda_pipeline.h>
#include <stdlib.h>
#include <string.h>

namespace pgw {

// Downward merge walk over the pressure-ascending source nodes of one pair of
// variables (interp_extrap_1d in 'constant' mode, functions.py:511-580).
// State: lo node (index, pressure, values) and the differences to the hi node.
// inv_w == 0 encodes "no interpolation": at/after the last node, or (after the
// walk has passed node 0) before the first node; then the lo values are returned.
// The node below lo is prefetched as raw (lo, hi) time slabs and blended when used.
struct Walk2 {
    int lo;                 // index of the lo node; -1 once the target is above node 0
    float p_lo, inv_p_lo, inv_w;
    float a_lo, a_d, b_lo, b_d;
    float a_n0, a_n1, b_n0, b_n1;     // raw slabs of node lo-1
    float a_m0, a_m1, b_m0, b_m1;     // raw slabs of node lo-2 (loads issued two advances ahead)
};

constexpr int kRing = 5;     // levels in flight per thread (cp.async ring, +1 spare slot)

// REF: the dtypes the reference computes in on a file with float32 PS and FIS (PGW_FLAG_REF_DTYPES): float32
// delta_ps / ps_pgw, the half-level geopotential as a float32 running sum that is rounded on every level, for the
// ERA state and for the PGW state of every iteration, pressures as the two rounded operations ak + ps*bk.
// LOCAL: PGW_FLAG_LOCAL_PREF, p_ref per column and iteration among zg's levels (step_03:219-251).  Phase 1
// records the ERA-state sums at every candidate level (the `ncand` zg levels >= p_floor) the column's p_ref can
// move up to; phase 2 re-picks p_ref in every iteration and integrates the parked levels up to it.
// RI: PGW_FLAG_REINTERP, i_reinterp = 1 (step_03:155-173, :202-216, :330-343).  The stash holds the ERA state
// (T, RELHUM); every iteration after the first re-interpolates it, in ln p, onto that iteration's pressures
// and adds the deltas there.  `replay` (RI only, else null): pgw_timestep_finalize's relaunch that rewrites the
// outputs for iteration N when the speculative run went further (see PGW_FLAG_REINTERP in the header).
template <int NT, bool FAST, bool REF, bool LOCAL = false, bool RI = false>
__global__ void __launch_bounds__(NT, REF ? 2 : 3)
pgw_column_kernel(const __grid_constant__ pgw_timestep_args a, const int lst, const int np, const int ncand,
                  const pgw_timestep_result *replay) {
    static_assert(!(REF && LOCAL), "PGW_FLAG_LOCAL_PREF runs with float64 accumulation only");
    static_assert(!(RI && (REF || LOCAL)), "PGW_FLAG_REINTERP runs with a scalar p_ref and float64 accumulation");
    int k_spec = a.k_spec;
    if constexpr (RI) {
        if (replay) {                       // the same word for every thread: the whole grid returns or runs
            if (!replay->rewritten) return;
            k_spec = replay->n_iter;
        }
    }
    extern __shared__ __align__(16) unsigned char smem[];
    const int L = a.nlev, K = a.nplev;
    // ---- shared memory carve-up
    double2 *s_hl = reinterpret_cast<double2 *>(smem);                  // [L+1] (ak, bk)
    float2 *st_Te = reinterpret_cast<float2 *>(s_hl + (L + 1));         // [np][NT] (T_pgw rounded to fp32, e_pgw)
    float *ring = reinterpret_cast<float *>(st_Te + (size_t)np * NT);   // [kRing+1][4][NT]
    float2 *s_m = reinterpret_cast<float2 *>(ring + (size_t)(kRing + 1) * 4 * NT);   // [L] (akm, bkm)
    float *s_plev = reinterpret_cast<float *>(s_m + L);                 // [K] ascending
    float *s_inv_plev = s_plev + K;                                     // [K]
    float *s_inv_w = s_inv_plev + K;                                    // [K] 1/log2(p[j+1]/p[j])
    float *st_r = s_inv_w + K;                                          // REF: [np][NT] (T_era + dta) - fp32 T_pgw
    // LOCAL: zg's levels in file order, the candidates by descending pressure, per candidate and column
    // (phi_era - FIS, residual sum) at that pressure, and the candidate slot of each zg level (-1: below p_floor)
    double *s_zgp = reinterpret_cast<double *>((reinterpret_cast<uintptr_t>(st_r) + 15) & ~uintptr_t(15));  // [nzg]
    double *s_cp = s_zgp + a.nzg;                                                                            // [ncand]
    double2 *st_c = reinterpret_cast<double2 *>((reinterpret_cast<uintptr_t>(s_cp + ncand) + 15) & ~uintptr_t(15));
    int *s_slot = reinterpret_cast<int *>(st_c + (size_t)ncand * NT);                                       // [nzg]

    const int tid = threadIdx.x;
    for (int i = tid; i <= L; i += NT) s_hl[i] = make_double2(a.ak[i], a.bk[i]);
    for (int i = tid; i < L; i += NT) s_m[i] = make_float2((float)a.akm[i], (float)a.bkm[i]);
    for (int i = tid; i < K; i += NT) {
        const int f0 = a.plev_descending ? (K - 1 - i) : i;
        const float p0 = (float)a.plev[f0];
        s_plev[i] = p0;
        s_inv_plev[i] = 1.0f / p0;
        if (i + 1 < K) {
            const float p1 = (float)a.plev[a.plev_descending ? (K - 2 - i) : (i + 1)];
            s_inv_w[i] = 1.0f / log2f(p1 / p0);
        } else s_inv_w[i] = 0.0f;
    }
    if constexpr (LOCAL) {
        for (int i = tid; i < a.nzg; i += NT) {
            const double p = a.zg_plev[i];
            int r = -1;
            if (p >= a.p_floor) {
                r = 0;
                for (int j = 0; j < a.nzg; ++j) r += (a.zg_plev[j] >= a.p_floor && a.zg_plev[j] > p);
                s_cp[r] = p;
            }
            s_zgp[i] = p;
            s_slot[i] = r;
        }
    }
    __syncthreads();

    const uint32_t n = (uint32_t)a.ncol;
    uint32_t c = blockIdx.x * NT + tid;
    // Threads past the last column mirror column n-1: they compute and store exactly the
    // same values to the same addresses, which keeps the whole kernel free of tail branches.
    if (c >= n) c = n - 1;
    unsigned errbits = 0;
    int k_pref = INT32_MAX, k_bound = INT32_MAX;     // first iteration in which the two ps-dependent checks fired

    // ---- async ring: this thread's T, QV, U, V of one level per slot
    const float *gT = a.T, *gQ = a.QV, *gU = a.U, *gV = a.V;
    float *oT = a.T_out, *oQ = a.QV_out, *oU = a.U_out, *oV = a.V_out;
    float *const my_ring = ring + tid;
    int slot_w = 0;                                  // slot the next prefetch writes
    uint32_t off_w = (uint32_t)(L - 1) * n + c;      // element offset of the next prefetched level
    int lev_w = L - 1;
    // `zero` is 0, but computed from values just read out of the slot about to be overwritten
    // (pair loops): it makes the async copy wait for those shared-memory reads.
    auto prefetch = [&](int zero = 0) {
        if (lev_w >= 0) {
            float *dst = my_ring + slot_w * (4 * NT) + zero;
            __pipeline_memcpy_async(dst, gT + off_w, 4);
            __pipeline_memcpy_async(dst + NT, gQ + off_w, 4);
            __pipeline_memcpy_async(dst + 2 * NT, gU + off_w, 4);
            __pipeline_memcpy_async(dst + 3 * NT, gV + off_w, 4);
        }
        __pipeline_commit();
        --lev_w; off_w -= n;
        slot_w = (slot_w == kRing) ? 0 : slot_w + 1;
    };
#pragma unroll
    for (int i = 0; i < kRing; ++i) prefetch();
    int slot_r = 0;                                  // slot the next level is read from

    // ---------------- surface, skin and soil (step_03:103-146) ----------------
    const float ps_f = __ldg(a.PS + c);
    const Pair2 r_sic = load_pair(a.siconc, c), r_ts = load_pair(a.ts, c), r_tos = load_pair(a.tos, c);
    const Pair2 r_psh = load_pair(a.ps_hist, c), r_tas = load_pair(a.tas, c), r_hurs = load_pair(a.hurs, c);
    Pair2 r_zg{0.0f, 0.0f};
    if constexpr (!LOCAL) r_zg = load_pair(a.zg_ref, c);
    const float r_ice = __ldg(a.FR_SEA_ICE + c), r_land = __ldg(a.FR_LAND + c), r_skin = __ldg(a.T_SKIN + c);
    const float r_clim = __ldg(a.ts_clim + c), r_fis = __ldg(a.FIS + c);
    const double PSd = (double)ps_f;
    {
        // FR_SEA_ICE is float32 in the file and updated in place there
        float sic = (float)((double)r_ice + blend_f64(a.siconc, r_sic) / 100.0);
        sic = sic < 0.0f ? 0.0f : (sic > 1.0f ? 1.0f : sic);           // np.clip keeps NaN
        const double dts = blend_f64(a.ts, r_ts);
        const double dtos = blend_f64(a.tos, r_tos);
        double comb = dts;                                            // integrate_tos
        if (!isnan(sic) && !isnan(dtos)) {
            float fr = sic + r_land;
            fr = fr < 0.0f ? 0.0f : (fr > 1.0f ? 1.0f : fr);
            comb = (double)fr * dts + (double)(1.0f - fr) * dtos;
        }
        const double clim = (double)r_clim;
        a.FR_SEA_ICE_out[c] = sic;
        a.T_SKIN_out[c] = (float)((double)r_skin + comb);
        for (int s = 0; s < a.nsoil; ++s) {
            const double dso = clim + a.soil_decay[s] * (comb - clim);
            a.T_SO_out[(uint32_t)s * n + c] = (float)((double)__ldg(a.T_SO + (uint32_t)s * n + c) + dso);
        }
    }

    // ---------------- delta walkers (functions.py:343-431) ----------------
    // The 3-D deltas are packed per node and column as float4 (ta, hur, ua, va): walker A reads the
    // .xy half, walker B the .zw half (`pair` = 0 / 1), one 8-byte load per time slab.
    const float w_t = slab_weight(a.d4);
    const float2 *const d4lo = reinterpret_cast<const float2 *>(a.d4.lo);
    const float2 *const d4hi = reinterpret_cast<const float2 *>(a.d4.hi);
    const int desc = a.plev_descending;
    // raw loads of node j of a variable pair (time slabs lo/hi); blended when consumed
    auto load_raw = [&](int pair, int j, float &a0, float &a1, float &b0, float &b1) {
        const uint32_t off = ((uint32_t)(desc ? (K - 1 - j) : j) * n + c) * 2u + pair;
        const float2 x0 = __ldg(d4lo + off), x1 = __ldg(d4hi + off);
        a0 = x0.x; b0 = x0.y; a1 = x1.x; b1 = x1.y;
    };
    auto blend = [&](float x0, float x1) { return blend_f32(w_t, x0, x1); };
    // The register prefetch above covers two advances (~2 levels of work), less than a DRAM
    // round trip under load; the lines of node j are therefore pulled into L2 kL2Ahead
    // advances ahead, which costs neither registers nor shared memory.
    auto l2_prefetch = [&](int pair, int j) {
        const uint32_t off = ((uint32_t)(desc ? (K - 1 - j) : j) * n + c) * 2u + pair;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(d4lo + off));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(d4hi + off));
    };

    Walk2 wA, wB;
    // Both walkers at the bottom of the column (RI: again at the start of every iteration's sweep).
    auto init_walkers = [&]() {
        // replace_delta_sfc: node s carries (ps_hist, surface delta); the nodes after it all
        // hold the surface delta, so node s acts as the last node of the column.
        const float psh = (float)blend_f64(a.ps_hist, r_psh);
        int s = K - 1;
        if (!(psh > s_plev[K - 1])) {
            s = -1;
            for (int k = K - 1; k >= 0; --k)
                if (s_plev[k] < psh) { s = k; break; }
        }
        if (s < 0) { errbits |= PGW_ERR_PS_HIST_RANGE; s = 0; }
        wA.lo = s; wA.p_lo = psh; wA.inv_p_lo = fast_rcp(psh); wA.inv_w = 0.0f;
        wA.a_lo = (float)blend_f64(a.tas, r_tas); wA.a_d = 0.0f;
        wA.b_lo = (float)blend_f64(a.hurs, r_hurs); wA.b_d = 0.0f;
        wA.a_n0 = wA.a_n1 = wA.b_n0 = wA.b_n1 = 0.0f;
        wA.a_m0 = wA.a_m1 = wA.b_m0 = wA.b_m1 = 0.0f;
        if (s >= 1) load_raw(0, s - 1, wA.a_n0, wA.a_n1, wA.b_n0, wA.b_n1);
        if (s >= 2) load_raw(0, s - 2, wA.a_m0, wA.a_m1, wA.b_m0, wA.b_m1);

        float x0, x1, y0, y1;
        load_raw(1, K - 1, x0, x1, y0, y1);
        wB.lo = K - 1; wB.p_lo = s_plev[K - 1]; wB.inv_p_lo = s_inv_plev[K - 1]; wB.inv_w = 0.0f;
        wB.a_lo = blend(x0, x1); wB.a_d = 0.0f;
        wB.b_lo = blend(y0, y1); wB.b_d = 0.0f;
        load_raw(1, K - 2, wB.a_n0, wB.a_n1, wB.b_n0, wB.b_n1);
        wB.a_m0 = wB.a_m1 = wB.b_m0 = wB.b_m1 = 0.0f;
        if (K >= 3) load_raw(1, K - 3, wB.a_m0, wB.a_m1, wB.b_m0, wB.b_m1);
#pragma unroll
        for (int d = 3; d <= kL2Ahead; ++d) {
            if (s - d >= 0) l2_prefetch(0, s - d);
            if (K - 1 - d >= 0) l2_prefetch(1, K - 1 - d);
        }
    };
    init_walkers();
    float min_src_p = (wA.lo == 0) ? wA.p_lo : s_plev[0];

    // One downward step of a walker, split in two so that the steps of both walkers can be
    // ordered "consume, consume, load, load": the prefetched registers of a walker are read
    // (which waits for loads issued one step, i.e. several levels, ago) before ANY new load is
    // issued.  Issued the other way round, the second walker's register reads wait on the
    // scoreboard of the first walker's brand-new loads: a full DRAM round trip per step.
    auto step_consume = [&](Walk2 &w) {
        const float hi_p = w.p_lo, hi_a = w.a_lo, hi_b = w.b_lo;
        const bool from_synth = (hi_p != s_plev[w.lo]);     // leaving the (ps_hist, sfc) node
        --w.lo;
        if (w.lo >= 0) {
            w.p_lo = s_plev[w.lo]; w.inv_p_lo = s_inv_plev[w.lo];
            w.a_lo = blend(w.a_n0, w.a_n1); w.b_lo = blend(w.b_n0, w.b_n1);
            w.a_d = hi_a - w.a_lo; w.b_d = hi_b - w.b_lo;
            w.inv_w = from_synth ? fast_rcp(fast_lg2(hi_p * w.inv_p_lo)) : s_inv_w[w.lo];
            w.a_n0 = w.a_m0; w.a_n1 = w.a_m1; w.b_n0 = w.b_m0; w.b_n1 = w.b_m1;
        } else {
            // above node 0: constant extrapolation with node 0's values; p_lo = 0 ends the walk
            w.a_d = 0.0f; w.b_d = 0.0f; w.inv_w = 0.0f; w.p_lo = 0.0f; w.inv_p_lo = 1.0f;
        }
    };
    // `zero` (== 0) carries a data dependency on the registers consumed above
    auto step_load = [&](Walk2 &w, int pair, int zero) {
        if (w.lo >= 2) load_raw(pair, w.lo - 2 + zero, w.a_m0, w.a_m1, w.b_m0, w.b_m1);
        if (w.lo >= kL2Ahead) l2_prefetch(pair, w.lo - kL2Ahead);
    };
    // advance both walkers until p_lo <= p (or the first node has been passed)
    auto advance = [&](float p) {
        do {
            const bool sa = wA.p_lo > p, sb = wB.p_lo > p;
            if (sa) step_consume(wA);
            if (sb) step_consume(wB);
            const int zero = reg_fence(wA.a_n1, wA.b_n1, wB.a_n1, wB.b_n1);
            if (sa) step_load(wA, 0, zero);
            if (sb) step_load(wB, 1, zero);
        } while (fmaxf(wA.p_lo, wB.p_lo) > p);
    };

    LnConst lk{2.0 / 3.0, 2.0 / 5.0, 2.0 / 7.0};
    asm volatile("" : "+d"(lk.c3), "+d"(lk.c5), "+d"(lk.c7));     // keep the constants in registers

    double pref = a.p_ref;
    // LOCAL: jsel = index in zg_plev of p_ref_k (-1: none); cj = next candidate slot phase 1 records
    int jsel = -1, cj = 0;
    int k_nopref = INT32_MAX, k_floor = INT32_MAX;
    const double pe = 0.95 * PSd;                   // determine_p_ref's p_min_era (step_03:221-226)
    if constexpr (LOCAL) {
        for (int i = 0; i < a.nzg; ++i)
            if (pe > s_zgp[i]) { jsel = i; break; }   // first iteration: ps_pgw == PS, both tests agree
        if (jsel < 0) {
            errbits |= PGW_ERR_NO_PREF; k_nopref = 0; pref = NAN; cj = ncand;
        } else {
            pref = s_zgp[jsel];
            cj = s_slot[jsel];
            if (cj < 0) { errbits |= PGW_ERR_PREF_FLOOR; k_floor = 0; cj = ncand; }
        }
        a.pref_traj[c] = (uint8_t)(jsel < 0 ? 255 : jsel);
    }
    const int cj0 = cj;                             // LOCAL: slot of p_ref_1
    const double2 hl_sfc = s_hl[L];
    double pb_era = fma(PSd, hl_sfc.y, hl_sfc.x);
    double acc_era = 0.0;
    bool era_open = pb_era >= pref;                 // still below p_ref
    if (!era_open && !(LOCAL && jsel < 0)) { errbits |= PGW_ERR_PREF_BELOW_SFC; k_pref = 0; }
    float psn_f = ps_f;                             // ps used for QV; replaced after the iteration
    // REF: ak + ps*bk as numpy evaluates it (two rounded operations, step_03:64-66, :196-199)
    auto hyb = [](double ps, double2 h) { return __dadd_rn(h.x, __dmul_rn(ps, h.y)); };
    float phi32_era = r_fis;                        // REF: float32 half-level geopotential of the ERA state
    double phi_ref_era = 0.0;

    const auto read_fence = [](float x0, float x1, float x2, float x3) { return reg_fence(x0, x1, x2, x3); };
    // The per-level work is split into the (sequential, cheap) walker step and the (independent,
    // expensive) thermodynamics.  The sweeps process levels in PAIRS: both walker steps first,
    // then the thermodynamics of the two levels in one branch-free block so that the two
    // dependency chains interleave (the kernel is issue-latency bound, not DRAM bound).
    struct Dlt { float ta, hur, ua, va; };
    auto walk = [&](float p) {
        if (fmaxf(wA.p_lo, wB.p_lo) > p) advance(p);
        const float l2b = fast_lg2(p * wB.inv_p_lo);
        const float l2a = (wA.inv_p_lo == wB.inv_p_lo) ? l2b : fast_lg2(p * wA.inv_p_lo);
        const float tA = l2a * wA.inv_w, tB = l2b * wB.inv_w;
        // t == 0: exact node hit or constant extrapolation -> the node value itself (NaN-safe)
        Dlt d;
        d.ta = (tA == 0.0f) ? wA.a_lo : fmaf(tA, wA.a_d, wA.a_lo);
        d.hur = (tA == 0.0f) ? wA.b_lo : fmaf(tA, wA.b_d, wA.b_lo);
        d.ua = (tB == 0.0f) ? wB.a_lo : fmaf(tB, wB.a_d, wB.a_lo);
        d.va = (tB == 0.0f) ? wB.b_lo : fmaf(tB, wB.b_d, wB.b_lo);
        return d;
    };
    auto thermo = [&](bool cold, float p, float t, float q, const Dlt &d) -> float {
        return thermo_e_pgw(cold, p, t, q, d.ta, d.hur);
    };

    // ---------------- phase 1: surface .. p_ref, parked in shared memory ----------------
    uint32_t off = (uint32_t)(L - 1) * n + c;
    // T_pgw is parked as fp32.  Its rounding residual r_l (|r_l| <= 1.5e-5 K) enters the
    // geopotential as Rd * sum_l r_l dlnp_l; that sum is taken once with the ERA pressures
    // (its change over the iteration is < 1e-8 m2/s2) and added to every iteration's sum.
    double acc_res = 0.0, acc_pgw0 = 0.0, t_low_d = 0.0;
    // RI: the state of iteration 1 is the output only when it is the last one; later ones are written by the
    // last iteration's sweep
    const bool out1 = !RI || k_spec == 1;
    {
        float2 *pTe = st_Te + (size_t)(L - 1 - lst) * NT + tid;
        // ERA geopotential of one layer (functions.py:128-189), sequential in the column
        // The first iteration of the fixed point (dps = 0) integrates the PGW state over the
        // same pressures, so its sum is taken here as well and phase 2 starts at iteration 1.
        float *pTr = st_r + (size_t)(L - 1 - lst) * NT + tid;
        auto era_layer = [&](int l, float p, float t, float q, float dta, float t_pgw, float e_pgw) {
            if constexpr (REF) {
                const double tpd = (double)t_pgw;
                pTr[-(L - 1 - l) * NT] = (float)(((double)t + (double)dta) - tpd);
                if (era_open) {
                    const double Pt = hyb(PSd, s_hl[l]);
                    const double rtv = rd_tv(t, q);                  // CON_RD * tav, float32 products (:144, :151)
                    if (Pt < pref) {                                 // functions.py:174-179, float64
                        phi_ref_era = (double)phi32_era + rtv * ln_ratio_ref(pb_era, pref);
                        era_open = false;
                    } else {                                         // functions.py:147-152, stored as float32
                        phi32_era = (float)((double)phi32_era + rtv * ln_ratio_ref(pb_era, Pt));
                        pb_era = Pt;
                    }
                }
                return;
            }
            if constexpr (LOCAL) {
                // integ_geopot (functions.py:141-179) of the ERA state and of the residual, evaluated at every
                // candidate level inside this layer; the PGW sum of the first iteration stops at p_ref_1
                const double2 hl = s_hl[l];
                const double pt = fma(PSd, hl.y, hl.x);
                const double td = (double)t, tpd = (double)t_pgw;
                const double rtv = rd_tv(t, q);
                const float g = fast_rcp(fmaf(-0.378f, e_pgw, p));
                const double tvp = fma(tpd, (double)((0.61f * 0.622f) * e_pgw * g), tpd);
                const double res = (td + (double)dta) - tpd;
                for (; cj < ncand && s_cp[cj] > pt; ++cj) {
                    const double dl = ln_ratio<FAST>(pb_era, s_cp[cj], lk);
                    st_c[(size_t)cj * NT + tid] = make_double2(fma(rtv, dl, acc_era), fma(res, dl, acc_res));
                    if (cj == cj0) acc_pgw0 = fma(tvp, dl, acc_pgw0);
                }
                const double dl = ln_ratio<FAST>(pb_era, pt, lk);
                acc_era = fma(rtv, dl, acc_era);
                acc_res = fma(res, dl, acc_res);
                if (cj == cj0) acc_pgw0 = fma(tvp, dl, acc_pgw0);
                pb_era = pt;
                return;
            }
            if (era_open) {
                const double2 hl = s_hl[l];
                double pt = fma(PSd, hl.y, hl.x);
                if (pt < pref) { pt = pref; era_open = false; }     // layer that contains p_ref (:174-179)
                const double td = (double)t, tpd = (double)t_pgw;
                const double rtv = rd_tv(t, q);                      // Rd * Tv of the ERA state, float32 products
                const float g = fast_rcp(fmaf(-0.378f, e_pgw, p));
                const double tvp = fma(tpd, (double)((0.61f * 0.622f) * e_pgw * g), tpd);
                const double dl = ln_ratio<FAST>(pb_era, pt, lk);
                acc_era = fma(rtv, dl, acc_era);
                acc_pgw0 = fma(tvp, dl, acc_pgw0);
                acc_res = fma((td + (double)dta) - tpd, dl, acc_res);
                pb_era = pt;
            }
        };
        int l = L - 1;
        for (; l - 1 >= lst; l -= 2, off -= 2 * n, pTe -= 2 * NT) {
            __pipeline_wait_prior(kRing - 2);
            const float *sl0 = my_ring + slot_r * (4 * NT);
            const float t0 = sl0[0], q0 = sl0[NT], u0 = sl0[2 * NT], v0 = sl0[3 * NT];
            slot_r = (slot_r == kRing) ? 0 : slot_r + 1;
            const float *sl1 = my_ring + slot_r * (4 * NT);
            const float t1 = sl1[0], q1 = sl1[NT], u1 = sl1[2 * NT], v1 = sl1[3 * NT];
            slot_r = (slot_r == kRing) ? 0 : slot_r + 1;
            const float2 m0 = s_m[l], m1 = s_m[l - 1];
            prefetch(); prefetch(read_fence(t0, q0, u0, v0));   // 2nd copy reuses the slot of level l
            const float p0 = fmaf(ps_f, m0.y, m0.x), p1 = fmaf(ps_f, m1.y, m1.x);
            const Dlt d0 = walk(p0);
            const Dlt d1 = walk(p1);
            const bool cold = __all_sync(0xffffffffu, is_cold(t0, d0.ta) && is_cold(t1, d1.ta));
            const float e0 = thermo(cold, p0, t0, q0, d0), e1 = thermo(cold, p1, t1, q1, d1);
            const float tp0 = t0 + d0.ta, tp1 = t1 + d1.ta;   // == (float)((double)t + (double)dta)
            if (out1) {
                st_stream(oT + off, tp0); st_stream(oU + off, u0 + d0.ua); st_stream(oV + off, v0 + d0.va);
                st_stream(oT + off - n, tp1); st_stream(oU + off - n, u1 + d1.ua); st_stream(oV + off - n, v1 + d1.va);
                if constexpr (RI) { st_stream(oQ + off, qv_from_e(e0, ps_f, m0)); st_stream(oQ + off - n, qv_from_e(e1, ps_f, m1)); }
            }
            if constexpr (RI) {
                pTe[0] = make_float2(t0, rh_era_f32(p0, t0, q0));
                pTe[-NT] = make_float2(t1, rh_era_f32(p1, t1, q1));
            } else {
                pTe[0] = make_float2(tp0, e0);
                pTe[-NT] = make_float2(tp1, e1);
            }
            if (l == L - 1) t_low_d = (double)t0 + (double)d0.ta;
            era_layer(l, p0, t0, q0, d0.ta, tp0, e0);
            era_layer(l - 1, p1, t1, q1, d1.ta, tp1, e1);
        }
        if (l >= lst) {                                   // odd number of parked levels
            __pipeline_wait_prior(kRing - 1);
            const float *sl0 = my_ring + slot_r * (4 * NT);
            const float t0 = sl0[0], q0 = sl0[NT], u0 = sl0[2 * NT], v0 = sl0[3 * NT];
            slot_r = (slot_r == kRing) ? 0 : slot_r + 1;
            const float2 m0 = s_m[l];
            prefetch();
            const float p0 = fmaf(ps_f, m0.y, m0.x);
            const Dlt d0 = walk(p0);
            const float e0 = thermo(false, p0, t0, q0, d0);
            const float tp0 = t0 + d0.ta;
            if (out1) {
                st_stream(oT + off, tp0); st_stream(oU + off, u0 + d0.ua); st_stream(oV + off, v0 + d0.va);
                if constexpr (RI) st_stream(oQ + off, qv_from_e(e0, ps_f, m0));
            }
            if constexpr (RI) pTe[0] = make_float2(t0, rh_era_f32(p0, t0, q0));
            else pTe[0] = make_float2(tp0, e0);
            if (l == L - 1) t_low_d = (double)t0 + (double)d0.ta;
            era_layer(l, p0, t0, q0, d0.ta, tp0, e0);
            off -= n;
        }
    }
    const double fis = (double)r_fis;
    double phi_era = REF ? phi_ref_era : fis + acc_era;              // acc_era holds Rd * Tv * dlnp
    double gdzg = blend_f64(a.zg_ref, r_zg) * kG;                    // step_03:292-295
    // LOCAL: phi_era, the residual sum and the climate term (the zg delta of both time slabs, blended) at zg
    // level j; a level below p_floor is outside the stash: flagged, the values are left as they are
    auto take_level = [&](int j, int k) {
        const int s = s_slot[j];
        if (s < 0) {
            errbits |= PGW_ERR_PREF_FLOOR; k_floor = min(k_floor, k);
        } else {
            const double2 v = st_c[(size_t)s * NT + tid];
            phi_era = fis + v.x;
            acc_res = v.y;
        }
        gdzg = blend_f64(a.zg, load_pair(a.zg, (uint32_t)j * n + c)) * kG;
    };
    if constexpr (LOCAL) {
        if (jsel >= 0) take_level(jsel, 0);
        else phi_era = NAN;
    }
    const float2 *const bTe = st_Te + (size_t)(L - 1 - lst) * NT + tid;  // lowest level of the stash
    double t_low = t_low_d;                                       // ta_pgw on the lowest level (RI: per iteration)

    // ---------------- phase 2: surface-pressure fixed point (step_03:182-319) ----------------
    // The loads of the upper column are already in flight and overlap this phase.
    double dps = 0.0, adj = 0.0, psn = PSd;
    int ltop = lst + 1;                 // first layer (from the top) lying entirely below p_ref

    // RI: the ERA state at a target pressure of this iteration, interp_logp_4d in 'constant' mode
    // (functions.py:434-580, float64): a merge walk over the ERA levels (pressures akm + PS bkm) as the targets
    // move up the column.  lo = level rj, hi = level rj + 1.  A level comes from the stash, or from global
    // memory above it (a target lowered by dps < 0 brackets with level lst - 1) or in phase 3; U and V, needed
    // for the outputs only, from global memory.  Level `lring` takes (t, q, u, v) just read from the ring.
    struct Era { double pe; float t, r, u, v; };
    int rj = L - 1;
    Era elo{}, ehi{};
    double inv_den = 0.0;                                         // 1 / ln(p_hi / p_lo)
    auto era_at = [&](int j, bool uv, int lring, float t, float q, float u, float v) {
        Era x;
        x.pe = fma(PSd, __ldg(a.bkm + j), __ldg(a.akm + j));
        const uint32_t o = (uint32_t)j * n + c;
        if (j >= lst) {
            const float2 s = st_Te[(size_t)(j - lst) * NT + tid];
            x.t = s.x; x.r = s.y;
        } else {
            const float2 m = s_m[j];
            if (j != lring) { t = __ldg(gT + o); q = __ldg(gQ + o); }
            x.t = t;
            x.r = rh_era_f32(fmaf(ps_f, m.y, m.x), t, q);
        }
        if (uv && j != lring) { u = __ldg(gU + o); v = __ldg(gV + o); }
        x.u = uv ? u : 0.0f;
        x.v = uv ? v : 0.0f;
        return x;
    };
    auto win_reset = [&](int j, bool uv) { rj = j; elo = era_at(j, uv, -1, 0.0f, 0.0f, 0.0f, 0.0f); };
    // move the window down to target pt; returns the weight of hi, 0 for lo's value as it is (an exact hit,
    // or constant extrapolation below level L-1 or above level 0)
    auto win_move = [&](double pt, bool uv, int lring, float t, float q, float u, float v) -> double {
        while (rj > 0 && elo.pe > pt) {
            ehi = elo;
            --rj;
            elo = era_at(rj, uv, lring, t, q, u, v);
            inv_den = 1.0 / ln_ratio<false>(ehi.pe, elo.pe, lk);
        }
        // ln(pt / p_lo) from pt - p_lo (= bkm dps on the level itself): no float32 log of a ratio near 1
        return (rj == L - 1 || !(elo.pe < pt)) ? 0.0 : ln_ratio<false>(pt, elo.pe, lk) * inv_den;
    };
    auto lerp = [](double w, float lo, float hi) {
        return w == 0.0 ? (double)lo : fma(w, (double)hi - (double)lo, (double)lo);
    };
    // level l at this iteration's pressures: T_pgw (float64), e and 1/(p - 0.378 e) (functions.py:118-125),
    // with `uv` also U and V
    struct RiLev { double tp, u, v; float e, g; };
    auto ri_level = [&](int l, bool uv, int lring, float t, float q, float u, float v) {
        const double pt = fma(psn, __ldg(a.bkm + l), __ldg(a.akm + l));
        const float2 m = s_m[l];
        const float ptf = fmaf(psn_f, m.y, m.x);
        const double w = win_move(pt, uv, lring, t, q, u, v);
        const Dlt d = walk(ptf);
        RiLev r;
        r.tp = lerp(w, elo.t, ehi.t) + (double)d.ta;
        const float rh = (float)(lerp(w, elo.r, ehi.r) + (double)d.hur);
        r.e = rh * 0.01f * es_water_ice((float)(r.tp - 273.0));
        r.g = fast_rcp(fmaf(-0.378f, r.e, ptf));
        r.u = uv ? lerp(w, elo.u, ehi.u) + (double)d.ua : 0.0;
        r.v = uv ? lerp(w, elo.v, ehi.v) + (double)d.va : 0.0;
        return r;
    };
    auto ri_store = [&](int l, const RiLev &r) {
        const uint32_t o = (uint32_t)l * n + c;
        st_stream(oT + o, (float)r.tp);
        st_stream(oQ + o, 0.622f * r.e * r.g);
        st_stream(oU + o, (float)r.u);
        st_stream(oV + o, (float)r.v);
    };

    float *traj = a.dps_traj + c;
    for (int k = 0; k < k_spec; ++k, traj += n) {
        if constexpr (REF) {
            // delta_ps is float32 (zeros_like(PS)) and += keeps that; ps_pgw = PS + delta_ps is a float32 sum
            // (step_03_apply_to_era.py:186-195)
            const float dps32 = (float)(dps + adj);
            dps = (double)dps32;
            psn_f = __fadd_rn(ps_f, dps32);
            psn = (double)psn_f;
        } else {
            dps += adj;
            psn = PSd + dps;
            psn_f = (float)psn;
        }
        *traj = (float)dps;
        if (psn > a.ps_bound) { errbits |= PGW_ERR_PS_BOUND; k_bound = min(k_bound, k); }
        if constexpr (LOCAL) {
            if (k > 0) {
                // determine_p_ref (functions.py:583-598): the first zg level, in file order, below 0.95 PS and
                // 0.95 ps_pgw, at most the previous choice (min(p, p_ref_last) ignores a NaN p_ref_last)
                const double pp = 0.95 * psn;
                int j = -1;
                for (int i = 0; i < a.nzg; ++i) {
                    const double p = s_zgp[i];
                    if (pe > p && pp > p) { j = i; break; }
                }
                if (j < 0) { errbits |= PGW_ERR_NO_PREF; k_nopref = min(k_nopref, k); }
                else if (jsel >= 0 && !(s_zgp[j] < pref)) j = jsel;
                if (j != jsel) {
                    jsel = j;
                    if (j < 0) { pref = NAN; phi_era = NAN; }
                    else { pref = s_zgp[j]; take_level(j, k); }
                }
                a.pref_traj[(size_t)k * n + c] = (uint8_t)(jsel < 0 ? 255 : jsel);
            }
        }
        double pb = REF ? hyb(psn, hl_sfc) : fma(psn, hl_sfc.y, hl_sfc.x);
        if (pb < pref) { errbits |= PGW_ERR_PREF_BELOW_SFC; k_pref = min(k_pref, k); }
        if constexpr (REF) {
            // integ_geopot of the PGW state with the float32 half-level geopotential (functions.py:141-152)
            float phi32 = r_fis;
            double phi_pgw = 0.0;
            bool open = true;
            const float2 *pTe = bTe;
            const float *pTr = st_r + (size_t)(L - 1 - lst) * NT + tid;
            for (int l = L - 1; l >= lst; --l, pTe -= NT, pTr -= NT) {
                const float2 m = s_m[l];
                const float2 te = *pTe;
                const double Td = (double)te.x + (double)*pTr;
                const double Pt = hyb(psn, s_hl[l]);
                const float g = fast_rcp(fmaf(-0.378f, te.y, fmaf(psn_f, m.y, m.x)));
                const double rtv = kRd * (Td * (1.0 + (double)((0.61f * 0.622f) * te.y * g)));
                if (Pt < pref) {
                    phi_pgw = (double)phi32 + rtv * ln_ratio_ref(pb, pref);
                    open = false;
                    break;
                }
                phi32 = (float)((double)phi32 + rtv * ln_ratio_ref(pb, Pt));
                pb = Pt;
            }
            if (open) { phi_pgw = (double)phi32; errbits |= PGW_ERR_PS_BOUND; k_bound = min(k_bound, k); }
            const double err = (phi_pgw - phi_era) - gdzg;
            // -adj_factor * ps_pgw is a float32 product (python scalar x float32 array, step_03:302-303)
            const float aps = __fmul_rn((float)(-a.adj_factor), psn_f);
            adj = (double)aps / (kRd * t_low) * err;
            double ae = isnan(err) ? 0.0 : fabs(err);
            ae = warp_max(ae);
            if ((tid & 31) == 0 && ae > 0.0)
                atomicMax(reinterpret_cast<unsigned long long *>(a.maxerr + k),
                          (unsigned long long)__double_as_longlong(ae));
            continue;
        }
        double acc = acc_res;
        if (k == 0) {
            acc += acc_pgw0;            // psn == PS: summed in phase 1 together with the ERA state
        } else if constexpr (RI) {
            // re-interpolate the parked levels bottom-up to the layer that contains p_ref (step_03:202-216);
            // the last iteration goes on over every parked level and writes its state
            const bool last = k == k_spec - 1;
            init_walkers();
            win_reset(L - 1, last);
            acc = 0.0;                  // T_pgw is formed in float64: no fp32 residual
            bool open = pb >= pref;
            for (int l = L - 1; l >= lst; --l) {
                const RiLev r = ri_level(l, last, -1, 0.0f, 0.0f, 0.0f, 0.0f);
                if (l == L - 1) t_low = r.tp;                           // ta_pgw[:, -1] of this iteration
                if (open) {
                    const double tv = fma(r.tp, (double)((0.61f * 0.622f) * r.e * r.g), r.tp);
                    const double2 hl = s_hl[l];
                    const double pt = fma(psn, hl.y, hl.x);
                    if (pt < pref) {                                    // layer that contains p_ref (:174-179)
                        acc = fma(tv, ln_ratio<FAST>(pb, pref, lk), acc);
                        open = false;
                    } else {
                        acc = fma(tv, ln_ratio<FAST>(pb, pt, lk), acc);
                        pb = pt;
                    }
                }
                if (last) ri_store(l, r);
                else if (!open) break;
            }
        } else {
        // layers ltop..L-1 are entirely below p_ref for this ps; it moves by at most a level or two
        while (ltop > lst) { const double2 h = s_hl[ltop - 1]; if (fma(psn, h.y, h.x) >= pref) --ltop; else break; }
        while (ltop < L) { const double2 h = s_hl[ltop]; if (fma(psn, h.y, h.x) < pref) ++ltop; else break; }
        const float2 *pTe = bTe;
        int l = L - 1;
#pragma unroll 4
        for (; l >= ltop; --l, pTe -= NT) {
            const double2 hl = s_hl[l];
            const float2 m = s_m[l];
            const float2 te = *pTe;
            const float e = te.y;
            const double Td = (double)te.x;
            const double pt = fma(psn, hl.y, hl.x);
            // Tv = T (1 + 0.61 hus), hus = 0.622 e / (p - 0.378 e)   (functions.py:66-72, :144)
            const float g = fast_rcp(fmaf(-0.378f, e, fmaf(psn_f, m.y, m.x)));
            const double tv = fma(Td, (double)((0.61f * 0.622f) * e * g), Td);
            acc = fma(tv, ln_ratio<FAST>(pb, pt, lk), acc);
            pb = pt;
        }
        if (l >= lst && pb >= pref) {                              // layer that contains p_ref (:174-179)
            const float2 m = s_m[l];
            const float2 te = *pTe;
            const float e = te.y;
            const double Td = (double)te.x;
            const float g = fast_rcp(fmaf(-0.378f, e, fmaf(psn_f, m.y, m.x)));
            const double tv = fma(Td, (double)((0.61f * 0.622f) * e * g), Td);
            acc = fma(tv, ln_ratio<FAST>(pb, pref, lk), acc);
        }
        }
        const double phi_pgw = fis + kRd * acc;
        const double err = (phi_pgw - phi_era) - gdzg;
        adj = -a.adj_factor * psn / (kRd * t_low) * err;
        double ae = isnan(err) ? 0.0 : fabs(err);                  // max skips NaN (step_03:308)
        ae = warp_max(ae);
        if ((tid & 31) == 0 && ae > 0.0)
            atomicMax(reinterpret_cast<unsigned long long *>(a.maxerr + k),
                      (unsigned long long)__double_as_longlong(ae));
    }

    // ---------------- phase 3: PS, QV of the parked levels, then the upper column ----------------
    if constexpr (LOCAL) a.p_ref_out[c] = jsel < 0 ? (double)NAN : s_zgp[jsel];
    a.PS_out[c] = psn_f;
    a.dps_out[c] = (float)dps;
    if constexpr (RI) {
        // the upper column at the final pressures (step_03:330-343 for U and V); the window goes on from the
        // top of the stash (the last sweep left it there; with one iteration, place it there)
        if (k_spec == 1) win_reset(lst, true);
        for (int l = lst - 1; l >= 0; --l) {
            __pipeline_wait_prior(kRing - 1);
            const float *sl0 = my_ring + slot_r * (4 * NT);
            const float t0 = sl0[0], q0 = sl0[NT], u0 = sl0[2 * NT], v0 = sl0[3 * NT];
            slot_r = (slot_r == kRing) ? 0 : slot_r + 1;
            prefetch();                                  // overwrites the slot read one level ago
            ri_store(l, ri_level(l, true, l, t0, q0, u0, v0));
        }
    } else {
    {
        const float2 *pTe = bTe;
        uint32_t o2 = (uint32_t)(L - 1) * n + c;
        for (int l = L - 1; l >= lst; --l, pTe -= NT, o2 -= n) {
            const float2 m = s_m[l];
            const float e = pTe->y;
            st_stream(oQ + o2, 0.622f * e * fast_rcp(fmaf(-0.378f, e, fmaf(psn_f, m.y, m.x))));
        }
    }
    {
        auto qv_of = [&](float e, float2 m) {     // functions.py:66-72 with the adjusted ps
            return 0.622f * e * fast_rcp(fmaf(-0.378f, e, fmaf(psn_f, m.y, m.x)));
        };
        int l = lst - 1;
        for (; l - 1 >= 0; l -= 2, off -= 2 * n) {
            __pipeline_wait_prior(kRing - 2);
            const float *sl0 = my_ring + slot_r * (4 * NT);
            const float t0 = sl0[0], q0 = sl0[NT], u0 = sl0[2 * NT], v0 = sl0[3 * NT];
            slot_r = (slot_r == kRing) ? 0 : slot_r + 1;
            const float *sl1 = my_ring + slot_r * (4 * NT);
            const float t1 = sl1[0], q1 = sl1[NT], u1 = sl1[2 * NT], v1 = sl1[3 * NT];
            slot_r = (slot_r == kRing) ? 0 : slot_r + 1;
            const float2 m0 = s_m[l], m1 = s_m[l - 1];
            prefetch(); prefetch(read_fence(t0, q0, u0, v0));
            const float p0 = fmaf(ps_f, m0.y, m0.x), p1 = fmaf(ps_f, m1.y, m1.x);
            const Dlt d0 = walk(p0);
            const Dlt d1 = walk(p1);
            const bool cold = __all_sync(0xffffffffu, is_cold(t0, d0.ta) && is_cold(t1, d1.ta));
            const float e0 = thermo(cold, p0, t0, q0, d0), e1 = thermo(cold, p1, t1, q1, d1);
            st_stream(oT + off, t0 + d0.ta); st_stream(oU + off, u0 + d0.ua); st_stream(oV + off, v0 + d0.va);
            st_stream(oQ + off, qv_of(e0, m0));
            st_stream(oT + off - n, t1 + d1.ta); st_stream(oU + off - n, u1 + d1.ua); st_stream(oV + off - n, v1 + d1.va);
            st_stream(oQ + off - n, qv_of(e1, m1));
        }
        if (l >= 0) {
            __pipeline_wait_prior(kRing - 1);
            const float *sl0 = my_ring + slot_r * (4 * NT);
            const float t0 = sl0[0], q0 = sl0[NT], u0 = sl0[2 * NT], v0 = sl0[3 * NT];
            slot_r = (slot_r == kRing) ? 0 : slot_r + 1;
            const float2 m0 = s_m[l];
            prefetch();
            const float p0 = fmaf(ps_f, m0.y, m0.x);
            const Dlt d0 = walk(p0);
            const float e0 = thermo(false, p0, t0, q0, d0);
            st_stream(oT + off, t0 + d0.ta); st_stream(oU + off, u0 + d0.ua); st_stream(oV + off, v0 + d0.va);
            st_stream(oQ + off, qv_of(e0, m0));
            off -= n;
        }
    }
    }
    __pipeline_wait_prior(0);

    // ---------------- bookkeeping for the host-side checks ----------------
    float p_top = fmaf(ps_f, s_m[0].y, s_m[0].x);                        // functions.py:417
    if constexpr (RI) p_top = fminf(p_top, fmaf(psn_f, s_m[0].y, s_m[0].x));    // targets of the last iteration
    p_top = warp_min(p_top);
    min_src_p = warp_min(min_src_p);
    if ((tid & 31) == 0) {
        atomicMin(reinterpret_cast<unsigned *>(a.stats), __float_as_uint(fmaxf(p_top, 0.0f)));
        atomicMin(reinterpret_cast<unsigned *>(a.stats) + 1, __float_as_uint(fmaxf(min_src_p, 0.0f)));
    }
    if (errbits) {
        atomicOr(a.err, errbits);
        if (a.first_k) {
            if (k_pref != INT32_MAX) atomicMin(a.first_k, k_pref);
            if (k_bound != INT32_MAX) atomicMin(a.first_k + 1, k_bound);
            if constexpr (LOCAL) {
                if (k_nopref != INT32_MAX) atomicMin(a.first_k + 2, k_nopref);
                if (k_floor != INT32_MAX) atomicMin(a.first_k + 3, k_floor);
            }
        }
    }
}

__global__ void pgw_timestep_init_kernel(uint64_t *maxerr, float *stats, uint32_t *err, int32_t *first_k,
                                         uint32_t *poly_fallback) {
    const int i = threadIdx.x;
    if (i == 0 && poly_fallback) *poly_fallback = 0u;
    if (i < PGW_MAX_ITER) maxerr[i] = 0ull;
    if (i < 2) stats[i] = INFINITY;
    if (i < 4 && first_k) first_k[i] = INT32_MAX;
    if (i == 0) *err = 0u;
}

// N = first k with max|err_k| <= thresh (step_03:189,308)
__global__ void pgw_converge_kernel(const uint64_t *maxerr, int k_spec, double thresh,
                                    pgw_timestep_result *res) {
    int n_iter = 0;
    for (int k = 0; k < k_spec; ++k) {
        const double e = __longlong_as_double((long long)maxerr[k]);
        if (!(e > thresh)) { n_iter = k + 1; break; }
    }
    res->n_iter = n_iter;
    res->converged = n_iter > 0;
    res->rewritten = (n_iter > 0 && n_iter < k_spec);
    res->reserved = 0;
}

// If the field converged before k_spec, PS and QV (and p_ref) were written for iteration k_spec;
// rewrite them for iteration N.  e_pgw is recovered from the speculative QV.
__global__ void __launch_bounds__(256)
pgw_rewrite_kernel(const __grid_constant__ pgw_timestep_args a, const pgw_timestep_result *res) {
    if (!res->rewritten) return;
    const long long n = a.ncol;
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    const int N = res->n_iter;
    if (a.flags & PGW_FLAG_LOCAL_PREF) {
        const int j = a.pref_traj[(long long)(N - 1) * n + c];
        a.p_ref_out[c] = j < a.nzg ? a.zg_plev[j] : (double)NAN;
    }
    const double PSd = (double)a.PS[c];
    const double dps_n = (double)a.dps_traj[(long long)(N - 1) * n + c];
    const double dps_s = (double)a.dps_traj[(long long)(a.k_spec - 1) * n + c];
    double ps_n = PSd + dps_n, ps_s = PSd + dps_s;
    if (a.flags & PGW_FLAG_REF_DTYPES) { ps_n = (double)(float)ps_n; ps_s = (double)(float)ps_s; }   // float32 ps_pgw
    a.PS_out[c] = (float)ps_n;
    a.dps_out[c] = (float)dps_n;
    for (int l = 0; l < a.nlev; ++l) {
        const double bm = a.bkm[l];
        if (bm == 0.0) continue;                 // pressure independent of ps
        const double am = a.akm[l];
        const float p_s = (float)fma(ps_s, bm, am);
        const float p_n = (float)fma(ps_n, bm, am);
        const long long off = (long long)l * n + c;
        const float q = a.QV_out[off];
        const float e = __fdividef(q * p_s, 0.622f + 0.378f * q);
        a.QV_out[off] = __fdividef(0.622f * e, p_n - 0.378f * e);
    }
}

// Latitude-band mode: the status block as float64 words that an element-wise MAX over the bands merges
// (max error per iteration as is; minima negated; one word per error bit), and back.
__global__ void pgw_band_pack_kernel(const pgw_timestep_status *s, double *w) {
    const int i = threadIdx.x;
    if (i < PGW_MAX_ITER) w[i] = __longlong_as_double((long long)s->maxerr[i]);
    else if (i < PGW_MAX_ITER + 2) w[i] = -(double)s->stats[i - PGW_MAX_ITER];
    else if (i < PGW_MAX_ITER + 34) w[i] = (double)((s->err >> (i - PGW_MAX_ITER - 2)) & 1u);
    else if (i < PGW_BAND_WORDS) w[i] = -(double)s->first_k[i - PGW_MAX_ITER - 34];
}
__global__ void pgw_band_unpack_kernel(const double *w, pgw_timestep_status *s) {
    const int i = threadIdx.x;
    if (i < PGW_MAX_ITER) s->maxerr[i] = (uint64_t)__double_as_longlong(w[i]);
    else if (i < PGW_MAX_ITER + 2) s->stats[i - PGW_MAX_ITER] = (float)(-w[i]);
    else if (i == PGW_MAX_ITER + 2) {
        uint32_t e = 0;
        for (int b = 0; b < 32; ++b) if (w[PGW_MAX_ITER + 2 + b] != 0.0) e |= 1u << b;
        s->err = e;
    } else if (i >= PGW_MAX_ITER + 34 && i < PGW_BAND_WORDS) s->first_k[i - PGW_MAX_ITER - 34] = (int32_t)(-w[i]);
}

// Latitude-band exchange fused into the step: pack, store into every peer's inbox over NVLink, release a flag,
// wait for all peers' flags, merge (MAX), unpack.  One CTA of 128 threads; see pgw_band_exchange in the header.
__device__ __forceinline__ void st_sys_f64(double *p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys_f64(double *p, double v) {
    asm volatile("st.release.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ double ld_acquire_sys_f64(const double *p) {
    double v;
    asm volatile("ld.acquire.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_sys_f64(const double *p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(128)
pgw_band_exchange_kernel(pgw_timestep_status *s, double *const *inbox, int rank, int world, unsigned long long seq,
                         long long timeout_ns) {
    __shared__ double merged[PGW_BAND_WORDS];
    __shared__ int timed_out;
    const int i = threadIdx.x;
    const size_t par = (size_t)(seq % PGW_BAND_PARITIES);
    const double tag = (double)seq;
    if (i == 0) timed_out = 0;
    // ---- pack (same words as pgw_band_pack_kernel)
    double w = 0.0;
    if (i < PGW_MAX_ITER) w = __longlong_as_double((long long)s->maxerr[i]);
    else if (i < PGW_MAX_ITER + 2) w = -(double)s->stats[i - PGW_MAX_ITER];
    else if (i < PGW_MAX_ITER + 34) w = (double)((s->err >> (i - PGW_MAX_ITER - 2)) & 1u);
    else if (i < PGW_BAND_WORDS) w = -(double)s->first_k[i - PGW_MAX_ITER - 34];
    // ---- push this band's block into slot [par][rank] of every inbox (its own included)
    const size_t slot = (par * (size_t)world + (size_t)rank) * PGW_BAND_SLOT;
    if (i < PGW_BAND_WORDS)
        for (int r = 0; r < world; ++r) st_sys_f64(inbox[r] + slot + i, w);
    __threadfence_system();
    __syncthreads();
    if (i < world) st_release_sys_f64(inbox[i] + slot + PGW_BAND_WORDS, tag);     // thread i publishes to peer i
    // ---- wait for the blocks of all bands in the own inbox
    const double *mine = inbox[rank] + par * (size_t)world * PGW_BAND_SLOT;
    if (i < world) {
        long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        while (ld_acquire_sys_f64(mine + (size_t)i * PGW_BAND_SLOT + PGW_BAND_WORDS) != tag) {
            long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > timeout_ns) { timed_out = 1; break; }
            __nanosleep(200);
        }
    }
    __syncthreads();
    if (timed_out) {
        if (i == 0) atomicOr(&s->err, PGW_ERR_BAND_TIMEOUT);
        return;
    }
    // ---- merge (element-wise MAX over the bands) and unpack
    if (i < PGW_BAND_WORDS) {
        double m = ld_sys_f64(mine + i);
        for (int r = 1; r < world; ++r) m = fmax(m, ld_sys_f64(mine + (size_t)r * PGW_BAND_SLOT + i));
        merged[i] = m;
    }
    __syncthreads();
    if (i < PGW_MAX_ITER) s->maxerr[i] = (uint64_t)__double_as_longlong(merged[i]);
    else if (i < PGW_MAX_ITER + 2) s->stats[i - PGW_MAX_ITER] = (float)(-merged[i]);
    else if (i == PGW_MAX_ITER + 2) {
        uint32_t e = 0;
        for (int b = 0; b < 32; ++b) if (merged[PGW_MAX_ITER + 2 + b] != 0.0) e |= 1u << b;
        s->err = e;
    } else if (i >= PGW_MAX_ITER + 34 && i < PGW_BAND_WORDS) s->first_k[i - PGW_MAX_ITER - 34] = (int32_t)(-merged[i]);
}

}  // namespace pgw

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
namespace {

using pgw::kColumnThreads;

// First (topmost) full level whose layer can reach p_ref for any ps <= ps_bound:
// the layer above the first half level with ak + ps_bound*bk >= p_ref.
int stash_top(const double *ak, const double *bk, int nlev, double p_ref, double ps_bound) {
    int h = nlev;
    for (int i = 0; i <= nlev; ++i)
        if (ak[i] + ps_bound * bk[i] >= p_ref) { h = i; break; }
    int lst = h - 1;
    if (lst < 0) lst = 0;
    if (lst > nlev - 1) lst = nlev - 1;
    return lst;
}

size_t column_smem(int nlev, int nplev, int np, int nt, bool ref) {
    return sizeof(double) * 2 * (size_t)(nlev + 1) +                       // (ak, bk)
           (size_t)np * nt * (2 * sizeof(float)) +                         // (T_pgw, e_pgw) stash
           sizeof(float) * (size_t)(pgw::kRing + 1) * 4 * nt +             // cp.async ring
           sizeof(float) * 2 * (size_t)nlev + sizeof(float) * 3 * (size_t)nplev + 16 +
           (ref ? (size_t)np * nt * sizeof(float) : 0);                    // residual of the fp32 T_pgw
}

// PGW_FLAG_LOCAL_PREF: zg levels, candidates, the per-candidate ERA sums and the slot table (+ alignment)
size_t local_pref_smem(int nzg, int ncand, int nt) {
    return 16 + sizeof(double) * (size_t)(nzg + ncand) + 16 + 2 * sizeof(double) * (size_t)ncand * nt +
           sizeof(int) * (size_t)nzg;
}

int validate(const pgw_timestep_args *a) {
    if (!a) return PGW_E_INVALID;
    if (a->ncol <= 0 || a->nlev < 2 || a->nplev < 2 || a->nplev > 64) return PGW_E_INVALID;
    // 32-bit element offsets inside the kernels (the packed deltas hold 4 floats per node and column)
    if ((unsigned long long)a->ncol * (unsigned long long)(a->nlev + 1) >= (1ull << 30)) return PGW_E_INVALID;
    if ((unsigned long long)a->ncol * (unsigned long long)a->nplev >= (1ull << 29)) return PGW_E_INVALID;
    if (a->nsoil < 0 || a->nsoil > PGW_MAX_SOIL) return PGW_E_INVALID;
    if (a->k_spec < 1 || a->k_spec > PGW_MAX_ITER) return PGW_E_INVALID;
    const void *need[] = {a->ak_host, a->bk_host, a->ak, a->bk, a->akm, a->bkm, a->plev, a->PS, a->FIS, a->FR_LAND, a->FR_SEA_ICE,
                          a->T_SKIN, a->T, a->QV, a->U, a->V, a->d4.lo, a->d4.hi, a->tas.lo, a->tas.hi, a->hurs.lo,
                          a->hurs.hi, a->ps_hist.lo, a->ps_hist.hi, a->ts.lo, a->ts.hi, a->tos.lo, a->tos.hi,
                          a->siconc.lo, a->siconc.hi, a->zg_ref.lo, a->zg_ref.hi, a->ts_clim, a->PS_out,
                          a->T_SKIN_out, a->FR_SEA_ICE_out, a->T_out, a->QV_out, a->U_out, a->V_out,
                          a->dps_out, a->dps_traj, a->maxerr, a->stats, a->err};
    for (const void *p : need) if (!p) return PGW_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(a->d4.lo) | reinterpret_cast<uintptr_t>(a->d4.hi)) & 15u) return PGW_E_INVALID;
    if (a->nsoil > 0 && (!a->T_SO || !a->T_SO_out)) return PGW_E_INVALID;
    if ((a->flags & PGW_FLAG_REINTERP) && (a->flags & (PGW_FLAG_LOCAL_PREF | PGW_FLAG_REF_DTYPES))) return PGW_E_INVALID;
    if (a->flags & PGW_FLAG_LOCAL_PREF) {
        if (a->flags & PGW_FLAG_REF_DTYPES) return PGW_E_INVALID;
        if (a->nzg < 1 || a->nzg > 64 || !(a->p_floor > 0.0)) return PGW_E_INVALID;
        if ((unsigned long long)a->ncol * (unsigned long long)a->nzg >= (1ull << 31)) return PGW_E_INVALID;
        if (!a->zg.lo || !a->zg.hi || !a->zg_plev || !a->zg_plev_host || !a->pref_traj || !a->p_ref_out)
            return PGW_E_INVALID;
    }
    return PGW_OK;
}

// PGW_COLUMN_PATH=generic forces the cp.async flavour (the parity tests run both)
bool tma_allowed() {
    const char *e = getenv("PGW_COLUMN_PATH");
    return !(e && strcmp(e, "generic") == 0);
}

pgw_column_plan plan_column(const pgw_timestep_args *a) {
    pgw_column_plan p;
    p.local = (a->flags & PGW_FLAG_LOCAL_PREF) != 0;
    // with a per-column p_ref the stash reaches up to the lowest p_ref it is sized for
    const double p_stash = p.local ? a->p_floor : a->p_ref;
    p.lst = stash_top(a->ak_host, a->bk_host, a->nlev, p_stash, a->ps_bound);
    p.np = a->nlev - p.lst;
    p.ref = (a->flags & PGW_FLAG_REF_DTYPES) != 0;
    p.reinterp = (a->flags & PGW_FLAG_REINTERP) != 0;
    p.smem = column_smem(a->nlev, a->nplev, p.np, kColumnThreads, p.ref);
    p.ncand = 0;
    if (p.local) {
        for (int i = 0; i < a->nzg; ++i) p.ncand += a->zg_plev_host[i] >= a->p_floor;
        p.smem += local_pref_smem(a->nzg, p.ncand, kColumnThreads);
    }
    p.tma = false;
    int lst_tma = 0;
    size_t smem_tma = 0;
    // the TMA flavour handles a scalar p_ref only, and parks (T_pgw, e_pgw) that do not change over the iteration
    if (tma_allowed() &&
        !(a->flags & (PGW_FLAG_DIRECT | PGW_FLAG_REF_DTYPES | PGW_FLAG_LOCAL_PREF | PGW_FLAG_REINTERP)) &&
        pgw_tma_eligible(a, p.lst, &lst_tma, &smem_tma)) {
        p.tma = true;
        p.lst = lst_tma;
        p.np = a->nlev - lst_tma;
        p.smem = smem_tma;
    }
    // FAST: every layer the iteration can touch has s = (pb-pt)/(pb+pt) < 0.06 for all ps in
    // [p_ref, ps_bound] (s is monotone in ps), so the series needs no exact-log fallback.
    p.fast = true;
    for (int l = p.lst; l < a->nlev; ++l)
        for (double ps : {p_stash, a->ps_bound}) {
            const double pt = a->ak_host[l] + ps * a->bk_host[l], pb = a->ak_host[l + 1] + ps * a->bk_host[l + 1];
            if (!(pt > 0.0) || !((pb - pt) / (pb + pt) < 0.055)) p.fast = false;
        }
    return p;
}

// PGW_FLAG_REINTERP: the column kernel, or (replay != null) its replay for iteration N
int launch_reinterp(const pgw_timestep_args *a, const pgw_column_plan &plan, const pgw_timestep_result *replay,
                    cudaStream_t st) {
    auto kern = plan.fast ? pgw::pgw_column_kernel<kColumnThreads, true, false, false, true>
                          : pgw::pgw_column_kernel<kColumnThreads, false, false, false, true>;
    int rc = pgw_ensure_smem((const void *)kern, plan.fast ? 11 : 10, plan.smem, plan.np);
    if (rc != PGW_OK) return rc;
    const unsigned grid = (unsigned)((a->ncol + kColumnThreads - 1) / kColumnThreads);
    kern<<<grid, kColumnThreads, plan.smem, st>>>(*a, plan.lst, plan.np, plan.ncand, replay);
    return pgw_check_launch("pgw_column_kernel");
}

}  // namespace

extern "C" {

long long pgw_timestep_smem_bytes(const pgw_timestep_args *a) {
    int rc = validate(a);
    if (rc != PGW_OK) return rc;
    return (long long)plan_column(a).smem;
}

int pgw_timestep_uses_tma(const pgw_timestep_args *a) {
    int rc = validate(a);
    if (rc != PGW_OK) return rc;
    return plan_column(a).tma ? 1 : 0;
}

int pgw_timestep_plan_info(const pgw_timestep_args *a, int info[6]) {
    int rc = validate(a);
    if (rc != PGW_OK || !info) return PGW_E_INVALID;
    const pgw_column_plan p = plan_column(a);
    info[0] = p.tma ? 1 : 0;
    info[1] = p.fast && !p.ref ? 1 : 0;           // PGW_FLAG_REF_DTYPES has one instance, the exact-log one
    info[2] = p.lst;
    info[3] = p.np;
    info[4] = p.tma ? pgw_tma_tmem_cols(p.np) : 0;
    info[5] = p.tma && pgw_tma_l137(a, p) ? 1 : 0;
    return PGW_OK;
}

int pgw_timestep(const pgw_timestep_args *a, void *stream) {
    int rc = validate(a);
    if (rc != PGW_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const pgw_column_plan plan = plan_column(a);
    pgw::pgw_timestep_init_kernel<<<1, 64, 0, st>>>(a->maxerr, a->stats, a->err, a->first_k, a->poly_fallback);
    if (plan.tma) return pgw_launch_column_tma(a, plan, st);

    if (plan.reinterp) return launch_reinterp(a, plan, nullptr, st);
    const int variant = plan.local ? (plan.fast ? 9 : 8) : plan.ref ? 2 : (plan.fast ? 1 : 0);
    auto kern = plan.local ? (plan.fast ? pgw::pgw_column_kernel<kColumnThreads, true, false, true>
                                        : pgw::pgw_column_kernel<kColumnThreads, false, false, true>)
              : plan.ref   ? pgw::pgw_column_kernel<kColumnThreads, false, true>
                           : (plan.fast ? pgw::pgw_column_kernel<kColumnThreads, true, false>
                                        : pgw::pgw_column_kernel<kColumnThreads, false, false>);
    if ((rc = pgw_ensure_smem((const void *)kern, variant, plan.smem, plan.np)) != PGW_OK) return rc;
    const unsigned grid = (unsigned)((a->ncol + kColumnThreads - 1) / kColumnThreads);
    kern<<<grid, kColumnThreads, plan.smem, st>>>(*a, plan.lst, plan.np, plan.ncand, nullptr);
    return pgw_check_launch("pgw_column_kernel");
}

int pgw_timestep_finalize(const pgw_timestep_args *a, pgw_timestep_result *result_dev, void *stream) {
    int rc = validate(a);
    if (rc != PGW_OK || !result_dev) return PGW_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    pgw::pgw_converge_kernel<<<1, 1, 0, st>>>(a->maxerr, a->k_spec, a->thresh_phi_ref_max_error, result_dev);
    // PGW_FLAG_REINTERP: the speculative QV does not give e_pgw of iteration N back (T and RELHUM move with the
    // pressures), so the column kernel itself runs again for k_spec = N when the result was rewritten
    if (a->flags & PGW_FLAG_REINTERP) {
        if ((rc = launch_reinterp(a, plan_column(a), result_dev, st)) != PGW_OK) return rc;
        return pgw_check_launch("pgw_timestep_finalize");
    }
    const unsigned grid = (unsigned)((a->ncol + 255) / 256);
    pgw::pgw_rewrite_kernel<<<grid, 256, 0, st>>>(*a, result_dev);
    return pgw_check_launch("pgw_timestep_finalize");
}

long long pgw_sizeof_timestep_status(void) { return (long long)sizeof(pgw_timestep_status); }

static bool status_matches(const pgw_timestep_args *a, pgw_timestep_status *s) {
    return s && a->maxerr == s->maxerr && a->stats == s->stats && a->err == &s->err && a->first_k == s->first_k &&
           a->poly_fallback == &s->poly_fallback;
}

int pgw_timestep_finish(const pgw_timestep_args *a, pgw_timestep_status *status_dev,
                        pgw_timestep_status *status_host, void *stream) {
    if (!a || !status_matches(a, status_dev)) return PGW_E_INVALID;
    int rc = pgw_timestep_finalize(a, &status_dev->result, stream);
    if (rc != PGW_OK) return rc;
    if (status_host &&
        cudaMemcpyAsync(status_host, status_dev, sizeof(pgw_timestep_status), cudaMemcpyDeviceToHost,
                        (cudaStream_t)stream) != cudaSuccess)
        return pgw_check_launch("cudaMemcpyAsync(status)");
    return PGW_OK;
}

int pgw_timestep_run(const pgw_timestep_args *a, pgw_timestep_status *status_dev,
                     pgw_timestep_status *status_host, int run_flags, void *stream) {
    if (!a || !status_matches(a, status_dev)) return PGW_E_INVALID;
    int rc = pgw_timestep(a, stream);
    if (rc != PGW_OK || (run_flags & PGW_RUN_NO_FINALIZE)) return rc;
    return pgw_timestep_finish(a, status_dev, status_host, stream);
}

int pgw_band_pack(const pgw_timestep_status *status_dev, double *words_dev, void *stream) {
    if (!status_dev || !words_dev) return PGW_E_INVALID;
    pgw::pgw_band_pack_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(status_dev, words_dev);
    return pgw_check_launch("pgw_band_pack");
}

int pgw_band_exchange(pgw_timestep_status *status_dev, double *const *inbox_ptrs_dev, int rank, int world,
                      unsigned long long seq, double timeout_s, void *stream) {
    if (!status_dev || !inbox_ptrs_dev || world < 1 || world > 128 || rank < 0 || rank >= world || seq == 0 ||
        !(timeout_s > 0.0))
        return PGW_E_INVALID;
    pgw::pgw_band_exchange_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(status_dev, inbox_ptrs_dev, rank, world, seq,
                                                                        (long long)(timeout_s * 1e9));
    return pgw_check_launch("pgw_band_exchange");
}

int pgw_band_unpack(const double *words_dev, pgw_timestep_status *status_dev, void *stream) {
    if (!status_dev || !words_dev) return PGW_E_INVALID;
    pgw::pgw_band_unpack_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(words_dev, status_dev);
    return pgw_check_launch("pgw_band_unpack");
}

}  // extern "C"
