// The TMA flavour of the fused per-timestep column kernel of libpgw_b200 (sm_100a).
//
// Same algorithm and reference semantics as pgw_timestep.cu (see the header comment there):
// one thread owns one ERA5 column, the column is swept bottom-up, the levels below p_ref are
// parked for the surface-pressure fixed point, the rest is streamed with the adjusted surface
// pressure already known.  What differs is how the 3-D fields move and where the parked levels live:
//
//  * the CTA is two warpgroups.  The first (producer) gives its registers to the second with
//    setmaxnreg (64 at launch -> 24 / 104), so 4 CTAs = 16 column warps fit on an SM, and one
//    elected thread of it streams level PAIRS of the CTA's 128 columns through a ring of
//    shared-memory slots [T,QV,U,V][2 levels][128] with cp.async.bulk.tensor (TMA, box 2 x 128 of a
//    [nlev, ncol] tensor map per field);
//  * the second warpgroup holds the four column warps; column thread i parks (T_pgw, e_pgw) of its
//    levels in TENSOR MEMORY lane i (tcgen05.st / tcgen05.ld), which leaves shared memory to the ring
//    and the tables;
//  * the four column warps wait on full[slot], read their column from the slot, compute, write
//    the results back IN PLACE, fence them for the async proxy and arrive on done[slot];
//  * the producer then stores the slot with TMA (bulk group), and, once the previous slot's
//    store has left shared memory, refills that slot with the pair kTmaSlots ahead.  Pairs
//    further ahead are pulled into L2 with cp.async.bulk.prefetch.tensor.
//
// Per-thread global accesses are left only for the 2-D fields, the delta nodes and QV of the
// parked levels.  The column threads run two loops over the 69 level pairs -- parked pairs, then the
// fixed point, then streamed pairs -- generated from one body with a compile-time phase tag (a single
// loop with run-time phase tests executes 12 % more instructions), and ONE delta walker serves all four
// variables: the packed float4 deltas (ta, hur, ua, va) share their pressure nodes, and the surface node
// that replace_delta_sfc (functions.py:343-366) inserts into the ta/hur columns only matters below the
// node under ps_hist, where it is applied as an override.  The hot code stays small (an early version
// with two walkers was instruction-cache bound; unrolling the loops costs more than it saves).
// Per pair, the barrier probe is issued first, the two walks (which need no slot data) hide its round
// trip; the walker's loads are issued once per pair iteration, a whole iteration before their first use.
//
// The fixed point does not re-integrate the parked levels in every iteration: their geopotential sum is
// expanded once, during the sweep, as a polynomial in dps (see "the geopotential sums of the parked
// levels" below); only the three layers around p_ref are integrated per iteration, and a warp whose
// dps leaves the range of the polynomial falls back to the full integration for that iteration.
//
// Needs ncol % 4 == 0 (16-byte global strides), 16-byte aligned fields and nlev <= kTmaMaxLev;
// anything else takes the cp.async flavour.
#include "pgw_column.cuh"

#include <stdlib.h>
#include <string.h>

namespace pgw {

// PGW_X2: the arithmetic both levels of a pair share is issued as packed float32 pair instructions (FADD2 / FMUL2 /
// FFMA2 of sm_100): same operations per lane, ~8 % fewer instructions in the sweep loops, 1.295 -> 1.271 ms.
#ifndef PGW_X2
#define PGW_X2 1
#endif
// PGW_UNIFORM_TOP: levels whose full-level pressure does not depend on ps (bkm == 0: the pure pressure levels at
// the top of the model) have a column-independent walker position and interpolation weight; they are tabulated once
// per CTA (with the very instructions the per-column walk uses, hence bit-identical) and the streamed pairs made of
// such levels skip the lg2, the weight multiply, the step tests and the exact-hit selects.
#ifndef PGW_UNIFORM_TOP
#define PGW_UNIFORM_TOP 0
#endif
#ifndef PGW_TMA_SLOTS
#define PGW_TMA_SLOTS 4
#endif
constexpr int kTmaSlots = PGW_TMA_SLOTS;   // ring of level pairs, 4 KB each
#ifndef PGW_TMA_L2_AHEAD
#define PGW_TMA_L2_AHEAD 0
#endif
constexpr int kTmaL2Ahead = PGW_TMA_L2_AHEAD;   // level pairs prefetched into L2 beyond the ones in the ring
#ifndef PGW_TMA_UNROLL_PARKED
#define PGW_TMA_UNROLL_PARKED 1
#endif
#ifndef PGW_TMA_UNROLL_STREAMED
#define PGW_TMA_UNROLL_STREAMED 1
#endif
// unrolling either sweep loop costs more in instruction-cache misses than it saves (streamed x2: +4 %, x4: +13 %)
constexpr int kUnrollParked = PGW_TMA_UNROLL_PARKED, kUnrollStreamed = PGW_TMA_UNROLL_STREAMED;
constexpr double kTaylorMaxRel = 0.012;    // |ps_pgw - ps_era| / ps_era up to which the polynomial of the fixed point is used
constexpr int kTmaMaxLev = 160;      // capacity of the parameter-space table of the upper levels

// tiled tensor maps [nlev, ncol] (box 2 x 128) of the four 3-D inputs and outputs, and (akm, bkm)
// as float2 for the levels above the stash, read through the constant bank
struct TmaParams {
    CUtensorMap in[4];      // T, QV, U, V
    CUtensorMap out[4];     // T_out, QV_out, U_out, V_out
    float2 m[kTmaMaxLev];
};

struct F4 { float x, y, z, w; };
struct TagParked { static constexpr bool value = true; };
struct TagStreamed { static constexpr bool value = false; };
__device__ __forceinline__ F4 ldg4(const float4 *p) { const float4 v = __ldg(p); return F4{v.x, v.y, v.z, v.w}; }

// NLEV_C / NP_C: number of levels and of parked levels as compile-time constants (0 = taken from the
// arguments).  The loop bounds of the sweep are then immediates; with run-time bounds every pair iteration
// waits on a constant-bank load before it can resolve its branches.  The host picks the instance that
// matches (137 levels with 56 parked ones: ERA5 L137, p_ref = 300 hPa) or the generic one.
//
// Tensor memory: `ncols` columns (host: next power of two >= max(32, 2 np)); parked level l sits in columns
// 2 (L-1-l) (T_pgw) and 2 (L-1-l) + 1 (e_pgw), so a parked level pair is one 4-column store.
template <bool FAST, int NLEV_C, int NP_C>
__global__ void __launch_bounds__(2 * kColumnThreads, 4)
pgw_column_tma_kernel(const __grid_constant__ pgw_timestep_args a, const __grid_constant__ TmaParams tp,
                      const int lst_arg, const int np_arg, const uint32_t ncols) {
    constexpr int NT = kColumnThreads, NTHR = 2 * kColumnThreads;
    extern __shared__ __align__(1024) unsigned char smem[];
    const int L = NLEV_C ? NLEV_C : a.nlev, K = a.nplev;
    const int np = NP_C ? NP_C : np_arg;
    const int lst = NLEV_C ? NLEV_C - NP_C : lst_arg;
    // ---- shared memory: pair ring | (ak,bk)[np+1] | (akm,bkm)[np] | plev tables | barriers | TMEM address
    float *const ring = reinterpret_cast<float *>(smem);                          // [kTmaSlots][4][2][NT]
    double2 *const hl0 = reinterpret_cast<double2 *>(ring + kTmaSlots * 8 * NT);
    float2 *const m0p = reinterpret_cast<float2 *>(hl0 + (np + 1));
    float *const s_plev = reinterpret_cast<float *>(m0p + np);                     // [K] ascending
    float *const s_inv_plev = s_plev + K;                                          // [K]
    float *const s_inv_w = s_inv_plev + K;                                         // [K] 1/log2(p[j+1]/p[j])
#if PGW_UNIFORM_TOP
    const int K3 = 3 * K + ((3 * K) & 1), Lp = L + (L & 1);
    float *const s_ut = s_plev + K3;                                               // [L] weight of a uniform level
    int *const s_un = reinterpret_cast<int *>(s_ut + Lp);                          // [L] its node (lo) index
    uint64_t *const bar_full = reinterpret_cast<uint64_t *>(s_un + Lp);
#else
    uint64_t *const bar_full = reinterpret_cast<uint64_t *>(s_plev + 3 * K + ((3 * K) & 1));
#endif
    uint64_t *const bar_done = bar_full + kTmaSlots;
    uint32_t *const s_tmem = reinterpret_cast<uint32_t *>(bar_done + kTmaSlots);
    int *const s_lstar = reinterpret_cast<int *>(s_tmem + 1);                     // [NT]
    const double2 *const s_hl = hl0 - lst;      // indexed by the half level, l >= lst
    const float2 *const s_m = m0p - lst;        // indexed by the full level, l >= lst

    const int tid = threadIdx.x;
    for (int i = tid; i <= np; i += NTHR) hl0[i] = make_double2(a.ak[lst + i], a.bk[lst + i]);
    for (int i = tid; i < np; i += NTHR) m0p[i] = make_float2((float)a.akm[lst + i], (float)a.bkm[lst + i]);
    for (int i = tid; i < K; i += NTHR) {
        const int f0 = a.plev_descending ? (K - 1 - i) : i;
        const float p0 = (float)a.plev[f0];
        s_plev[i] = p0;
        s_inv_plev[i] = 1.0f / p0;
        if (i + 1 < K) {
            const float p1 = (float)a.plev[a.plev_descending ? (K - 2 - i) : (i + 1)];
            s_inv_w[i] = 1.0f / log2f(p1 / p0);
        } else s_inv_w[i] = 0.0f;
    }
    if (tid == 0) {
        for (int i = 0; i < kTmaSlots; ++i) { mbar_init(bar_full + i, 1); mbar_init(bar_done + i, NT); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if ((tid >> 5) == NT / 32) tmem_alloc(s_tmem, ncols);        // the first column warp
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
#if PGW_UNIFORM_TOP
    // walker position and weight of the levels whose pressure is akm alone, by the instructions of walk()
    for (int l = tid; l < L; l += NTHR) {
        const float2 m = tp.m[l];
        int nd = -1;
        for (int k = K - 1; k >= 0; --k)
            if (s_plev[k] <= m.x) { nd = k; break; }
        s_un[l] = nd;
        s_ut[l] = nd >= 0 ? fast_lg2(m.x * s_inv_plev[nd]) * s_inv_w[nd] : 0.0f;
    }
    __syncthreads();
#endif

    const uint32_t n = (uint32_t)a.ncol;
    const int npairs = (L + 1) >> 1, np1 = np >> 1;     // level pairs in total / parked (np is even)

    // ------------------------------------------------------------------ producer warpgroup
    if (tid < NT) {
        regs_dec<24>();                                     // all four warps, before any of them exits
        if (tid != 0) return;
        const int c0 = (int)(blockIdx.x * NT);
        // pair j = levels L-1-2j (row 1) and L-2-2j (row 0).  TMA coordinates must not be negative,
        // so the last pair of an odd column is levels (1, 0): level 1 is simply done twice.
        auto pair_row = [&](int j) { const int r = L - 2 - 2 * j; return r < 0 ? 0 : r; };
        auto load_pair_slot = [&](int j) {
            const int s = j % kTmaSlots;
            float *dst = ring + s * 8 * NT;
            mbar_arrive_expect_tx(bar_full + s, 4u * 2u * NT * sizeof(float));
#pragma unroll
            for (int v = 0; v < 4; ++v) tma_load_2d(dst + v * 2 * NT, &tp.in[v], c0, pair_row(j), bar_full + s);
        };
        auto l2_pair = [&](int j) {
            if (j < npairs) {
#pragma unroll
                for (int v = 0; v < 4; ++v) tma_prefetch_2d(&tp.in[v], c0, pair_row(j));
            }
        };
        for (int j = 0; j < kTmaSlots && j < npairs; ++j) load_pair_slot(j);
        for (int j = kTmaSlots; j < kTmaSlots + kTmaL2Ahead; ++j) l2_pair(j);
#pragma unroll 1
        for (int j = 0; j < npairs; ++j) {
            const int s = j % kTmaSlots;
            const float *src = ring + s * 8 * NT;
            mbar_wait_backoff(bar_done + s, (j / kTmaSlots) & 1);
            const int row = pair_row(j);
            tma_store_2d(&tp.out[0], c0, row, src);
            if (j >= np1) tma_store_2d(&tp.out[1], c0, row, src + 2 * NT);   // QV of the parked levels: phase 3
            tma_store_2d(&tp.out[2], c0, row, src + 4 * NT);
            tma_store_2d(&tp.out[3], c0, row, src + 6 * NT);
            tma_commit();
            tma_wait_read<1>();                     // the stores of pair j-1 have left shared memory
            if (j >= 1 && j - 1 + kTmaSlots < npairs) load_pair_slot(j - 1 + kTmaSlots);
            l2_pair(j + kTmaSlots + kTmaL2Ahead);
        }
        tma_wait_all();
        return;
    }

    // ------------------------------------------------------------------ column threads
    regs_inc<104>();
    const int ct = tid - NT;                                // column of the CTA = TMEM lane
    const uint32_t tm = *s_tmem + ((uint32_t)(ct & ~31) << 16);   // column 0 of this warp's 32 lanes
    const uint32_t c_raw = blockIdx.x * NT + ct;
    // Threads past the last column read column n-1 for the 2-D fields; their slot columns are
    // zero-filled by TMA and clipped on store, and their per-thread stores are masked.
    const uint32_t c = (c_raw >= n) ? n - 1 : c_raw;
    const bool valid = c_raw < n;
    unsigned errbits = 0;
    int k_pref = INT32_MAX, k_bound = INT32_MAX;     // first iteration in which the two ps-dependent checks fired

    // ---------------- surface, skin and soil (step_03:103-146) ----------------
    const float ps_f = __ldg(a.PS + c);
    const Pair2 r_sic = load_pair(a.siconc, c), r_ts = load_pair(a.ts, c), r_tos = load_pair(a.tos, c);
    const Pair2 r_psh = load_pair(a.ps_hist, c), r_tas = load_pair(a.tas, c), r_hurs = load_pair(a.hurs, c);
    const Pair2 r_zg = load_pair(a.zg_ref, c);
    const float r_ice = __ldg(a.FR_SEA_ICE + c), r_land = __ldg(a.FR_LAND + c), r_skin = __ldg(a.T_SKIN + c);
    const float r_clim = __ldg(a.ts_clim + c), r_fis = __ldg(a.FIS + c);
    const double PSd = (double)ps_f;

    // ---------------- the delta walker (functions.py:343-431, 511-580) ----------------
    // Downward merge walk over the pressure-ascending nodes: state = lo node (index, pressure,
    // values of the four variables) and the differences to the hi node; inv_w == 0 encodes
    // "no interpolation" (at/after the last node, or above node 0): the lo values are returned.
    // Node lo-1 is kept blended, node lo-2 as raw (before, after) time slabs that are blended one step after their loads;
    // nodes further down are pulled into L2.
    const float w_t = slab_weight(a.d4);
    const float4 *const d4lo = reinterpret_cast<const float4 *>(a.d4.lo);
    const float4 *const d4hi = reinterpret_cast<const float4 *>(a.d4.hi);
    const int desc = a.plev_descending;
    auto node_off = [&](int j) { return (uint32_t)(desc ? (K - 1 - j) : j) * n + c; };
    auto blend4 = [&](const F4 &x0, const F4 &x1) {
        return F4{blend_f32(w_t, x0.x, x1.x), blend_f32(w_t, x0.y, x1.y), blend_f32(w_t, x0.z, x1.z),
                  blend_f32(w_t, x0.w, x1.w)};
    };
    auto l2_node = [&](int j) {
        const uint32_t off = node_off(j);
        asm volatile("prefetch.global.L2 [%0];" ::"l"(d4lo + off));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(d4hi + off));
    };

    const float2 m_bot = s_m[L - 1];
    const float p_bot = fmaf(ps_f, m_bot.y, m_bot.x);           // the first level of the sweep
    int w_lo = -1;                                              // max{k: plev[k] <= p_bot}
    for (int k = K - 1; k >= 0; --k)
        if (s_plev[k] <= p_bot) { w_lo = k; break; }
    // replace_delta_sfc: node s of the ta/hur columns carries (ps_hist, surface delta) and all
    // nodes after it hold the surface delta.  s = max{k: plev[k] < ps_hist}.
    const float psh = (float)blend_f64(a.ps_hist, r_psh);
    int s_node = K - 1;
    if (!(psh > s_plev[K - 1])) {
        s_node = -1;
        for (int k = K - 1; k >= 0; --k)
            if (s_plev[k] < psh) { s_node = k; break; }
    }
    if (s_node < 0) { errbits |= PGW_ERR_PS_HIST_RANGE; s_node = 0; }
    const float min_src_p0 = (s_node == 0) ? psh : s_plev[0];

    // raw nodes: hi = w_lo+1, lo = w_lo, then the two prefetched ones, and node s-1 for the override
    const int j_lo = w_lo < 0 ? 0 : w_lo, j_hi = (w_lo >= 0 && w_lo + 1 < K) ? w_lo + 1 : j_lo;
    const F4 rl0 = ldg4(d4lo + node_off(j_lo)), rl1 = ldg4(d4hi + node_off(j_lo));
    const F4 rh0 = ldg4(d4lo + node_off(j_hi)), rh1 = ldg4(d4hi + node_off(j_hi));
    const int j_s1 = s_node >= 1 ? s_node - 1 : 0;
    const F4 rs0 = ldg4(d4lo + node_off(j_s1)), rs1 = ldg4(d4hi + node_off(j_s1));
    // node lo-1 (raw here, kept blended in the walker state) and the raw slabs of node lo-2
    F4 n0{0.f, 0.f, 0.f, 0.f}, n1 = n0, m0 = n0, m1 = n0;
    if (w_lo >= 1) { n0 = ldg4(d4lo + node_off(w_lo - 1)); n1 = ldg4(d4hi + node_off(w_lo - 1)); }
    if (w_lo >= 2) { m0 = ldg4(d4lo + node_off(w_lo - 2)); m1 = ldg4(d4hi + node_off(w_lo - 2)); }
#pragma unroll
    for (int d = 3; d <= kL2Ahead; ++d)
        if (w_lo - d >= 0) l2_node(w_lo - d);

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
        if (valid) {
            a.FR_SEA_ICE_out[c] = sic;
            a.T_SKIN_out[c] = (float)((double)r_skin + comb);
        }
        for (int s = 0; s < a.nsoil; ++s) {
            const double dso = clim + a.soil_decay[s] * (comb - clim);
            const float so = (float)((double)__ldg(a.T_SO + (uint32_t)s * n + c) + dso);
            if (valid) a.T_SO_out[(uint32_t)s * n + c] = so;
        }
    }

    // walker state
    float w_p_lo, w_inv_p_lo, w_inv_w;
    F4 x_lo = blend4(rl0, rl1), x_d{0.f, 0.f, 0.f, 0.f};
    F4 nb = blend4(n0, n1);                                     // node lo-1, blended
    if (w_lo >= 0) {
        w_p_lo = s_plev[w_lo]; w_inv_p_lo = s_inv_plev[w_lo]; w_inv_w = s_inv_w[w_lo];   // inv_w[K-1] == 0
        if (w_lo + 1 < K) {
            const F4 x_hi = blend4(rh0, rh1);
            x_d = F4{x_hi.x - x_lo.x, x_hi.y - x_lo.y, x_hi.z - x_lo.z, x_hi.w - x_lo.w};
        }
    } else {
        w_p_lo = 0.0f; w_inv_p_lo = 1.0f; w_inv_w = 0.0f;       // whole column above node 0
    }
    // Override for ta, hur while p > plev[s-1]: the surface delta for p >= ps_hist, else the segment
    // between node s-1 and the (ps_hist, surface delta) node.  s == 0: the surface delta everywhere.
    const float sfc_ta = (float)blend_f64(a.tas, r_tas), sfc_hur = (float)blend_f64(a.hurs, r_hurs);
    bool bot_on = true;
    float b_p1, b_inv_p1, b_inv_w, b_psh, b_ta1, b_hur1, b_dta, b_dhur;
    {
        const F4 xs = blend4(rs0, rs1);
        const bool has = s_node >= 1;
        b_p1 = has ? s_plev[j_s1] : 0.0f;
        b_inv_p1 = has ? s_inv_plev[j_s1] : 1.0f;
        b_psh = has ? psh : 0.0f;
        b_inv_w = has ? fast_rcp(fast_lg2(psh * b_inv_p1)) : 0.0f;
        b_ta1 = has ? xs.x : sfc_ta; b_hur1 = has ? xs.y : sfc_hur;
        b_dta = sfc_ta - b_ta1; b_dhur = sfc_hur - b_hur1;
    }

    struct Dlt { float ta, hur, ua, va; };
    // element offset of node w_lo - 2 (the next one to fetch); one node down = +-ncol in the file
    const int32_t off_step = desc ? (int32_t)n : -(int32_t)n;
    uint32_t off_m = node_off(w_lo >= 2 ? w_lo - 2 : 0);
    // A step only switches the bracket (x_lo <- nb); bringing nb and the raw slabs up to date (`refresh`) is
    // deferred to ONE place per pair iteration, after both walks.  The lanes of a warp cross a node at
    // different levels, and the scoreboard tracks registers per warp: with the loads issued inside the step,
    // the step of the next lanes (same iteration, or the next one) waited on loads it did not need.  Now the
    // first use of a load is at least one whole pair iteration after its issue.
    bool stale = false;
    auto refresh = [&]() {
        nb = blend4(m0, m1);                                    // node w_lo-1: first use of its loads
        // the new loads are ordered behind the reads of the registers they replace
        const int zero = reg_fence(nb.x, nb.y, nb.z, nb.w);
        off_m += off_step;
        if (w_lo >= 2) { m0 = ldg4(d4lo + off_m + zero); m1 = ldg4(d4hi + off_m + zero); }
        if (w_lo >= kL2Ahead) {
            const uint32_t off = off_m + (uint32_t)((kL2Ahead - 2) * off_step);
            asm volatile("prefetch.global.L2 [%0];" ::"l"(d4lo + off));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(d4hi + off));
        }
        stale = false;
    };
    auto step_to = [&](float p) {
        while (w_p_lo > p) {
            if (stale) refresh();                               // a second step within one pair iteration (rare)
            const F4 hi = x_lo;
            --w_lo;
            if (w_lo >= 0) {
                w_p_lo = s_plev[w_lo]; w_inv_p_lo = s_inv_plev[w_lo]; w_inv_w = s_inv_w[w_lo];
                x_lo = nb;
                x_d = F4{hi.x - x_lo.x, hi.y - x_lo.y, hi.z - x_lo.z, hi.w - x_lo.w};
                stale = true;
            } else {
                // above node 0: constant extrapolation with node 0's values; p_lo = 0 ends the walk
                x_d = F4{0.f, 0.f, 0.f, 0.f}; w_inv_w = 0.0f; w_p_lo = 0.0f; w_inv_p_lo = 1.0f;
            }
        }
    };
    auto interp = [&](float p) {
        const float t = fast_lg2(p * w_inv_p_lo) * w_inv_w;
        // t == 0: exact node hit or constant extrapolation -> the node value itself (NaN-safe)
        const bool ex = (t == 0.0f);
        Dlt d;
#if PGW_X2
        const float2 tt = make_float2(t, t);
        const float2 ab = __ffma2_rn(tt, make_float2(x_d.x, x_d.y), make_float2(x_lo.x, x_lo.y));
        const float2 cd = __ffma2_rn(tt, make_float2(x_d.z, x_d.w), make_float2(x_lo.z, x_lo.w));
        d.ta = ex ? x_lo.x : ab.x;
        d.hur = ex ? x_lo.y : ab.y;
        d.ua = ex ? x_lo.z : cd.x;
        d.va = ex ? x_lo.w : cd.y;
#else
        d.ta = ex ? x_lo.x : fmaf(t, x_d.x, x_lo.x);
        d.hur = ex ? x_lo.y : fmaf(t, x_d.y, x_lo.y);
        d.ua = ex ? x_lo.z : fmaf(t, x_d.z, x_lo.z);
        d.va = ex ? x_lo.w : fmaf(t, x_d.w, x_lo.w);
#endif
        return d;
    };
    auto walk = [&](float p) { step_to(p); return interp(p); };
#if PGW_UNIFORM_TOP
    // the same for a level with a column-independent pressure: node and weight from the CTA's table
    auto walk_uniform = [&](int l) {
        const int nd = s_un[l];
        while (w_lo > nd) {
            if (stale) refresh();
            const F4 hi = x_lo;
            --w_lo;
            if (w_lo >= 0) {
                w_p_lo = s_plev[w_lo]; w_inv_p_lo = s_inv_plev[w_lo]; w_inv_w = s_inv_w[w_lo];
                x_lo = nb;
                x_d = F4{hi.x - x_lo.x, hi.y - x_lo.y, hi.z - x_lo.z, hi.w - x_lo.w};
                stale = true;
            } else {
                x_d = F4{0.f, 0.f, 0.f, 0.f}; w_inv_w = 0.0f; w_p_lo = 0.0f; w_inv_p_lo = 1.0f;
            }
        }
        const float t = s_ut[l];
        Dlt d;
        if (t == 0.0f) {                     // CTA-uniform: exact node hit or constant extrapolation
            d.ta = x_lo.x; d.hur = x_lo.y; d.ua = x_lo.z; d.va = x_lo.w;
        } else {
            const float2 tt = make_float2(t, t);
            const float2 ab = __ffma2_rn(tt, make_float2(x_d.x, x_d.y), make_float2(x_lo.x, x_lo.y));
            const float2 cd = __ffma2_rn(tt, make_float2(x_d.z, x_d.w), make_float2(x_lo.z, x_lo.w));
            d.ta = ab.x; d.hur = ab.y; d.ua = cd.x; d.va = cd.y;
        }
        return d;
    };
#endif
    auto sfc_override = [&](float p, Dlt &d) {
        if (bot_on) {
            if (p > b_p1) {
                const float tb = fast_lg2(p * b_inv_p1) * b_inv_w;
                const bool below = p >= b_psh;
                d.ta = below ? sfc_ta : fmaf(tb, b_dta, b_ta1);
                d.hur = below ? sfc_hur : fmaf(tb, b_dhur, b_hur1);
            } else bot_on = false;
        }
    };

    LnConst lk{2.0 / 3.0, 2.0 / 5.0, 2.0 / 7.0};
    asm volatile("" : "+d"(lk.c3), "+d"(lk.c5), "+d"(lk.c7));     // keep the constants in registers

    const double pref = a.p_ref;
    const double2 hl_sfc = s_hl[L];
    double pb_era = fma(PSd, hl_sfc.y, hl_sfc.x);
    double acc_era = 0.0;
    bool era_open = pb_era >= pref;                 // still below p_ref
    if (!era_open) { errbits |= PGW_ERR_PREF_BELOW_SFC; k_pref = 0; }
    float psn_f = ps_f;                             // ps used for QV; replaced after the iteration

    // ---------------- the geopotential sums of the parked levels ----------------
    // The fixed point needs phi(p_ref) of the PGW state for ps = PS + x, x = dps_k.  (T, e) of the parked
    // levels are kept in tensor memory, but instead of re-integrating all of them in every iteration, the
    // sum over the layers that lie safely below p_ref is expanded ONCE, during the sweep, as a polynomial
    // in x:
    //   ln(P_h + b_h x) = ln P_h + u x - (u x)^2/2 + (u x)^3/3 - (u x)^4/4,  u = b_h / P_h <= 1/PS,
    //   Tv_l(x) = T_l + (T c e/Q)(1 - w x + w^2 x^2 - w^3 x^3),  Q = p_l - 0.378 e,  w = bm_l / Q,
    // dry part in float64 to x^4, humidity part (1 % of the sum) in float32 to x^3: for |x| <= 0.012 PS the
    // truncation error is below 2e-5 m2/s2 (the fp32 storage of e costs as much).  Only the three layers
    // around p_ref (whose membership changes with x) are integrated directly in every iteration.  A warp
    // in which some column leaves that range in iteration k (the first step of the iteration can overshoot
    // by several thousand Pa over high terrain) integrates all its parked levels for that k, as before.
    // T_pgw enters as fp32; its rounding residual r_l (|r_l| <= 1.5e-5 K) enters the geopotential as
    // Rd * sum_l r_l dlnp_l, taken once with the ERA pressures (change over the iteration < 1e-8 m2/s2).
    double acc_res = 0.0, acc_T0 = 0.0, acc_part0 = 0.0, t_low_d = 0.0;
    double S1 = 0.0, S2 = 0.0, S3 = 0.0, S4 = 0.0;            // sum_l T_l (ub^k - ut^k)
    float H1 = 0.0f, H2 = 0.0f, H3 = 0.0f;                    // humidity part, coefficients of x, x^2, x^3
    // the layer that contains p_ref for x = 0 (-1: none).  Written once, in shared memory: a register for it across
    // the parked pairs costs a spill there.
    s_lstar[ct] = -1;
    auto rcp64 = [](double v) { double r = rcp64_approx(v); return fma(r, fma(-v, r, 1.0), r); };
    // add sgn * (contribution of the fully-below layer l) to the polynomial
    auto taylor_add = [&](int l, double Pb, double Pt, double tpd, float hq, float w, float dl, double sgn) {
        const double ub = s_hl[l + 1].y * rcp64(Pb), ut = s_hl[l].y * rcp64(Pt);
        const double d1 = ub - ut, sm = ub + ut, m2 = ub * ut;
        const double q2 = fma(sm, sm, -2.0 * m2);            // ub^2 + ut^2
        const double d2 = d1 * sm, d3 = d1 * (q2 + m2), d4 = d2 * q2;
        const double ts = sgn * tpd;
        S1 = fma(ts, d1, S1); S2 = fma(ts, d2, S2); S3 = fma(ts, d3, S3); S4 = fma(ts, d4, S4);
        const float D1 = (float)d1, D2 = -0.5f * (float)d2, D3 = (1.0f / 3.0f) * (float)d3;
        const float hs = (float)sgn * hq, w2 = w * w;
        H1 = fmaf(hs, fmaf(-w, dl, D1), H1);
        H2 = fmaf(hs, fmaf(w2, dl, fmaf(-w, D1, D2)), H2);
        H3 = fmaf(hs, fmaf(-w2 * w, dl, fmaf(w2, D1, fmaf(-w, D2, D3))), H3);
    };
    // One parked level, bottom-up: the ERA geopotential (functions.py:128-189), iteration 0 of the
    // PGW state (same pressures) and the polynomial of the later iterations.
    auto era_layer = [&](int l, float p, float bm, float t, float q, float dta, float t_pgw, float e_pgw) {
        if (era_open) {
            const double2 hl = s_hl[l];
            const double Pt = fma(PSd, hl.y, hl.x);
            double pt = Pt;
            if (pt < pref) { pt = pref; era_open = false; s_lstar[ct] = l; }   // layer that contains p_ref (:174-179)
            const double td = (double)t, tpd = (double)t_pgw;
            const double rtv = rd_tv(t, q);                          // Rd * Tv of the ERA state, float32 products
            const float g = fast_rcp(fmaf(-0.378f, e_pgw, p));
            const float hq_t = (0.61f * 0.622f) * e_pgw * g;         // (Tv - T) / T of the PGW state
            const double tvp = fma(tpd, (double)hq_t, tpd);
            const double dl = ln_ratio<FAST>(pb_era, pt, lk);
            acc_era = fma(rtv, dl, acc_era);
            acc_res = fma((td + (double)dta) - tpd, dl, acc_res);
            if (era_open) {
                acc_T0 = fma(tvp, dl, acc_T0);
                taylor_add(l, pb_era, Pt, tpd, t_pgw * hq_t, bm * g, (float)dl, 1.0);
            } else {
                acc_part0 = tvp * dl;
            }
            pb_era = Pt;
        }
    };

    // ---------------- phase 2: surface-pressure fixed point (step_03:182-319) ----------------
    // and phase 3a: PS and QV of the parked levels.  Runs once, between the parked and the
    // streamed pairs; the TMA loads of the next pairs are in flight meanwhile.
    auto fixed_point = [&]() {
        const double fis = (double)r_fis;
        const double phi_era = fis + acc_era;                            // acc_era holds Rd * Tv * dlnp
        const double gdzg = blend_f64(a.zg_ref, r_zg) * kG;              // step_03:292-295
        const double t_low = t_low_d;                                 // ta_pgw on the lowest level
        int lstar = s_lstar[ct];
        const bool no_star = lstar < 0;                               // p_ref not reached among the parked levels
        if (no_star) lstar = lst;
        const double acc_k0 = acc_T0 + acc_part0;                     // iteration 0: x = 0, all layers
        // the layer right below l* joins the directly integrated ones: take it out of the polynomial
        const int ld_hi = min(lstar + 1, L - 1), ld_lo = max(lstar - 1, lst);
        auto scol = [&](int l) { return tm + (uint32_t)(2 * (L - 1 - l)); };   // stash columns of level l
        tmem_wait_st();
        // (T_pgw, e_pgw) of the directly integrated layers ld_hi, ld_hi-1, ld_hi-2 (>= ld_lo) in registers.  The
        // lanes' layers differ and a TMEM load takes one column address per warp: walk the warp's range.
        float2 te_d0 = make_float2(0.f, 0.f), te_d1 = te_d0, te_d2 = te_d0;
        for (int l = __reduce_max_sync(0xffffffffu, ld_hi), lo = __reduce_min_sync(0xffffffffu, ld_lo); l >= lo; --l) {
            const float2 v = tmem_ld2(scol(l));
            if (l == ld_hi) te_d0 = v;
            if (l == ld_hi - 1) te_d1 = v;
            if (l == ld_hi - 2) te_d2 = v;
        }
        if (lstar + 1 <= L - 1) {
            const int l = lstar + 1;
            const double2 ht = s_hl[l], hb = s_hl[l + 1];
            const float2 m = s_m[l];
            const float2 te = te_d0;                                  // l == ld_hi
            const double Pt = fma(PSd, ht.y, ht.x), Pb = fma(PSd, hb.y, hb.x);
            const float g = fast_rcp(fmaf(-0.378f, te.y, fmaf(ps_f, m.y, m.x)));
            const float hq_t = (0.61f * 0.622f) * te.y * g;
            const double tpd = (double)te.x;
            const double dl = ln_ratio<FAST>(Pb, Pt, lk);
            acc_T0 = fma(-fma(tpd, (double)hq_t, tpd), dl, acc_T0);
            taylor_add(l, Pb, Pt, tpd, te.x * hq_t, m.y * g, (float)dl, -1.0);
        }
        const double c1 = S1 + (double)H1, c2 = fma(-0.5, S2, (double)H2), c3 = fma(1.0 / 3.0, S3, (double)H3),
                     c4 = -0.25 * S4;
        const double2 h_hi = s_hl[ld_hi + 1];
        const double x_max = kTaylorMaxRel * PSd;
        double dps = 0.0, adj = 0.0, psn = PSd;
        int ltop = lst + 1;                 // direct integration: first layer (from the top) entirely below p_ref
        float *traj = a.dps_traj + c;
        for (int k = 0; k < a.k_spec; ++k, traj += n) {
            dps += adj;
            psn = PSd + dps;
            psn_f = (float)psn;
            if (valid) *traj = (float)dps;
            if (psn > a.ps_bound) { errbits |= PGW_ERR_PS_BOUND; k_bound = min(k_bound, k); }
            double pb = fma(psn, hl_sfc.y, hl_sfc.x);
            if (pb < pref) { errbits |= PGW_ERR_PREF_BELOW_SFC; k_pref = min(k_pref, k); }
            // Tv = T (1 + 0.61 hus), hus = 0.622 e / (p - 0.378 e)   (functions.py:66-72, :144)
            auto layer = [&](int l, const float2 te, double pt_or_ref, double acc_in) {
                const float2 m = s_m[l];
                const double Td = (double)te.x;
                const float g = fast_rcp(fmaf(-0.378f, te.y, fmaf(psn_f, m.y, m.x)));
                const double tv = fma(Td, (double)((0.61f * 0.622f) * te.y * g), Td);
                return fma(tv, ln_ratio<FAST>(pb, pt_or_ref, lk), acc_in);
            };
            double acc = acc_res;
            // polynomial usable by every column of the warp for this x?
            const double p_edge = fma(psn, h_hi.y, h_hi.x);       // bottom of the directly integrated layers
            const bool poly_ok = !(no_star || !(fabs(dps) <= x_max) || p_edge < pref ||
                                   fma(psn, s_hl[ld_lo].y, s_hl[ld_lo].x) >= pref);
            if (k == 0) {
                acc += acc_k0;              // psn == PS: summed in phase 1 together with the ERA state
            } else if (__all_sync(0xffffffffu, poly_ok || !valid)) {
                acc = fma(dps, fma(dps, fma(dps, fma(dps, c4, c3), c2), c1), acc + acc_T0);
                // the layers around p_ref, top-down from the polynomial's upper edge (functions.py:174-179)
                pb = p_edge;
                for (int l = ld_hi; l >= ld_lo; --l) {
                    const double2 hl = s_hl[l];
                    const double pt = fma(psn, hl.y, hl.x);
                    const bool part = pt < pref;
                    acc = layer(l, l == ld_hi ? te_d0 : (l == ld_hi - 1 ? te_d1 : te_d2), part ? pref : pt, acc);
                    pb = pt;
                    if (part) break;
                }
            } else {
                if ((tid & 31) == 0 && a.poly_fallback) atomicAdd(a.poly_fallback, 1u);
                // layers ltop..L-1 are entirely below p_ref for this ps; it moves by at most a level or two
                while (ltop > lst) { const double2 h = s_hl[ltop - 1]; if (fma(psn, h.y, h.x) >= pref) --ltop; else break; }
                while (ltop < L) { const double2 h = s_hl[ltop]; if (fma(psn, h.y, h.x) < pref) ++ltop; else break; }
                // bottom-up: the whole layers ltop..L-1, then ltop-1 (>= lst) up to p_ref if it lies below it
                // (:174-179).  The stash is read for the whole warp, four levels per load, as far as any lane goes.
                const int nlv = __reduce_max_sync(0xffffffffu, min(L - ltop + 1, np));
#pragma unroll 1
                for (int g = 0; g < nlv; g += 4) {
                    float v[8];
                    tmem_ld8(tm + (uint32_t)(2 * g), v);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int l = L - 1 - g - q;
                        const bool whole = l >= ltop, part = !whole && l == ltop - 1 && l >= lst && pb >= pref;
                        if (whole || part) {
                            const double2 hl = s_hl[l];
                            const double pt = whole ? fma(psn, hl.y, hl.x) : pref;
                            acc = layer(l, make_float2(v[2 * q], v[2 * q + 1]), pt, acc);
                            pb = pt;
                        }
                    }
                }
            }
            const double phi_pgw = fis + kRd * acc;
            const double err = (phi_pgw - phi_era) - gdzg;
            adj = -a.adj_factor * psn / (kRd * t_low) * err;
            double ae = (isnan(err) || !valid) ? 0.0 : fabs(err);      // max skips NaN (step_03:308)
            ae = warp_max(ae);
            if ((tid & 31) == 0 && ae > 0.0)
                atomicMax(reinterpret_cast<unsigned long long *>(a.maxerr + k),
                          (unsigned long long)__double_as_longlong(ae));
        }
        if (valid) {
            a.PS_out[c] = psn_f;
            a.dps_out[c] = (float)dps;
        }
        uint32_t o2 = (uint32_t)(L - 1) * n + c;
        float *const oQ = a.QV_out;
#pragma unroll 1
        for (int g = 0; g < np; g += 8) {
            float v[16];
            tmem_ld16(tm + (uint32_t)(2 * g), v);          // levels L-1-g .. L-8-g
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int l = L - 1 - g - q;
                if (l >= lst) {
                    const float qv = qv_from_e(v[2 * q + 1], psn_f, s_m[l]);
                    if (valid) st_stream(oQ + o2, qv);
                    o2 -= n;
                }
            }
        }
        // the stash is dead: give the columns back now rather than at exit (the next CTA on this SM waits for them)
        tmem_fence_before_sync();
        asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");    // the four column warps
        if (ct < 32) {
            tmem_fence_after_sync();
            tmem_dealloc(tm, ncols);
        }
    };

    // ---------------- the sweep: parked pairs, fixed point, streamed pairs ----------------
    // one level pair; `parked` is a compile-time tag so that each of the two loops below gets its own body
    auto pair_body = [&](const int j, auto parked_c) {
        constexpr bool parked = decltype(parked_c)::value;
        const int l = max(L - 1 - 2 * j, 1);          // last pair of an odd column: levels (1, 0) again
        float2 mm0, mm1;
        if (parked) { mm0 = s_m[l]; mm1 = s_m[l - 1]; } else { mm0 = tp.m[l]; mm1 = tp.m[l - 1]; }
        float *const sl = ring + (j % kTmaSlots) * 8 * NT + ct;
        // the walks need no slot data: they cover the round trip of the barrier probe (~100 cycles)
        const bool ready = mbar_test(bar_full + (j % kTmaSlots), (j / kTmaSlots) & 1);
#if PGW_X2
        const float2 p01 = __ffma2_rn(make_float2(ps_f, ps_f), make_float2(mm0.y, mm1.y), make_float2(mm0.x, mm1.x));
        const float p0 = p01.x, p1 = p01.y;
#else
        const float p0 = fmaf(ps_f, mm0.y, mm0.x), p1 = fmaf(ps_f, mm1.y, mm1.x);
#endif
#if PGW_UNIFORM_TOP
        Dlt d0, d1;
        if (!parked && mm0.y == 0.0f && mm1.y == 0.0f) { d0 = walk_uniform(l); d1 = walk_uniform(l - 1); }
        else { d0 = walk(p0); d1 = walk(p1); }
#else
        Dlt d0 = walk(p0);
        Dlt d1 = walk(p1);
#endif
        if (stale) refresh();
        if (!ready) mbar_wait(bar_full + (j % kTmaSlots), (j / kTmaSlots) & 1);
        const float t0 = sl[NT], q0 = sl[3 * NT], u0 = sl[5 * NT], v0 = sl[7 * NT];    // row 1: level l
        const float t1 = sl[0], q1 = sl[2 * NT], u1 = sl[4 * NT], v1 = sl[6 * NT];     // row 0: level l-1
        if (__any_sync(0xffffffffu, bot_on)) { sfc_override(p0, d0); sfc_override(p1, d1); }
        const bool cold = __all_sync(0xffffffffu, is_cold(t0, d0.ta) && is_cold(t1, d1.ta));
#if PGW_X2
        const float2 e01 = thermo_e_pgw_x2(cold, make_float2(p0, p1), make_float2(t0, t1), make_float2(q0, q1),
                                           make_float2(d0.ta, d1.ta), make_float2(d0.hur, d1.hur));
        const float e0 = e01.x, e1 = e01.y;
#else
        const float e0 = thermo_e_pgw(cold, p0, t0, q0, d0.ta, d0.hur);
        const float e1 = thermo_e_pgw(cold, p1, t1, q1, d1.ta, d1.hur);
#endif
#if PGW_X2
        const float2 tp01 = __fadd2_rn(make_float2(t0, t1), make_float2(d0.ta, d1.ta));
        const float2 up01 = __fadd2_rn(make_float2(u0, u1), make_float2(d0.ua, d1.ua));
        const float2 vp01 = __fadd2_rn(make_float2(v0, v1), make_float2(d0.va, d1.va));
        const float tp0 = tp01.x, tp1 = tp01.y;
        sl[NT] = tp0; sl[5 * NT] = up01.x; sl[7 * NT] = vp01.x;
        sl[0] = tp1; sl[4 * NT] = up01.y; sl[6 * NT] = vp01.y;
#else
        const float tp0 = t0 + d0.ta, tp1 = t1 + d1.ta;   // == (float)((double)t + (double)dta)
        sl[NT] = tp0; sl[5 * NT] = u0 + d0.ua; sl[7 * NT] = v0 + d0.va;
        sl[0] = tp1; sl[4 * NT] = u1 + d1.ua; sl[6 * NT] = v1 + d1.va;
#endif
        if (parked) {
            fence_proxy_async();
            mbar_arrive(bar_done + (j % kTmaSlots));
            tmem_st4(tm + (uint32_t)(4 * j), tp0, e0, tp1, e1);     // levels l, l-1 = L-1-2j, L-2-2j
            if (j == 0) t_low_d = (double)t0 + (double)d0.ta;
            era_layer(l, p0, mm0.y, t0, q0, d0.ta, tp0, e0);
            era_layer(l - 1, p1, mm1.y, t1, q1, d1.ta, tp1, e1);
        } else {
#if PGW_X2
            const float2 pn = __ffma2_rn(make_float2(psn_f, psn_f), make_float2(mm0.y, mm1.y), make_float2(mm0.x, mm1.x));
            const float2 den = __ffma2_rn(make_float2(-0.378f, -0.378f), e01, pn);
            const float2 qv = __fmul2_rn(__fmul2_rn(make_float2(0.622f, 0.622f), e01),
                                         make_float2(fast_rcp(den.x), fast_rcp(den.y)));
            sl[3 * NT] = qv.x;                            // functions.py:66-72 with the adjusted ps
            sl[2 * NT] = qv.y;
#else
            sl[3 * NT] = qv_from_e(e0, psn_f, mm0);       // functions.py:66-72 with the adjusted ps
            sl[2 * NT] = qv_from_e(e1, psn_f, mm1);
#endif
            fence_proxy_async();
            mbar_arrive(bar_done + (j % kTmaSlots));
        }
    };
#ifdef PGW_TMA_ONE_LOOP
#pragma unroll 1
    for (int j = 0; j <= npairs; ++j) {
        if (j == np1) fixed_point();                  // np1 <= npairs: exactly once
        if (j == npairs) break;
        if (j < np1) pair_body(j, TagParked{}); else pair_body(j, TagStreamed{});
    }
#else
#pragma unroll kUnrollParked
    for (int j = 0; j < np1; ++j) pair_body(j, TagParked{});
    fixed_point();
#pragma unroll kUnrollStreamed
    for (int j = np1; j < npairs; ++j) pair_body(j, TagStreamed{});
#endif

    // ---------------- bookkeeping for the host-side checks ----------------
    const float2 m_top = tp.m[0];
    float p_top = fmaf(ps_f, m_top.y, m_top.x);                          // functions.py:417
    p_top = warp_min(p_top);
    const float min_src_p = warp_min(min_src_p0);
    if ((tid & 31) == 0) {
        atomicMin(reinterpret_cast<unsigned *>(a.stats), __float_as_uint(fmaxf(p_top, 0.0f)));
        atomicMin(reinterpret_cast<unsigned *>(a.stats) + 1, __float_as_uint(fmaxf(min_src_p, 0.0f)));
    }
    if (errbits && valid) {
        atomicOr(a.err, errbits);
        if (a.first_k) {
            if (k_pref != INT32_MAX) atomicMin(a.first_k, k_pref);
            if (k_bound != INT32_MAX) atomicMin(a.first_k + 1, k_bound);
        }
    }
}

}  // namespace pgw

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
namespace {

using pgw::kColumnThreads;

// sm_100: 228 KB of shared memory and 512 tensor-memory columns per SM, 1 KB of shared memory reserved per CTA
constexpr size_t kSmemPerSm = 228 * 1024, kSmemReservedPerCta = 1024;
constexpr int kTmemColsPerSm = 512;

// tensor-memory columns of a CTA: (T_pgw, e_pgw) of np levels, allocated in powers of two >= 32
int tmem_cols_tma(int np) {
    int c = 32;
    while (c < 2 * np) c <<= 1;
    return c;
}

// Shared memory per CTA.  It is padded to the CTA's share of the SM's tensor memory, so that the CTAs that fit by
// shared memory (of this kernel, whichever plan, e.g. the next launch on another stream) also fit by tensor memory
// and tcgen05.alloc never waits: 128 columns -> 56 KB (4 CTAs, the register limit anyway), 256 -> 113 KB, 512 -> 227 KB.
size_t column_smem_tma(int nplev, int np, int nlev) {
    const int nt = kColumnThreads;
    size_t b = sizeof(float) * (size_t)pgw::kTmaSlots * 8 * nt +            // pair ring
               sizeof(double) * 2 * (size_t)(np + 1) + sizeof(float) * 2 * (size_t)np;
    b += sizeof(float) * (size_t)(3 * nplev + ((3 * nplev) & 1));
#if PGW_UNIFORM_TOP
    b += 2 * sizeof(float) * (size_t)(nlev + (nlev & 1));
#endif
    b += sizeof(uint64_t) * 2 * pgw::kTmaSlots + sizeof(uint32_t) * (1 + nt);   // barriers, TMEM address, l*
    const size_t share = kSmemPerSm * (size_t)tmem_cols_tma(np) / kTmemColsPerSm - kSmemReservedPerCta;
    return b > share ? b : share;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

// libcuda is not linked: the encoder is looked up through the runtime
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        cudaGetLastError();
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Encoded maps are remembered per (base address, ncol, nlev): a pipeline cycles through a handful of input and
// output buffers, and eight driver calls per launch were a visible part of the host time per timestep.
struct MapCacheEntry { const float *base; long long ncol; int nlev; CUtensorMap map; };
constexpr int kMapCache = 128;

int encode_map(CUtensorMap *m, const float *base, long long ncol, int nlev);

int make_map(CUtensorMap *m, const float *base, long long ncol, int nlev) {
    static thread_local MapCacheEntry cache[kMapCache];
    static thread_local int used = 0, next = 0;
    for (int i = 0; i < used; ++i)
        if (cache[i].base == base && cache[i].ncol == ncol && cache[i].nlev == nlev) { *m = cache[i].map; return PGW_OK; }
    const int rc = encode_map(m, base, ncol, nlev);
    if (rc != PGW_OK) return rc;
    MapCacheEntry &e = cache[next];
    e.base = base; e.ncol = ncol; e.nlev = nlev; e.map = *m;
    next = (next + 1) % kMapCache;
    if (used < kMapCache) ++used;
    return PGW_OK;
}

int encode_map(CUtensorMap *m, const float *base, long long ncol, int nlev) {
    const cuuint64_t dims[2] = {(cuuint64_t)ncol, (cuuint64_t)nlev};
    const cuuint64_t strides[1] = {(cuuint64_t)ncol * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)kColumnThreads, 2u};
    const cuuint32_t estr[2] = {1u, 1u};
    CUresult r = encode_tiled()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box,
                                estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        pgw_set_error("cuTensorMapEncodeTiled failed (%d)", (int)r);
        return PGW_E_LAUNCH;
    }
    return PGW_OK;
}

}  // namespace

bool pgw_tma_eligible(const pgw_timestep_args *a, int lst_generic, int *lst_tma, size_t *smem) {
    const int np = a->nlev - lst_generic;
    const int lst_even = lst_generic - (np & 1);        // whole level pairs are parked
    if (!(a->akm_host && a->bkm_host) || lst_even < 0 || a->nlev > pgw::kTmaMaxLev || a->ncol % 4 != 0 ||
        a->ncol < kColumnThreads || a->ncol >= (1ll << 31))
        return false;
    const void *f[8] = {a->T, a->QV, a->U, a->V, a->T_out, a->QV_out, a->U_out, a->V_out};
    for (const void *p : f) if (!aligned16(p)) return false;
    if (!encode_tiled()) return false;
    *lst_tma = lst_even;
    *smem = column_smem_tma(a->nplev, a->nlev - lst_even, a->nlev);
    return true;
}

bool pgw_tma_l137(const pgw_timestep_args *a, const pgw_column_plan &plan) {
    return a->nlev == 137 && plan.np == 56 && plan.lst == 137 - 56;
}

int pgw_tma_tmem_cols(int np) { return tmem_cols_tma(np); }

int pgw_launch_column_tma(const pgw_timestep_args *a, const pgw_column_plan &plan, cudaStream_t st) {
    int rc;
    pgw::TmaParams tp;
    const float *in[4] = {a->T, a->QV, a->U, a->V};
    float *out[4] = {a->T_out, a->QV_out, a->U_out, a->V_out};
    for (int v = 0; v < 4; ++v) {
        if ((rc = make_map(&tp.in[v], in[v], a->ncol, a->nlev)) != PGW_OK) return rc;
        if ((rc = make_map(&tp.out[v], out[v], a->ncol, a->nlev)) != PGW_OK) return rc;
    }
    for (int l = 0; l < pgw::kTmaMaxLev; ++l)
        tp.m[l] = l < a->nlev ? make_float2((float)a->akm_host[l], (float)a->bkm_host[l]) : make_float2(0.f, 0.f);
    const bool l137 = pgw_tma_l137(a, plan);
    auto kern = plan.fast ? (l137 ? pgw::pgw_column_tma_kernel<true, 137, 56> : pgw::pgw_column_tma_kernel<true, 0, 0>)
                          : (l137 ? pgw::pgw_column_tma_kernel<false, 137, 56> : pgw::pgw_column_tma_kernel<false, 0, 0>);
    if ((rc = pgw_ensure_smem((const void *)kern, 4 + (plan.fast ? 1 : 0) + (l137 ? 2 : 0), plan.smem, plan.np)) != PGW_OK)
        return rc;
    const unsigned grid = (unsigned)((a->ncol + kColumnThreads - 1) / kColumnThreads);
    kern<<<grid, 2 * kColumnThreads, plan.smem, st>>>(*a, tp, plan.lst, plan.np, (uint32_t)tmem_cols_tma(plan.np));
    return pgw_check_launch("pgw_column_tma_kernel");
}

extern "C" int pgw_column_tma_layout(int nplev, int nlev, int np, int *tmem_cols, long long *smem_bytes) {
    if (nplev < 2 || nplev > 64 || nlev < 2 || nlev > pgw::kTmaMaxLev || np < 2 || np > nlev || (np & 1) ||
        !tmem_cols || !smem_bytes)
        return PGW_E_INVALID;
    *tmem_cols = tmem_cols_tma(np);
    *smem_bytes = (long long)column_smem_tma(nplev, np, nlev);
    return PGW_OK;
}
