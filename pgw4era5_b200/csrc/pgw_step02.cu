// step_02 kernels of libpgw_b200 (sm_100a): bilinear regridding of GCM deltas
// to the ERA5 grid (regrid_lat_lon, functions.py:748-898) and the spectral
// smoothing of daily annual cycles (filter_data / harmonic_ac_analysis,
// functions.py:606-740).  Both are pure streaming: regridding is write-bound
// (a 1 degree source field fits in L2, the 0.25 degree target is 16x larger),
// smoothing reads and writes every series once.
#include "pgw_common.cuh"

#include <cuda_pipeline.h>
#include <limits.h>
#include <stdlib.h>
#include <string.h>

int pgw_ensure_smem(const void *kernel, int slot, size_t smem, int np);

namespace pgw {

// zonal mean of the first and last source row of every field: the values the
// reference puts on the synthetic pole rows (functions.py:833-842).  The reference
// takes it with xarray's DataArray.mean, which skips NaN for float data: the mean of
// the valid points of the row, NaN only when the whole row is missing.
__global__ void __launch_bounds__(128)
zonal_mean_kernel(const float *__restrict__ src, float *__restrict__ polemean, long long nfield, int ny_s,
                  int nx_s) {
    const long long f = blockIdx.x;
    const int which = blockIdx.y;                   // 0: row 0, 1: row ny_s-1
    const float *row = src + (f * ny_s + (which ? ny_s - 1 : 0)) * (long long)nx_s;
    double s = 0.0;
    int n = 0;
    for (int i = threadIdx.x; i < nx_s; i += blockDim.x) {
        const float v = row[i];
        if (!isnan(v)) { s += (double)v; ++n; }
    }
    __shared__ double part[4];
    __shared__ int cnt[4];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        n += __shfl_xor_sync(0xffffffffu, n, o);
    }
    if ((threadIdx.x & 31) == 0) { part[threadIdx.x >> 5] = s; cnt[threadIdx.x >> 5] = n; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        int c = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { t += part[w]; c += cnt[w]; }
        polemean[f * 2 + which] = c ? (float)(t / (double)c) : NAN;
    }
}

__device__ __forceinline__ double src_at(const float *fld, const float *pm, int j, int i, int nx_s) {
    if (j == -1) return (double)pm[0];
    if (j == -2) return (double)pm[1];
    return (double)__ldg(fld + (long long)j * nx_s + i);
}

// one thread = VEC consecutive target longitudes of one (field, target row)
template <int VEC>
__global__ void __launch_bounds__(256)
regrid_kernel(const float *__restrict__ src, float *__restrict__ dst, const float *__restrict__ polemean,
              long long nfield, int ny_s, int nx_s, int ny_t, int nx_t, const int *__restrict__ j0,
              const int *__restrict__ j1, const double *__restrict__ wy, const int *__restrict__ i0,
              const int *__restrict__ i1, const double *__restrict__ wx) {
    const int nxv = nx_t / VEC;
    const long long total = nfield * ny_t * (long long)nxv;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int iv = (int)(idx % nxv);
        const long long r = idx / nxv;
        const int jt = (int)(r % ny_t);
        const long long f = r / ny_t;
        const float *fld = src + f * ny_s * (long long)nx_s;
        const float *pm = polemean + f * 2;
        const int ja = j0[jt], jb = j1[jt];
        const double wj = wy[jt];
        float res[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const int it = iv * VEC + v;
            const int ia = i0[it], ib = i1[it];
            // latitude pass (functions.py:859), then longitude pass (:892)
            const double a0 = src_at(fld, pm, ja, ia, nx_s), a1 = src_at(fld, pm, jb, ia, nx_s);
            const double b0 = src_at(fld, pm, ja, ib, nx_s), b1 = src_at(fld, pm, jb, ib, nx_s);
            const double a = (a1 - a0) * wj + a0;
            const double b = (b1 - b0) * wj + b0;
            res[v] = (float)((b - a) * wx[it] + a);
        }
        float *o = dst + (f * ny_t + jt) * (long long)nx_t + (long long)iv * VEC;
        if (VEC == 4) __stcs(reinterpret_cast<float4 *>(o), make_float4(res[0], res[1], res[2], res[3]));
        else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) __stcs(o + v, res[v]);
        }
    }
}

// Row-wise variant for target rows that fit one CTA (nx_t / VEC <= blockDim, nx_s <= 2048), the
// case of every ERA5 grid: a CTA walks over (field, target row) pairs.  Per row, (A) the two
// bracketing source rows are blended in latitude ONCE per source column into shared memory
// (functions.py:859), (B) every thread produces VEC adjacent target longitudes from that row with
// the longitude brackets and weights it keeps in registers for the whole kernel (:892).  The blended
// row is double buffered, so one barrier per row suffices.  Same expressions, hence bit-identical
// to regrid_kernel, at about a quarter of its instructions per point: the 16x larger target field
// makes this a store-bound kernel.
template <int VEC>
__global__ void __launch_bounds__(384)
regrid_rows_kernel(const float *__restrict__ src, float *__restrict__ dst, const float *__restrict__ polemean,
                   int nfield, int ny_s, int nx_s, int ny_t, int nx_t, const int *__restrict__ j0,
                   const int *__restrict__ j1, const double *__restrict__ wy, const int *__restrict__ i0,
                   const int *__restrict__ i1, const double *__restrict__ wx) {
    extern __shared__ double2 s_row[];              // [2 buffers][nx_s] (row of jt0, row of jt1)
    const int nxv = nx_t / VEC;
    const int tid = threadIdx.x;
    const bool owner = tid < nxv;
    int ia[VEC], ib[VEC];
    double w[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        const int it = owner ? tid * VEC + v : 0;
        ia[v] = i0[it]; ib[v] = i1[it]; w[v] = wx[it];
    }
    // work item = a PAIR of adjacent target rows (2 jp, 2 jp + 1) of one field.  The gathers of the
    // next item are issued before the barrier of the current one (registers), so their L2 latency
    // overlaps the longitude pass and the stores.
    const int npair = (ny_t + 1) >> 1;
    const int step_f = (int)(gridDim.x / (unsigned)npair), step_p = (int)(gridDim.x % (unsigned)npair);
    int f = (int)(blockIdx.x / (unsigned)npair), jp = (int)(blockIdx.x % (unsigned)npair);
    const int i_src = tid < nx_s ? tid : nx_s - 1;              // nx_s <= blockDim: one source column per thread
    float g[4];                                                 // src values at (ja0, jb0, ja1, jb1) x i_src
    double wj0 = 0.0, wj1 = 0.0;
    auto gather = [&](int ff, int jpp) {
        const int jt0 = 2 * jpp, jt1 = min(jt0 + 1, ny_t - 1);
        const float *fld = src + (unsigned)ff * (unsigned)(ny_s * nx_s);
        const float *pm = polemean + ff * 2;
        const int jj[4] = {j0[jt0], j1[jt0], j0[jt1], j1[jt1]};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            g[k] = jj[k] >= 0 ? __ldg(fld + (unsigned)(jj[k] * nx_s + i_src)) : __ldg(pm + (-1 - jj[k]));
        wj0 = wy[jt0]; wj1 = wy[jt1];
    };
    if (f < nfield) gather(f, jp);
    int buf = 0;
    while (f < nfield) {
        double2 *row = s_row + buf * nx_s;
        {
            const double a0 = (double)g[0], a1 = (double)g[1], c0 = (double)g[2], c1 = (double)g[3];
            if (tid < nx_s) row[tid] = make_double2((a1 - a0) * wj0 + a0, (c1 - c0) * wj1 + c0);
        }
        const int fc = f, jt0 = 2 * jp;
        const bool two = jt0 + 1 < ny_t;
        f += step_f; jp += step_p;
        if (jp >= npair) { jp -= npair; ++f; }
        if (f < nfield) gather(f, jp);
        __syncthreads();
        if (owner) {
            float r0[VEC], r1[VEC];
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const double2 a = row[ia[v]], b = row[ib[v]];
                r0[v] = (float)((b.x - a.x) * w[v] + a.x);
                r1[v] = (float)((b.y - a.y) * w[v] + a.y);
            }
            float *o0 = dst + ((long long)fc * ny_t + jt0) * nx_t + tid * VEC;
            float *o1 = o0 + nx_t;
            if (VEC == 4) {
                __stcs(reinterpret_cast<float4 *>(o0), make_float4(r0[0], r0[1], r0[2], r0[3]));
                if (two) __stcs(reinterpret_cast<float4 *>(o1), make_float4(r1[0], r1[1], r1[2], r1[3]));
            } else {
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    __stcs(o0 + v, r0[v]);
                    if (two) __stcs(o1 + v, r1[v]);
                }
            }
        }
        buf ^= 1;
    }
}

// Walking variant (the production path for ERA5-sized targets): a CTA takes CHUNKS of kRegridChunk consecutive
// target rows of one field.  (1) The few source rows the chunk needs (its rows j0..j1 span ~ chunk/4 + 2 rows of
// a 1 degree source; chunks of 8 / 16 / 32 rows: 6.76 / 6.52 / 6.22 ms) are fetched ONCE with coalesced loads -- into registers while the previous chunk is being
// computed, then parked in shared memory next to two rows holding the pole means (the reference's synthetic
// pole rows, functions.py:833-842) -- instead of four scattered gathers per thread and row pair.  A small table
// per chunk turns (j0, j1, wy) of each target row into shared-memory offsets, so the latitude pass has no index
// arithmetic and no pole-row branches.  (2) Per pair of target rows the two bracketing source rows are blended
// in latitude once per source column into shared memory (functions.py:859, float64), (3) every thread produces
// VEC adjacent target longitudes of both rows (:892) and writes one 16-byte streaming store per row.  On regular
// grids the VEC targets of every thread bracket (u0,u1) for the first N1 and (u1,u2) for the rest: three
// shared-memory loads serve all of them and N1 is a template constant (checked once per launch; N1 = 0: the
// general 2 VEC loads).  The older kernels spent 35 % of their instructions on addresses and ran out of issue
// slots at 0.54 of the HBM peak; this one needs about a third of the instructions per point.
// Same expressions as regrid_kernel, hence bit-identical.  `jt_begin, jt_end`: the band of target rows this
// launch produces (dst holds only those rows): several GPUs split one variable by target latitude.
#ifndef PGW_REGRID_F64
#define PGW_REGRID_F64 0
#endif
#ifndef PGW_REGRID_CHUNK
#define PGW_REGRID_CHUNK 32
#endif
#ifndef PGW_REGRID_SR
#define PGW_REGRID_SR 10
#endif
constexpr int kRegridChunk = PGW_REGRID_CHUNK;   // target rows per chunk
constexpr int kRegridGroup = 4;        // target rows per barrier (kRegridChunk is a multiple)
constexpr int kRegridSrcRows = PGW_REGRID_SR;      // source rows a chunk may span on the staged path (32 rows of a 4:1 regridding: 8 intervals + 2)
struct __align__(16) RegridRow { int off_a, off_b; double w; };   // shared-memory offsets of the two source rows
struct __align__(16) RegridQuad { double r[kRegridGroup]; };      // one source column, blended for a group of rows

template <int VEC, int N1>
__device__ __forceinline__ void regrid_walk_body(const float *__restrict__ src, float *__restrict__ dst,
                                                 const float *__restrict__ polemean, int nfield, int ny_s, int nx_s,
                                                 int nx_t, int jt_begin, int jt_end, const int *__restrict__ j0,
                                                 const int *__restrict__ j1, const double *__restrict__ wy,
                                                 const int (&ia)[VEC], const int (&ib)[VEC], const double (&w)[VEC],
                                                 unsigned char *smem_raw) {
    const int nrow = jt_end - jt_begin, nchunk = (nrow + kRegridChunk - 1) / kRegridChunk;
    constexpr int SR = kRegridSrcRows, G = kRegridGroup;
    RegridQuad *const s_row = reinterpret_cast<RegridQuad *>(smem_raw);                 // [2][nx_s]
#if PGW_REGRID_F64
    // float64 staging: the landed rows are converted ONCE per chunk (10 conversions per thread instead of 2 per
    // target row = 64), the latitude pass reads float64
    double *const s_srcd = reinterpret_cast<double *>(s_row + 2 * nx_s);                // [SR + 2][nx_s]
    RegridRow *const s_tab = reinterpret_cast<RegridRow *>(s_srcd + (SR + 2) * nx_s);   // [2][kRegridChunk]
    float *const s_src = reinterpret_cast<float *>(s_tab + 2 * kRegridChunk);           // [SR][nx_s] landing buffer
    const int2 *const s_chunk = reinterpret_cast<const int2 *>(s_src + SR * nx_s);      // [nchunk] (jmin, span)
#else
    float *const s_src = reinterpret_cast<float *>(s_row + 2 * nx_s);                   // [2][SR + 2][nx_s]
    RegridRow *const s_tab = reinterpret_cast<RegridRow *>(s_src + 2 * (SR + 2) * nx_s);   // [2][kRegridChunk]
    const int2 *const s_chunk = reinterpret_cast<const int2 *>(s_tab + 2 * kRegridChunk);  // [nchunk] (jmin, span)
#endif
    const int tid = threadIdx.x;
    const bool owner = tid < nx_t / VEC, col = tid < nx_s;
    const int u0 = ia[0], u1 = ib[0], u2 = ib[VEC - 1];

    // items (field, chunk) are walked with stride gridDim.x; (f, c) are advanced without a division
    const int step_f = (int)(gridDim.x / (unsigned)nchunk), step_c = (int)(gridDim.x % (unsigned)nchunk);
    int f = (int)(blockIdx.x / (unsigned)nchunk), c = (int)(blockIdx.x % (unsigned)nchunk);
    // the source rows of the NEXT chunk travel global -> shared asynchronously (cp.async, no registers held)
    // into the other half of s_src while this chunk is computed
    float pm0 = 0.f, pm1 = 0.f;
    auto prefetch = [&](int ff, int cc, int b) {
        if (ff < nfield && col) {
            const int2 ch = s_chunk[cc];
            pm0 = __ldg(polemean + 2 * ff); pm1 = __ldg(polemean + 2 * ff + 1);
            if (ch.y <= SR) {
                const float *base = src + ((size_t)ff * ny_s + ch.x) * (size_t)nx_s + tid;
#if PGW_REGRID_F64
                float *d = s_src + tid;
#else
                float *d = s_src + b * (SR + 2) * nx_s + tid;
#endif
#pragma unroll
                for (int r = 0; r < SR; ++r)
                    if (r < ch.y) __pipeline_memcpy_async(d + r * nx_s, base + (size_t)r * nx_s, 4);
            }
        }
        __pipeline_commit();
    };
    int buf = 0, pb = 0;
    prefetch(f, c, 0);
    while (f < nfield) {
        const int2 ch = s_chunk[c];
        const bool staged = ch.y <= SR;
        const int r_begin = c * kRegridChunk, r_end = min(r_begin + kRegridChunk, nrow);
#if PGW_REGRID_F64
        double *const ssrc = s_srcd;
#else
        float *const ssrc = s_src + buf * (SR + 2) * nx_s;
        if (col) {
            ssrc[SR * nx_s + tid] = pm0;                 // the two pole rows
            ssrc[(SR + 1) * nx_s + tid] = pm1;
        }
#endif
        if (tid < kRegridChunk) {
            const int jt = jt_begin + min(r_begin + tid, r_end - 1);
            const int a = j0[jt], b = j1[jt];
            // staged: offsets into ssrc; not staged (a chunk spanning many source rows): offsets into the field,
            // negative = pole row
            auto off = [&](int j) { return j == -1 ? SR * nx_s : (j == -2 ? (SR + 1) * nx_s : (j - ch.x) * nx_s); };
            RegridRow t;
            t.off_a = staged ? off(a) : (a < 0 ? a : a * nx_s);
            t.off_b = staged ? off(b) : (b < 0 ? b : b * nx_s);
            t.w = wy[jt];
            s_tab[buf * kRegridChunk + tid] = t;
        }
        const float *const fld = src + (size_t)f * ny_s * (size_t)nx_s;
        float *o0 = dst + ((size_t)f * nrow + r_begin) * (size_t)nx_t + tid * VEC;
        const float pc0 = pm0, pc1 = pm1;
        f += step_f; c += step_c;                   // next item
        if (c >= nchunk) { c -= nchunk; ++f; }
        __pipeline_wait_prior(0);                   // this chunk's rows have landed (own copies; barrier: everyone's)
        __syncthreads();                            // parked rows and the row table are visible
#if PGW_REGRID_F64
        if (col) {
            if (staged) {
#pragma unroll
                for (int r = 0; r < SR; ++r)
                    if (r < ch.y) s_srcd[r * nx_s + tid] = (double)s_src[r * nx_s + tid];
            }
            s_srcd[SR * nx_s + tid] = (double)pc0;       // the two pole rows
            s_srcd[(SR + 1) * nx_s + tid] = (double)pc1;
        }
        __syncthreads();                            // float64 rows visible, landing buffer free
#endif
        prefetch(f, c, buf ^ 1);                    // in flight while this chunk is computed; the last readers of
                                                    // that half passed the barrier above
        const RegridRow *tab = s_tab + buf * kRegridChunk;
        for (int r = r_begin; r < r_end; r += G, pb ^= 1, tab += G, o0 += G * (size_t)nx_t) {
            const int nvalid = min(G, r_end - r);
            RegridQuad *const row = s_row + pb * nx_s;
            if (col) {
                RegridQuad q;
#pragma unroll
                for (int k = 0; k < G; ++k) {
                    const RegridRow t = tab[k];
                    double a, b;
                    if (staged) {
                        a = (double)ssrc[t.off_a + tid]; b = (double)ssrc[t.off_b + tid];   // (no conversion with F64 staging)
                    } else {
                        auto at = [&](int o) { return (double)(o == -1 ? pc0 : (o == -2 ? pc1 : __ldg(fld + o + tid))); };
                        a = at(t.off_a); b = at(t.off_b);
                    }
                    q.r[k] = (b - a) * t.w + a;     // latitude pass (functions.py:859)
                }
                row[tid] = q;
            }
            __syncthreads();
            if (owner) {
                // two rows at a time: the 16-byte halves of the quads (keeps the live registers of a thread low)
#pragma unroll
                for (int h = 0; h < G; h += 2) {
                    if (h < nvalid) {
                        float r0[VEC], r1[VEC];
                        if (N1 > 0) {
                            const double2 q0 = *reinterpret_cast<const double2 *>(&row[u0].r[h]);
                            const double2 q1 = *reinterpret_cast<const double2 *>(&row[u1].r[h]);
                            const double2 q2 = *reinterpret_cast<const double2 *>(&row[u2].r[h]);
#pragma unroll
                            for (int v = 0; v < VEC; ++v) {
                                const double2 a = v < N1 ? q0 : q1, b = v < N1 ? q1 : q2;
                                r0[v] = (float)((b.x - a.x) * w[v] + a.x);      // longitude pass (:892)
                                r1[v] = (float)((b.y - a.y) * w[v] + a.y);
                            }
                        } else {
#pragma unroll
                            for (int v = 0; v < VEC; ++v) {
                                const double2 a = *reinterpret_cast<const double2 *>(&row[ia[v]].r[h]);
                                const double2 b = *reinterpret_cast<const double2 *>(&row[ib[v]].r[h]);
                                r0[v] = (float)((b.x - a.x) * w[v] + a.x);
                                r1[v] = (float)((b.y - a.y) * w[v] + a.y);
                            }
                        }
                        float *oa = o0 + (size_t)h * nx_t, *ob = oa + nx_t;
                        const bool two = h + 1 < nvalid;
                        if (VEC == 4) {
                            __stcs(reinterpret_cast<float4 *>(oa), make_float4(r0[0], r0[1], r0[2], r0[3]));
                            if (two) __stcs(reinterpret_cast<float4 *>(ob), make_float4(r1[0], r1[1], r1[2], r1[3]));
                        } else {
#pragma unroll
                            for (int v = 0; v < VEC; ++v) {
                                __stcs(oa + v, r0[v]);
                                if (two) __stcs(ob + v, r1[v]);
                            }
                        }
                    }
                }
            }
        }
        buf ^= 1;
    }
}

// the general path (any tables) out of line: its register needs must not shape the allocation of the hot bodies
template <int VEC>
__device__ __noinline__ void regrid_walk_general(const float *__restrict__ src, float *__restrict__ dst,
                                                 const float *__restrict__ polemean, int nfield, int ny_s, int nx_s,
                                                 int nx_t, int jt_begin, int jt_end, const int *__restrict__ j0,
                                                 const int *__restrict__ j1, const double *__restrict__ wy,
                                                 const int *__restrict__ i0, const int *__restrict__ i1,
                                                 const double *__restrict__ wx, unsigned char *smem_raw) {
    int ia[VEC], ib[VEC];
    double w[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        const int it = threadIdx.x < nx_t / VEC ? threadIdx.x * VEC + v : 0;
        ia[v] = i0[it]; ib[v] = i1[it]; w[v] = wx[it];
    }
    regrid_walk_body<VEC, 0>(src, dst, polemean, nfield, ny_s, nx_s, nx_t, jt_begin, jt_end, j0, j1, wy, ia, ib, w, smem_raw);
}

#ifndef PGW_REGRID_MINB
#define PGW_REGRID_MINB 3
#endif
template <int VEC>
__global__ void __launch_bounds__(384, PGW_REGRID_MINB)
regrid_walk_kernel(const float *__restrict__ src, float *__restrict__ dst, const float *__restrict__ polemean,
                   int nfield, int ny_s, int nx_s, int nx_t, int jt_begin, int jt_end,
                   const int *__restrict__ j0, const int *__restrict__ j1, const double *__restrict__ wy,
                   const int *__restrict__ i0, const int *__restrict__ i1, const double *__restrict__ wx) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int nrow = jt_end - jt_begin, nchunk = (nrow + kRegridChunk - 1) / kRegridChunk;
#if PGW_REGRID_F64
    int2 *const s_chunk = reinterpret_cast<int2 *>(smem_raw + sizeof(RegridQuad) * 2 * nx_s +
                                                   sizeof(double) * (kRegridSrcRows + 2) * nx_s +
                                                   sizeof(RegridRow) * 2 * kRegridChunk +
                                                   sizeof(float) * kRegridSrcRows * nx_s);
#else
    int2 *const s_chunk = reinterpret_cast<int2 *>(smem_raw + sizeof(RegridQuad) * 2 * nx_s +
                                                   sizeof(float) * 2 * (kRegridSrcRows + 2) * nx_s +
                                                   sizeof(RegridRow) * 2 * kRegridChunk);
#endif
    const int tid = threadIdx.x;
    const bool owner = tid < nx_t / VEC;
    // ---- per launch: span of source rows of every chunk; longitude brackets of this thread
    for (int c = tid; c < nchunk; c += blockDim.x) {
        int lo = INT_MAX, hi = -1;
        for (int r = 0; r < kRegridChunk; ++r) {
            const int jt = jt_begin + c * kRegridChunk + r;
            if (jt >= jt_end) break;
            const int a = j0[jt], b = j1[jt];
            if (a >= 0) { lo = min(lo, a); hi = max(hi, a); }
            if (b >= 0) { lo = min(lo, b); hi = max(hi, b); }
        }
        s_chunk[c] = hi < 0 ? make_int2(0, 0) : make_int2(lo, hi - lo + 1);
    }
    int ia[VEC], ib[VEC];
    double w[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        const int it = owner ? tid * VEC + v : 0;
        ia[v] = i0[it]; ib[v] = i1[it]; w[v] = wx[it];
    }
    // three-column pattern: the first n1 targets bracket (u0, u1), the rest (u1, u2); n1 the same for all threads
    const int u0 = ia[0], u1 = ib[0], u2 = ib[VEC - 1];
    int n1 = 0;
    bool pat = true;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        const bool first = ia[v] == u0 && ib[v] == u1, second = ia[v] == u1 && ib[v] == u2;
        if (first && n1 == v) n1 = v + 1;
        else if (!second) pat = false;
    }
    __shared__ int s_n1;
    if (tid == 0) s_n1 = n1;
    __syncthreads();                                // also publishes s_chunk
    const int n1_all = s_n1;
    const bool uniform = __syncthreads_and((pat && n1 == n1_all) || !owner) != 0;
#define PGW_WALK(N) regrid_walk_body<VEC, N>(src, dst, polemean, nfield, ny_s, nx_s, nx_t, jt_begin, jt_end, j0, j1, wy, \
                                             ia, ib, w, smem_raw)
    if (uniform && VEC == 4) {
        switch (n1_all) {
            case 1: PGW_WALK(1); return;
            case 2: PGW_WALK(2); return;
            case 3: PGW_WALK(3); return;
            case 4: PGW_WALK(4); return;
            default: break;
        }
    }
    regrid_walk_general<VEC>(src, dst, polemean, nfield, ny_s, nx_s, nx_t, jt_begin, jt_end, j0, j1, wy, i0, i1, wx, smem_raw);
#undef PGW_WALK
}

// One delta stamp of ta, hur, ua, va from the GCM grid straight into the column kernel's node layout: dst is
// float4 [K][jt_end - jt_begin][nx_t] = {ta, hur, ua, va}, what regrid_walk_kernel on each variable followed by
// pack_d4_kernel writes.  A CTA takes one (level, target row) at a time: (1) the four variables' two bracketing
// source rows are blended in latitude once per source column into shared memory (float64, functions.py:859),
// (2) every thread produces target longitudes from that row (:892) and writes one 16-byte streaming store per
// column.  Same expressions as regrid_kernel, hence bit-identical; the ~22 MB source of a stamp sits in L2, so
// the kernel is bound by the store of the stamp, which it writes once instead of three times.
constexpr int kRegridPackThreads = 256;

__global__ void __launch_bounds__(kRegridPackThreads)
regrid_pack_d4_kernel(const float *__restrict__ src, float4 *__restrict__ dst, const float *__restrict__ polemean,
                      int nlev, int ny_s, int nx_s, int nx_t, int jt_begin, int jt_end, const int *__restrict__ j0,
                      const int *__restrict__ j1, const double *__restrict__ wy, const int *__restrict__ i0,
                      const int *__restrict__ i1, const double *__restrict__ wx) {
    extern __shared__ double s_lat[];               // [4 variables][nx_s]: the row blended in latitude
    const int nrow = jt_end - jt_begin;
    const long long nitem = (long long)nlev * nrow;
    const size_t var_stride = (size_t)nlev * ny_s * nx_s;
    for (long long item = blockIdx.x; item < nitem; item += gridDim.x) {
        const int k = (int)(item / nrow), r = (int)(item % nrow), jt = jt_begin + r;
        const int ja = j0[jt], jb = j1[jt];
        const double wj = wy[jt];
        __syncthreads();                            // the previous item's longitude pass is done with s_lat
        for (int idx = threadIdx.x; idx < 4 * nx_s; idx += blockDim.x) {
            const int v = idx / nx_s, i = idx - v * nx_s;
            const float *fld = src + v * var_stride + (size_t)k * ny_s * nx_s;
            const float *pm = polemean + 2 * ((long long)v * nlev + k);
            const double a0 = src_at(fld, pm, ja, i, nx_s), a1 = src_at(fld, pm, jb, i, nx_s);
            s_lat[idx] = (a1 - a0) * wj + a0;       // latitude pass (functions.py:859)
        }
        __syncthreads();
        float4 *o = dst + ((size_t)k * nrow + r) * (size_t)nx_t;
        for (int it = threadIdx.x; it < nx_t; it += blockDim.x) {
            const int ia = __ldg(i0 + it), ib = __ldg(i1 + it);
            const double w = __ldg(wx + it);
            float res[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const double a = s_lat[v * nx_s + ia], b = s_lat[v * nx_s + ib];
                res[v] = (float)((b - a) * w + a);  // longitude pass (:892)
            }
            __stcs(o + it, make_float4(res[0], res[1], res[2], res[3]));
        }
    }
}

// harmonic_ac_analysis (functions.py:678-740): mean + harmonics 1..3 of an
// nt-long series per grid point.  One thread per grid point, lanes = adjacent
// points; cos/sin tables for the three harmonics are staged in shared memory.
#ifndef PGW_SMOOTH_ONLY
#define PGW_SMOOTH_ONLY 0     // experiments: 1 = read pass only, 2 = write pass only
#endif
#ifndef PGW_SMOOTH_BATCH
#define PGW_SMOOTH_BATCH 8
#endif
#ifndef PGW_SMOOTH_THREADS
#define PGW_SMOOTH_THREADS 128
#endif
#ifndef PGW_SMOOTH_CAP
#define PGW_SMOOTH_CAP 8
#endif
#ifndef PGW_SMOOTH_RING
#define PGW_SMOOTH_RING 16
#endif
constexpr int kSmoothBatch = PGW_SMOOTH_BATCH, kSmoothThreads = PGW_SMOOTH_THREADS;
constexpr int kSmoothRing = PGW_SMOOTH_RING;      // stamps in flight per thread (a multiple of kSmoothBatch)

__global__ void __launch_bounds__(kSmoothThreads)
smooth_kernel(const float *__restrict__ series, float *__restrict__ out, int nt, long long npoint) {
    extern __shared__ double tab[];                 // [nt][6]: cos1 sin1 cos2 sin2 cos3 sin3 | float ring
    float *const ring = reinterpret_cast<float *>(tab + (size_t)nt * 6);   // [kSmoothRing][kSmoothThreads]
    for (int t = threadIdx.x; t < nt; t += blockDim.x) {
        for (int k = 1; k <= 3; ++k) {
            const double br = 2. * 3.141592653589793 * k / (double)nt * (double)(t + 1);   // :726
            tab[t * 6 + 2 * (k - 1)] = cos(br);
            tab[t * 6 + 2 * (k - 1) + 1] = sin(br);
        }
    }
    __syncthreads();
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < npoint;
         p += (long long)gridDim.x * blockDim.x) {
        double sum = 0.0, a1 = 0, b1 = 0, a2 = 0, b2 = 0, a3 = 0, b3 = 0;
        bool bad = false;
        auto acc = [&](float xf, int t) {
            bad |= isnan(xf);
            const double x = (double)xf;
            const double *tb = tab + t * 6;
            sum += x;
            a1 = fma(x, tb[0], a1); b1 = fma(x, tb[1], b1);
            a2 = fma(x, tb[2], a2); b2 = fma(x, tb[3], b2);
            a3 = fma(x, tb[4], a3); b3 = fma(x, tb[5], b3);
        };
        // The series travels global -> shared memory with cp.async, kSmoothRing stamps ahead, in groups of
        // kSmoothBatch (every thread copies and later reads only its own column of the ring: no barrier).  With plain
        // loads the compiler kept 4 of them in flight per thread and the read pass waited on DRAM latency (half of all
        // stall samples at the first use of a load; read pass alone 0.58 ms for 1.8 GB); the ring holds
        // 4 x kSmoothRing bytes per thread in flight without a register (rings of 16 / 32 / 64 stamps: 0.956 / 1.03 /
        // 0.98 ms against 1.006 with plain loads: the latency is NOT what bounds the kernel, see DESIGN.md 3.3).
        // Same order of summation as before.
        const float *sp = series + p;
        float *const rg = ring + threadIdx.x;
        constexpr int G = kSmoothBatch, NG = kSmoothRing / kSmoothBatch;
        const int ngroups = nt / G;                                  // whole groups; the rest is read directly
        auto issue = [&](int g, int zero) {
            if (g < ngroups) {
                float *d = rg + (g % NG) * G * kSmoothThreads + zero;
#pragma unroll
                for (int k = 0; k < G; ++k)
                    __pipeline_memcpy_async(d + k * kSmoothThreads, sp + (long long)(g * G + k) * npoint, 4);
            }
            __pipeline_commit();
        };
#pragma unroll
        for (int g = 0; g < NG; ++g) issue(g, 0);
        for (int g = 0; g < ngroups; ++g) {
            __pipeline_wait_prior(NG - 1);                           // group g has landed
            const float *d = rg + (g % NG) * G * kSmoothThreads;
            float xv[G];
#pragma unroll
            for (int k = 0; k < G; ++k) xv[k] = d[k * kSmoothThreads];
            // refill the slot just read; `zero` (== 0) depends on the values read, so the copies cannot overtake the reads
            int bits = 0;
#pragma unroll
            for (int k = 0; k < G; ++k) bits |= __float_as_int(xv[k]);
            int zero;
            asm volatile("and.b32 %0, %1, 0;" : "=r"(zero) : "r"(bits));
            issue(g + NG, zero);
#pragma unroll
            for (int k = 0; k < G; ++k) acc(xv[k], g * G + k);
        }
        __pipeline_wait_prior(0);
        int t = ngroups * G;
        for (; t < nt; ++t) acc(__ldcs(sp + (long long)t * npoint), t);
        const double sc = 2. / (double)nt;
        const double mean = sum / (double)nt;
        a1 *= sc; b1 *= sc; a2 *= sc; b2 *= sc; a3 *= sc; b3 *= sc;
#if PGW_SMOOTH_ONLY == 1
        if (a1 + b1 + a2 + b2 + a3 + b3 + mean == 1.2345) out[p] = 0.f;            // (experiment: no write pass)
        else continue;
#endif
        for (t = 0; t < nt; ++t) {
            const double *tb = tab + t * 6;
            // sum(hcts[0:3]) + mean, functions.py:739 (python sum starts at 0)
            const double h = ((0.0 + (a1 * tb[0] + b1 * tb[1])) + (a2 * tb[2] + b2 * tb[3])) +
                             (a3 * tb[4] + b3 * tb[5]);
            __stcs(out + (long long)t * npoint + p, bad ? NAN : (float)(h + mean));
        }
    }
}

}  // namespace pgw

using namespace pgw;

extern "C" {

int pgw_zonal_mean_f32(const float *src, float *polemean, long long nfield, int ny_s, int nx_s, void *stream) {
    if (!src || !polemean || nfield <= 0 || ny_s < 1 || nx_s < 1) return PGW_E_INVALID;
    if (nfield > 2147483647LL) return PGW_E_INVALID;
    zonal_mean_kernel<<<dim3((unsigned)nfield, 2), 128, 0, (cudaStream_t)stream>>>(src, polemean, nfield, ny_s, nx_s);
    return pgw_check_launch("zonal_mean_kernel");
}

int pgw_regrid_bilinear_band_f32(const float *src, float *dst, const float *polemean, long long nfield, int ny_s,
                                 int nx_s, int ny_t, int nx_t, int jt_begin, int jt_end, const int *j0, const int *j1,
                                 const double *wy, const int *i0, const int *i1, const double *wx, void *stream) {
    if (!src || !dst || !polemean || !j0 || !j1 || !wy || !i0 || !i1 || !wx) return PGW_E_INVALID;
    if (nfield <= 0 || ny_s < 1 || nx_s < 1 || ny_t < 1 || nx_t < 1) return PGW_E_INVALID;
    if (jt_begin < 0 || jt_end > ny_t || jt_begin >= jt_end) return PGW_E_INVALID;
    const int nrow = jt_end - jt_begin;
    const bool vec = (nx_t % 4 == 0) && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
    const int nchunk = (nrow + kRegridChunk - 1) / kRegridChunk;
    const char *force = getenv("PGW_REGRID_PATH");          // "rows" / "generic": the older kernels (A/B runs, tests)
    const bool walk_ok = (vec ? nx_t / 4 : nx_t) <= 384 && nx_s <= 384 && nfield * (long long)nchunk < (1LL << 31) &&
                         nchunk <= 4096 && !(force && (!strcmp(force, "rows") || !strcmp(force, "generic")));
    if (walk_ok) {
#if PGW_REGRID_F64
        const size_t smem = sizeof(RegridQuad) * 2 * (size_t)nx_s + sizeof(RegridRow) * 2 * kRegridChunk +
                            sizeof(double) * (kRegridSrcRows + 2) * (size_t)nx_s +
                            sizeof(float) * kRegridSrcRows * (size_t)nx_s + sizeof(int2) * (size_t)nchunk;
#else
        const size_t smem = sizeof(RegridQuad) * 2 * (size_t)nx_s + sizeof(RegridRow) * 2 * kRegridChunk +
                            sizeof(float) * 2 * (kRegridSrcRows + 2) * (size_t)nx_s + sizeof(int2) * (size_t)nchunk;
#endif
        const long long nitem = nfield * (long long)nchunk;
        long long g = nitem < 148LL * 5 ? nitem : 148LL * 5;
        if (smem > 48 * 1024) {
            int rc;
            if ((rc = pgw_ensure_smem(vec ? (const void *)regrid_walk_kernel<4> : (const void *)regrid_walk_kernel<1>,
                                      vec ? 12 : 13, smem, 0)) != PGW_OK) return rc;
        }
        if (vec)
            regrid_walk_kernel<4><<<(unsigned)g, 384, smem, (cudaStream_t)stream>>>(
                src, dst, polemean, (int)nfield, ny_s, nx_s, nx_t, jt_begin, jt_end, j0, j1, wy, i0, i1, wx);
        else
            regrid_walk_kernel<1><<<(unsigned)g, 384, smem, (cudaStream_t)stream>>>(
                src, dst, polemean, (int)nfield, ny_s, nx_s, nx_t, jt_begin, jt_end, j0, j1, wy, i0, i1, wx);
        return pgw_check_launch("regrid_walk_kernel");
    }
    // the older kernels take whole grids only: shift the row tables and the destination
    if (jt_begin != 0 || jt_end != ny_t)
        return pgw_regrid_bilinear_f32(src, dst, polemean, nfield, ny_s, nx_s, nrow, nx_t, j0 + jt_begin, j1 + jt_begin,
                                       wy + jt_begin, i0, i1, wx, stream);
    return pgw_regrid_bilinear_f32(src, dst, polemean, nfield, ny_s, nx_s, ny_t, nx_t, j0, j1, wy, i0, i1, wx, stream);
}

int pgw_regrid_bilinear_f32(const float *src, float *dst, const float *polemean, long long nfield, int ny_s,
                            int nx_s, int ny_t, int nx_t, const int *j0, const int *j1, const double *wy,
                            const int *i0, const int *i1, const double *wx, void *stream) {
    if (!src || !dst || !polemean || !j0 || !j1 || !wy || !i0 || !i1 || !wx) return PGW_E_INVALID;
    if (nfield <= 0 || ny_s < 1 || nx_s < 1 || ny_t < 1 || nx_t < 1) return PGW_E_INVALID;
    const bool vec = (nx_t % 4 == 0) && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
    const char *force = getenv("PGW_REGRID_PATH");
    if (!(force && (!strcmp(force, "rows") || !strcmp(force, "generic"))) && (vec ? nx_t / 4 : nx_t) <= 384 &&
        nx_s <= 384 && (ny_t + kRegridChunk - 1) / kRegridChunk <= 4096)
        return pgw_regrid_bilinear_band_f32(src, dst, polemean, nfield, ny_s, nx_s, ny_t, nx_t, 0, ny_t, j0, j1, wy, i0,
                                            i1, wx, stream);
    if (!(force && !strcmp(force, "generic")) &&
        (vec ? nx_t / 4 : nx_t) <= 384 && nx_s <= 384 && nfield * ny_s * (long long)nx_s < (1LL << 31)) {
        const long long nitem = nfield * (long long)((ny_t + 1) / 2);
        long long g = nitem < 148LL * 5 ? nitem : 148LL * 5;
        const size_t smem = sizeof(double) * 4 * (size_t)nx_s;
        if (vec)
            regrid_rows_kernel<4><<<(unsigned)g, 384, smem, (cudaStream_t)stream>>>(
                src, dst, polemean, (int)nfield, ny_s, nx_s, ny_t, nx_t, j0, j1, wy, i0, i1, wx);
        else
            regrid_rows_kernel<1><<<(unsigned)g, 384, smem, (cudaStream_t)stream>>>(
                src, dst, polemean, (int)nfield, ny_s, nx_s, ny_t, nx_t, j0, j1, wy, i0, i1, wx);
        return pgw_check_launch("regrid_rows_kernel");
    }
    const long long total = nfield * ny_t * (long long)(vec ? nx_t / 4 : nx_t);
    long long g = (total + 255) / 256;
    const long long cap = 148LL * 32;
    if (g > cap) g = cap;
    if (vec)
        regrid_kernel<4><<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(src, dst, polemean, nfield, ny_s, nx_s,
                                                                         ny_t, nx_t, j0, j1, wy, i0, i1, wx);
    else
        regrid_kernel<1><<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(src, dst, polemean, nfield, ny_s, nx_s,
                                                                         ny_t, nx_t, j0, j1, wy, i0, i1, wx);
    return pgw_check_launch("regrid_kernel");
}

int pgw_regrid_pack_d4_f32(const float *src, float *dst, const float *polemean, int nlev, int ny_s, int nx_s,
                           int ny_t, int nx_t, int jt_begin, int jt_end, const int *j0, const int *j1,
                           const double *wy, const int *i0, const int *i1, const double *wx, float *scratch,
                           void *stream) {
    if (!src || !dst || !polemean || !j0 || !j1 || !wy || !i0 || !i1 || !wx) return PGW_E_INVALID;
    if (nlev < 1 || ny_s < 1 || nx_s < 1 || ny_t < 1 || nx_t < 1) return PGW_E_INVALID;
    if (jt_begin < 0 || jt_end > ny_t || jt_begin >= jt_end) return PGW_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(dst) & 15u) != 0) return PGW_E_INVALID;
    const int nrow = jt_end - jt_begin;
    if (nx_s <= PGW_REGRID_PACK_MAX_NX_S) {
        const size_t smem = sizeof(double) * 4 * (size_t)nx_s;          // <= 48 KB: no opt-in
        const long long nitem = (long long)nlev * nrow;
        const long long g = nitem < 148LL * 8 ? nitem : 148LL * 8;
        regrid_pack_d4_kernel<<<(unsigned)g, kRegridPackThreads, smem, (cudaStream_t)stream>>>(
            src, reinterpret_cast<float4 *>(dst), polemean, nlev, ny_s, nx_s, nx_t, jt_begin, jt_end, j0, j1, wy, i0,
            i1, wx);
        return pgw_check_launch("regrid_pack_d4_kernel");
    }
    // wider source rows: each variable regridded into the scratch, then packed (the same expressions)
    if (!scratch || (reinterpret_cast<uintptr_t>(scratch) & 15u) != 0) return PGW_E_INVALID;
    const long long n = (long long)nlev * nrow * nx_t, piece = (n + 3) / 4 * 4;
    const long long field = (long long)ny_s * nx_s;
    int rc;
    for (int v = 0; v < 4; ++v)
        if ((rc = pgw_regrid_bilinear_band_f32(src + v * nlev * field, scratch + v * piece, polemean + 2LL * v * nlev,
                                               nlev, ny_s, nx_s, ny_t, nx_t, jt_begin, jt_end, j0, j1, wy, i0, i1, wx,
                                               stream)) != PGW_OK)
            return rc;
    return pgw_pack_d4_f32(scratch, scratch + piece, scratch + 2 * piece, scratch + 3 * piece, dst, n, 0, stream);
}

int pgw_smooth_harmonic_f32(const float *series, float *out, int nt, long long npoint, void *stream) {
    if (!series || !out || nt < 8 || npoint <= 0) return PGW_E_INVALID;     // i < floor(nt/2) for i=1..3
    const size_t smem = sizeof(double) * 6 * (size_t)nt + sizeof(float) * kSmoothRing * kSmoothThreads;
    if (smem > 200 * 1024) return PGW_E_SMEM;
    if (smem > 48 * 1024) {
        int rc;
        if ((rc = pgw_ensure_smem((const void *)smooth_kernel, 14, smem, 0)) != PGW_OK) return rc;
    }
    long long g = (npoint + kSmoothThreads - 1) / kSmoothThreads;
    const long long cap = 148LL * PGW_SMOOTH_CAP;
    if (g > cap) g = cap;
    smooth_kernel<<<(unsigned)g, kSmoothThreads, smem, (cudaStream_t)stream>>>(series, out, nt, npoint);
    return pgw_check_launch("smooth_kernel");
}

}  // extern "C"
