// ensemble_kernel.cuh -- season-resident path for small grids (the 100 km calibration ensemble).
//
// One thread-block CLUSTER (2..8 CTAs) owns one ensemble member for the whole season; each CTA holds a strip of
// rows (strips are cut by the host so that their work balances).  Everything a member needs stays on chip for all
// T-1 days, and HBM only ever sees the output planes, written once, as large contiguous TMA bulk stores:
//   * ten output planes of the strip live in shared memory IN THE OUTPUT LAYOUT (rows x nx doubles, contiguous):
//     h0, h1 (also the state the stencils read), density, snowAdv, snowDiv, snowLead, snowAtm, snowWindPackLoss/
//     Gain/Net (also the running accumulators).  Measured on B200 (tools/micro): fragmented per-thread stores of
//     this pattern reach 1.6 TB/s, full-row st.global 4.4 TB/s, bulk stores 5.8 TB/s;
//   * every compute thread OWNS the same few cells for the whole season (KR raw-dynamics entries, KO ocean cells),
//     so all shared-memory addresses are computed once, before the first day; a day is straight-line fp64 code;
//   * the two boundary rows of each neighbour strip are pushed into halo rows through distributed shared memory
//     (st.shared::cluster); two split (arrive ... wait) cluster barriers per day order "I have read my halo" and
//     "my pushes have landed", so the halo is single-buffered and nobody ever waits at a barrier it just reached;
//   * a dedicated DMA warp issues every HBM write: ten cp.async.bulk shared->global per day for the planes, and
//     the member-independent snowAcc/snowOcean planes as bulk global->shared->global copies of the pre-pass sums.
// The land mask is compiled into per-strip cell lists once per context: only ocean cells are owned and advanced;
// only cells with an ocean cell in their 3x3 neighbourhood get raw advection/divergence; land cells (56 % of the
// 100 km grid) have closed-form outputs after the first step -- h and density NaN, every accumulator NaN if its
// switch is on and 0 otherwise (NaN + anything = NaN, x + 0 = x) -- so their plane entries are written twice per
// season and then simply ride along in every bulk store.
// The member-independent forcing is pre-digested once per season by two small kernels (drift gradients;
// snowfall -> accumulation/ocean flux and their running sums) and then shared by every member through L2.
//
// Arithmetic is the per-cell code of cell_math.cuh, shared with the general path: results are value-identical.
// The loops use only the bare three-operation constant divisions (cell_math.cuh div_const_bare): their operand
// range is guaranteed by guarding the INPUTS -- every depth the kernel publishes and every drift term of the
// pre-pass must be zero, NaN or within [2^-150, 2^150] (out_of_guard).  If anything ever leaves that guard (never,
// on physical data) EnsArgs::status is raised and the host discards the season and reruns it with the general
// per-day kernels, which carry the full IEEE division paths.
#pragma once
#include <cooperative_groups.h>

#include <type_traits>

#include "cell_math.cuh"
#include "day_kernels.cuh"

namespace nesosim {

namespace cg = cooperative_groups;

// ------------------------------------------------------------------ member-independent pre-pass (per season)
// DA[x][cell][2] = (ut, vt), (gx(ut), gy(vt))   drift displacement and its gradients   (NESOSIM.py:204-205)
// DB[x][cell]    = (acc, 1-C)                   accumulation delta (NESOSIM.py:260-263), open-water fraction
// cumAcc[x][cell], cumOc[x][cell] = snowAcc[x+1], snowOcean[x+1]   running sums (NESOSIM.py:264,268)

struct DeriveArgs {
    int ny, nx, steps, T, sets;        // steps = T-1; `sets` independent forcing sets [set][T][...] (1 = plain season)
    const double *P, *C, *UV;          // [T][plane], [T][plane], [T][2][plane]
    double2 *DA;                       // [steps][plane][2]
    double2 *DB;                       // [steps][plane]
    double *cumAcc, *cumOc;            // [steps][plane] each
    ModelConsts k;
    GradConsts g;
    ConstDiv rho_new;
    int *status;                       // raised when a drift term leaves the season kernel's operand guard
};

__global__ void derive_pointwise_kernel(const __grid_constant__ DeriveArgs a) {
    const int gx = blockIdx.x * blockDim.x + threadIdx.x;
    const int gy = blockIdx.y * blockDim.y + threadIdx.y;
    const int set = blockIdx.z / a.steps, x = blockIdx.z - set * a.steps;
    if (gx >= a.nx || gy >= a.ny) return;
    const long long plane = (long long)a.ny * a.nx, o = (long long)gy * a.nx + gx;
    const long long fin = ((long long)set * a.T + x) * plane;       // this day in the [set][T] forcing stacks
    const long long fout = ((long long)set * a.steps + x) * plane;  // ... and in the [set][steps] derived stacks
    const double *U = a.UV + fin * 2, *V = U + plane;
    const int xm = max(gx - 1, 0), xp = min(gx + 1, a.nx - 1), ym = max(gy - 1, 0), yp = min(gy + 1, a.ny - 1);
    auto ut = [&](int r, int c) { return mul(U[(long long)r * a.nx + c], a.k.deltaT); };
    auto vt = [&](int r, int c) { return mul(V[(long long)r * a.nx + c], a.k.deltaT); };
    const double utc = ut(gy, gx), vtc = vt(gy, gx);
    double2 *da = a.DA + (fout + o) * 2;
    const double gxu = gradient1d(ut(gy, xm), utc, ut(gy, xp), gx, a.nx, a.g);
    const double gyv = gradient1d(vt(ym, gx), vtc, vt(yp, gx), gy, a.ny, a.g);
    da[0] = make_double2(utc, vtc);
    da[1] = make_double2(gxu, gyv);
    if (out_of_guard(utc) | out_of_guard(vtc) | out_of_guard(gxu) | out_of_guard(gyv)) atomicOr(a.status, 1);
    const double C = a.C[fin + o];
    const double pd = div_const(a.P[fin + o], a.rho_new);
    const double omc = sub(1.0, C);
    a.DB[fout + o] = make_double2(mul(pd, C), omc);
    a.cumOc[fout + o] = -mul(pd, omc);   // parks oc until the scan
}

// One thread per cell, sequential in time, loads batched 8 days ahead (add-latency bound, not load-latency bound).
__global__ void derive_scan_kernel(const double2 *DB, double *cumAcc, double *cumOc, long long plane, int steps, int sets) {
    long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= plane * sets) return;
    {   // one thread per (set, cell): move to the set's stack
        const long long set = o / plane;
        o -= set * plane;
        DB += set * steps * plane;
        cumAcc += set * steps * plane;
        cumOc += set * steps * plane;
    }
    double sa = 0.0, so = 0.0;
    constexpr int B = 8;
    for (int x0 = 0; x0 < steps; x0 += B) {
        double da[B], dq[B];
#pragma unroll
        for (int j = 0; j < B; ++j) {
            const int x = min(x0 + j, steps - 1);
            da[j] = DB[(long long)x * plane + o].x;
            dq[j] = cumOc[(long long)x * plane + o];
        }
#pragma unroll
        for (int j = 0; j < B; ++j) {
            if (x0 + j < steps) {
                sa = add(sa, da[j]);
                so = add(so, dq[j]);
                cumAcc[(long long)(x0 + j) * plane + o] = sa;
                cumOc[(long long)(x0 + j) * plane + o] = so;
            }
        }
    }
}

// ------------------------------------------------------------------------------------ the season kernel

constexpr int ENS_MAX_CLUSTER = 8;
constexpr int ENS_SXR = 98;            // raw tile row stride (double2); column c lives at c+1 (zero pad each side)
constexpr int ENS_MAX_NX = 96;
constexpr int ENS_NPLANE = 10;         // staged output planes: h0, h1, density, adv, div, lead, atm, wpl, wpg, wp
constexpr int ENS_MIN_ROWS = 4;        // a strip's top two and bottom two rows must be distinct rows
constexpr int ENS_NTIMER = 64;           // [0..7] thread 0 phases, [8..15] DMA lane, [16..39] per-warp A, [40..63] per-warp B
constexpr int PF_DAYS = 3;               // forcing is pulled into L2 this many days ahead of its use

// plane index -> output variable
__device__ __constant__ const int ENS_PLANE_VAR[ENS_NPLANE] = {V_H0, V_H1, V_DENS, V_ADV, V_DIV, V_LEAD, V_ATM, V_WPL, V_WPG, V_WP};
enum { PL_H0 = 0, PL_H1, PL_DENS, PL_ADV, PL_DIV, PL_LEAD, PL_ATM, PL_WPL, PL_WPG, PL_WP };
enum { BAR_A = 1, BAR_DRAIN = 2, BAR_STORE = 3 };   // named CTA barriers (0 is __syncthreads)

// Shared memory of one CTA, sized by the host for the tallest strip (`rows`).  Byte offsets from the base:
//   h0 ext   [2 halo rows above][own rows][2 halo rows below]   (rows+4)*nx = PEX doubles; the rows below follow
//            the strip's own last row directly, so the rows r-1 / r+1 of ANY h cell are exactly -+nx doubles away
//   h1 ext   same, so layer 1 of ANY h cell sits exactly PEX doubles after layer 0
//   planes 2..9 [PE] each (own cells only)
//   staging  [2][PE]    snowAcc / snowOcean rows on their way global -> shared -> global (TMA only)
//   raw adv  [(rows+2)*SXR + 1] double2,  raw div likewise (the +1 is the slot idle list entries write to)
//   member coefficients [10], land codes (uint16), five mbarriers (staging loads, halo pushes, planes drained, and one
//   "done reading" barrier per neighbour)
struct EnsLayout {
    int PE, PEX;                       // doubles
    unsigned off_stage, off_adv, tile_bytes, off_coef, off_codes, off_mbar, total;   // bytes
    // planes 0,1: offset of the extended plane (own cell (lr,c) at +((lr+2)*nx+c)*8); planes 2..9: own cells
    __host__ __device__ unsigned plane_off(int p) const {
        return (unsigned)((p < 2 ? (long long)p * PEX : 2ll * PEX + (long long)(p - 2) * PE) * 8);
    }
};
__host__ __device__ inline EnsLayout ens_layout(int rows, int nx, int land_alloc) {
    EnsLayout L;
    L.PE = (rows * nx + 1) / 2 * 2;
    L.PEX = (rows + 4) * nx + ((rows * nx) & 1);
    L.off_stage = (unsigned)((2ll * L.PEX + 8ll * L.PE) * 8);
    L.off_adv = L.off_stage + (unsigned)(2 * L.PE * 8);
    L.tile_bytes = (unsigned)(((rows + 2) * ENS_SXR + 1) * 16);
    L.off_coef = L.off_adv + 2 * L.tile_bytes;
    L.off_codes = L.off_coef + (10 + 64) * 8;   // 10 coefficient products + 64 doubles of reduction scratch (misfit mode)
    L.off_mbar = (L.off_codes + (unsigned)land_alloc * 2u + 15u) / 16u * 16u;
    // [0] staging loads, [8] halo pushes, [16] the strip ABOVE has finished reading its halo, [24] planes drained,
    // [32] the strip BELOW has finished reading its halo
    L.total = L.off_mbar + 48;
    return L;
}

// Per-strip cell lists (uint16 code = row*128 + col; row is global for the raw list, strip-local for cells).
struct StripTables {
    const unsigned short *codes;       // all lists concatenated (device)
    int cluster;                       // CTAs per member
    int row0[ENS_MAX_CLUSTER + 1];     // strip k owns rows row0[k] .. row0[k+1]-1
    int raw_off[ENS_MAX_CLUSTER], raw_int_n[ENS_MAX_CLUSTER], raw_n[ENS_MAX_CLUSTER];   // interior entries first
    int ocean_off[ENS_MAX_CLUSTER], ocean_n[ENS_MAX_CLUSTER];
    int land_off[ENS_MAX_CLUSTER], land_n[ENS_MAX_CLUSTER];
    int hland_off[ENS_MAX_CLUSTER], hland_n[ENS_MAX_CLUSTER];   // land cells of the strip's four halo rows (ext row*128+col)
    int halo_tx[ENS_MAX_CLUSTER];      // bytes the neighbours push into the strip's halo rows per day (16 per ocean cell)
    int rows_alloc;                    // tallest strip
    int raw_max, ocean_max, land_alloc;   // longest lists
};

struct EnsArgs {
    int ny, nx, T, M;
    const double2 *DA, *DB;
    const double *cumAcc, *cumOc;
    const double *W;                   // wind [T][plane]
    const double *ic;                  // NULL -> zero depth
    long long ic_stride;               // 0 shared, plane per member
    const double *conc0;
    // forcing sets (multi-season batches): member m uses set member_set[m] of `sets` stacked seasons and runs
    // set_steps[set] steps; NULL = every member uses the one season and runs T-1 steps
    const int *member_set, *set_steps;
    double *out[NVAR];                 // member 0, slot 0 of each array (NULL: not stored)
    long long mstride[NVAR];
    const MemberCoef *coef;
    ModelConsts k;
    GradConsts g;
    ConstDiv conv_div;
    double w[9];
    Switches sw;
    StripTables st;
    // misfit mode (calibration driver, SURVEY.md 8f N3): the (cell, day) pairs at which snow depth is observed, sorted by
    // owning cell and day ("sample slots"); obs_first is indexed like `codes` (ocean list of every strip) and points at
    // the cell's first slot, every cell's run ends with a sentinel day (INT_MAX).  The thread that owns a cell stores the
    // two layers {h0, h1} of the observed days into sample_hh[member][slot] -- 16 bytes per observed cell-day instead of
    // 96 per cell-day -- fire and forget: nothing on the day's critical path waits for memory.  The observation operators
    // proper (depth over ice, volume, density: all functions of the two layers and the day's ice concentration) and the
    // sums of squares run in a small epilogue kernel.
    const int *obs_first, *obs_day;
    double2 *sample_hh;
    long long sample_stride;
    int dbg;                           // timing experiments only (NESOSIM_ENS_DBG): 1 forcing always from day 0, 2 no L2 prefetch, 4 no bulk stores
    int *status;                       // set to 1 if any operand left the fast divisions' proven range (host reruns)
    long long *timing;                 // debug: [gridDim.x][ENS_NTIMER] phase cycle totals (NULL = off)
    // misfit mode on forcing sets (nesosim_set_observations_sets): every set has its own obs_first table, obs_first_stride
    // entries apart; the sets' slots follow one another in obs_day, set s from obs_slot_base[s] on.  A member samples its
    // own set only, so its row of sample_hh holds that set's slots (from obs_slot_base[set]) and the stride is the
    // slot count of the largest set, not the sum
    long long obs_first_stride;
    const int *obs_slot_base;
};

__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_acquire() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// execution barrier only (no memory fence on the arriving side): orders "I have stopped READING" against later writers
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
// shared -> global bulk copy (TMA), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_store(double *gdst, unsigned ssrc, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
}
// global -> shared bulk copy (TMA), completion counted in bytes on an mbarrier of this CTA
__device__ __forceinline__ void bulk_load(unsigned sdst, const double *gsrc, unsigned bytes, unsigned mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sdst),
                 "l"(gsrc), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy writes to shared memory must be fenced before the async proxy (TMA) reads them
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned mbar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned mbar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(mbar), "r"(parity) : "memory");
}
// arrive (count 1) on an mbarrier of ANOTHER CTA of the cluster, without any memory ordering: used only to say
// "this CTA has stopped reading", after the reads' values have been consumed
__device__ __forceinline__ void mbar_arrive_remote_relaxed(unsigned rmbar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(rmbar) : "memory");
}
// pull a range of global memory into L2 ahead of its use (no registers, no shared memory)
__device__ __forceinline__ void l2_prefetch(const void *gsrc, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
// 8-byte store into another CTA's shared memory that also counts 8 bytes on that CTA's mbarrier: the consumer
// sees the data once its barrier phase completes -- no fence, no cluster barrier on the producer side
__device__ __forceinline__ void st_async(unsigned raddr, double v, unsigned rmbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(raddr),
                 "l"(__double_as_longlong(v)), "r"(rmbar) : "memory");
}
// Forcing loads that must be ISSUED where they are written (a phase ahead of their use): volatile, so the
// compiler cannot sink them below the barriers in between to shorten the registers' live ranges.
__device__ __forceinline__ double2 ldg_early2(const void *p) {
    double2 v;
    asm volatile("ld.global.nc.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double ldg_early(const void *p) {
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned map_to_rank(unsigned saddr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster(unsigned addr, double v) {
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

// One day for a compute thread:
//   A    raw advection/divergence of its KR list entries              (calcDynamics, NESOSIM.py:189-222)
//   B    for its KO ocean cells: 3x3 Gaussian of the four raw planes   (smooth_snow,  NESOSIM.py:170-187),
//        point-wise terms, accumulators, depth update, density         (calcBudget,   NESOSIM.py:260-347)
//        -- the cell's two depths and seven accumulators never leave its registers; once the previous day's bulk
//        stores have read the planes, the new values are copied into the planes and the neighbours' halo rows
// and for the DMA warp: drain, stage the running sums, issue the day's bulk stores.
// Cross-CTA ordering per day, both through mbarriers in each CTA's shared memory and neither with a memory fence
// (a fence or an acquiring wait would serialise with the forcing loads in flight): (1) "my neighbours have finished
// reading their halo rows" -- each CTA, after its phase A, arrives (relaxed) on its neighbours' barrier; only the
// threads that push wait on it; (2) "my neighbours' halo cells of day x+1 have landed" -- the barrier counts the
// bytes they deliver with st.async.  Cluster-wide barriers are used once per member only.
// SETS: members may use different forcing sets / season lengths (compiled apart so that the plain ensemble keeps its
// parameter-bank pointers and its uniform trip count); SETS && OBS: misfit mode with per-set observation tables
template <int NTC, int KR, int KO, bool TIMING, bool SETS, bool OBS = false>
__global__ void __launch_bounds__(NTC + 32, 1) ensemble_season_kernel(const __grid_constant__ EnsArgs a) {
    constexpr int SXR = ENS_SXR;
    constexpr int NTH = NTC + 32;
    extern __shared__ __align__(128) unsigned char smem[];
    const int ny = a.ny, nx = a.nx, CL = a.st.cluster;
    const int RA = a.st.rows_alloc;
    const EnsLayout L = ens_layout(RA, nx, a.st.land_alloc);
    const unsigned PEXB = (unsigned)L.PEX * 8u;        // layer 0 -> layer 1 of any h cell (bytes)
    const unsigned ROWB = (unsigned)nx * 8u;           // one row of h (bytes)
    const unsigned HOWN = 2u * ROWB;                   // own cell (lr,c) of h0: HOWN + (lr*nx+c)*8
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(smem);
    unsigned short *s_land_code = reinterpret_cast<unsigned short *>(smem + L.off_codes);
    const unsigned mbar_stage = sbase + L.off_mbar, mbar_halo = mbar_stage + 8u, mbar_done_up = mbar_stage + 16u, mbar_drain = mbar_stage + 24u,
                   mbar_done_dn = mbar_stage + 32u;

    auto LD = [&](unsigned off) -> double { return *reinterpret_cast<const double *>(smem + off); };
    auto LD2 = [&](unsigned off) -> double2 { return *reinterpret_cast<const double2 *>(smem + off); };
    auto ST = [&](unsigned off, double v) { *reinterpret_cast<double *>(smem + off) = v; };
    auto ST2 = [&](unsigned off, double2 v) { *reinterpret_cast<double2 *>(smem + off) = v; };

    cg::cluster_group cluster = cg::this_cluster();
    const int k = (int)cluster.block_rank();
    const int cid = blockIdx.x / CL, ncl = gridDim.x / CL;
    const long long plane = (long long)ny * nx;
    const int ra = a.st.row0[k], rb = a.st.row0[k + 1], nrow = rb - ra;
    const int ncell = nrow * nx;
    const int tid = threadIdx.x;
    const bool comp = tid < NTC;       // compute thread; the last warp is the DMA warp
    const bool dma_lane = (tid == NTC);
    const int max_steps = a.T - 1;

    const int n_raw_int = a.st.raw_int_n[k], n_raw = a.st.raw_n[k];
    const int n_ocean = a.st.ocean_n[k], n_land = a.st.land_n[k];
    for (int i = tid; i < n_land; i += NTH) s_land_code[i] = a.st.codes[a.st.land_off[k] + i];
    for (unsigned i = tid; i < 2u * L.tile_bytes / 16u; i += NTH)   // zero padding of convolve(boundary='fill')
        ST2(L.off_adv + i * 16u, make_double2(0.0, 0.0));
    for (unsigned i = tid; i < 2u * (unsigned)L.PEX; i += NTH) ST(i * 8u, 0.0);   // halo rows nobody pushes to
    if (dma_lane) {
        mbar_init(mbar_stage, 1);
        mbar_init(mbar_halo, 1);
        mbar_init(mbar_drain, 1);
        // One "done reading" barrier PER NEIGHBOUR (count 1 each).  A single barrier counting both neighbours would
        // complete a phase on two arrivals of the SAME neighbour -- which happens when that neighbour needs no bytes
        // from this strip (this strip's two rows facing it hold no ocean cell) and so runs a day ahead -- and this CTA
        // would then push into the other neighbour's halo while it is still being read.
        mbar_init(mbar_done_up, 1);
        mbar_init(mbar_done_dn, 1);
    }

    // neighbour's halo cell (shared::cluster address, layer 0) that mirrors my local row lr, column c; 0 = none.
    // My top two rows are the rows below the strip above; my bottom two rows are the rows above the strip below.
    auto halo_target = [&](int lr, int c) -> unsigned {
        if (lr < 2 && k > 0) {
            const int nrow_up = ra - a.st.row0[k - 1];
            return map_to_rank(sbase + (unsigned)((nrow_up + 2 + lr) * nx + c) * 8u, (unsigned)(k - 1));
        }
        if (lr >= nrow - 2 && k < CL - 1) return map_to_rank(sbase + (unsigned)((lr - (nrow - 2)) * nx + c) * 8u, (unsigned)(k + 1));
        return 0u;
    };
    const unsigned rmbar_up = k > 0 ? map_to_rank(mbar_halo, (unsigned)(k - 1)) : 0u;
    const unsigned rmbar_dn = k < CL - 1 ? map_to_rank(mbar_halo, (unsigned)(k + 1)) : 0u;
    // I am the strip BELOW my upper neighbour and the strip ABOVE my lower one
    const unsigned rdone_up = k > 0 ? map_to_rank(mbar_done_dn, (unsigned)(k - 1)) : 0u;
    const unsigned rdone_dn = k < CL - 1 ? map_to_rank(mbar_done_up, (unsigned)(k + 1)) : 0u;

    // Work split: list entry i belongs to thread i % NTC, so every warp carries floor or ceil of the average and
    // the four schedulers of the SM see the same load.  nqA / nqB = entries of this WARP (warp-uniform: the phase
    // bodies are instantiated per count, so a warp never executes an entry none of its lanes owns).
    const int wbase = tid & ~31;
    // Raw-list entries on the grid edge (the last n_raw - n_raw_int of the list; one-sided differences, and often a
    // whole column, i.e. bank-conflicting) are dealt one per thread from the LAST thread downwards, in a slot of
    // their own, so they fall on the warps with the fewest interior entries and only that slot runs the edge code.
    const int n_edge = n_raw - n_raw_int;
    const int nqA = a.sw.dynamics ? min(KR, max(0, (n_raw_int - wbase + NTC - 1) / NTC)) : 0;
    const bool hasE = a.sw.dynamics && (NTC - 1 - (wbase + 31)) < n_edge;   // some lane of this warp holds an edge entry
    const int nqB = min(KO, max(0, (n_ocean - wbase + NTC - 1) / NTC));

    // ---- the raw-list entries this thread computes every day (interior entries tid + q*NTC in slots 0..KR-1, at most
    // one edge entry in slot KR): offset of the centre cell in the extended h0 plane and of the entry's slot in the raw
    // tiles.  flags: bit 8+j = owned cell j valid, bit 20+j = cell j's halo mirror is in the strip below (else above).
    // eflags (edge slot): first column, last column, first row, last row.
    unsigned a_c[KR + 1], a_t[KR + 1];
    unsigned flags = 0, eflags = 0;
#pragma unroll
    for (int q = 0; q <= KR; ++q) {
        const int idx = (q < KR) ? tid + q * NTC : n_raw_int + (NTC - 1 - tid);
        const bool valid = comp && ((q < KR) ? idx < n_raw_int : idx < n_raw);
        a_c[q] = HOWN + 8u;                                      // idle entry: reads around cell (0,1), writes the spare slot
        a_t[q] = L.off_adv + (unsigned)((RA + 2) * SXR) * 16u;
        if (valid) {
            const unsigned code = a.st.codes[a.st.raw_off[k] + idx];
            const int r = (int)(code >> 7), c = (int)(code & 127u);
            a_c[q] = (unsigned)((r - ra + 2) * nx + c) * 8u;
            a_t[q] = L.off_adv + (unsigned)((r - ra + 1) * SXR + c + 1) * 16u;
            if (q == KR) eflags = (c == 0 ? 1u : 0u) | (c == nx - 1 ? 2u : 0u) | (r == 0 ? 4u : 0u) | (r == ny - 1 ? 8u : 0u);
        }
    }
    // ---- the ocean cells this thread owns for the whole season (entries tid + j*NTC): offset of the cell in an
    // own-cells plane, of its top-left 3x3 tap in the raw tiles, and its mirror in a neighbour's halo
    unsigned b_ci[KO], b_t[KO], b_rem[KO];
    int o_first[OBS ? KO : 1];         // misfit mode: the cell's first observation (SETS: loaded per member, by its set)
#pragma unroll
    for (int j = 0; j < KO; ++j) {
        const int idx = tid + j * NTC;
        b_t[j] = L.off_adv;
        b_ci[j] = 0;
        b_rem[j] = 0;
        if (OBS) o_first[j] = -1;
        if (comp && idx < n_ocean) {
            if (OBS && !SETS) o_first[j] = a.obs_first[a.st.ocean_off[k] + idx];
            const unsigned code = a.st.codes[a.st.ocean_off[k] + idx];
            const int lr = (int)(code >> 7), c = (int)(code & 127u);
            b_t[j] = L.off_adv + (unsigned)(lr * SXR + c) * 16u;
            b_ci[j] = (unsigned)(lr * nx + c) * 8u;
            b_rem[j] = halo_target(lr, c);
            flags |= 1u << (8 + j);
            if (lr >= 2) flags |= 1u << (20 + j);
        }
    }

    const double nan = qnan();
    unsigned badacc = 0;               // sticky: some division operand left the proven range
    // global offsets of this strip's forcing relative to a day's plane: cell (ra-2, 0) for the raw entries
    // (a_c counts from the first halo row), cell (ra, 0) for the owned cells
    const long long go_raw = (long long)(ra - 2) * nx, go_own = (long long)ra * nx;

    long long tacc[TIMING ? 8 : 1] = {0};
    long long twA = 0, twB = 0, tw0 = 0;   // per-warp durations of the two compute phases (lane 0 of each warp)
    const bool wtiming = TIMING && a.timing != nullptr && comp && (tid & 31) == 0 && (tid >> 5) < 24;
    const bool timing = TIMING && a.timing != nullptr && (tid == 0 || dma_lane);
    long long tlast = 0;
#define ENS_TICK(slot)                                   \
    if (TIMING && timing) {                              \
        const long long now_ = clock64();                \
        tacc[slot] += now_ - tlast;                      \
        tlast = now_;                                    \
    }

    unsigned stage_parity = 0, halo_parity = 0, done_parity = 0, drain_parity = 0;
    const bool want_cum = a.out[V_ACC] != nullptr || a.out[V_OCEAN] != nullptr;

    for (int m = cid; m < a.M; m += ncl) {
        // Every CTA of the cluster is running and has zeroed its tiles (first member) / has finished the previous member's
        // last day, i.e. has stopped reading its halo rows (later members), before anyone writes slot 0 into a neighbour's
        // halo: a strip whose rows facing a neighbour hold no ocean cell never waits for that neighbour inside the day loop.
        cluster_arrive_release();
        cluster_wait_acquire();
        // this member's forcing set and season length
        const int fset = SETS ? a.member_set[m] : 0;
        const int steps = SETS ? a.set_steps[fset] : max_steps;
        const long long set_d = SETS ? (long long)fset * max_steps * plane : 0, set_f = SETS ? (long long)fset * a.T * plane : 0;
        const double2 *mDA = a.DA + set_d * 2, *mDB = a.DB + set_d;
        const double *mCumAcc = a.cumAcc + set_d, *mCumOc = a.cumOc + set_d, *mW = a.W + set_f, *mConc0 = a.conc0 + set_f;
        // output address of variable v, time slot `slot` of member m, first cell of this strip
        const long long mo_plane = (long long)m * a.mstride[V_DENS] + (long long)ra * nx;
        const long long mo_depth = (long long)m * a.mstride[V_H0] + (long long)ra * nx;
        auto outp = [&](int v, int slot) -> double * {
            return (v == V_H0 || v == V_H1) ? a.out[v] + (mo_depth + (long long)slot * 2 * plane)
                                            : a.out[v] + (mo_plane + (long long)slot * plane);
        };

        if (!comp) {
            // =============================================================== DMA warp
            if (dma_lane) bulk_wait_read<0>();   // the previous member's stores have read the planes
            __syncwarp();
            bar_arrive(BAR_DRAIN, NTH);
            cluster_arrive_release();
            cluster_wait_acquire();
            if (TIMING && timing) tlast = clock64();
            for (int x = 0; x < steps; ++x) {
                if (dma_lane) {
                    if (x + PF_DAYS < steps && !(a.dbg & 2)) {   // pull the forcing of day x+PF_DAYS into L2
                        const long long gp = (long long)(x + PF_DAYS) * plane;
                        const int r0 = ra > 0 ? ra - 1 : ra, r1 = rb < ny ? rb + 1 : rb;
                        if (a.sw.dynamics) l2_prefetch(mDA + (gp + (long long)r0 * nx) * 2, (unsigned)((r1 - r0) * nx) * 32u);
                        l2_prefetch(mDB + gp + go_own, (unsigned)ncell * 16u);
                        l2_prefetch(mW + gp + go_own, (unsigned)ncell * 8u);
                        if (a.out[V_ACC]) l2_prefetch(mCumAcc + gp + go_own, (unsigned)ncell * 8u);
                        if (a.out[V_OCEAN]) l2_prefetch(mCumOc + gp + go_own, (unsigned)ncell * 8u);
                    }
                    bulk_wait_read<0>();         // day x-1: planes and staging rows have been read
                    ENS_TICK(0)                  // drain
                    if (want_cum) {
                        const unsigned bytes = (unsigned)ncell * 8u;
                        const long long go = (long long)x * plane + go_own;
                        mbar_expect_tx(mbar_stage, (a.out[V_ACC] ? bytes : 0u) + (a.out[V_OCEAN] ? bytes : 0u));
                        if (a.out[V_ACC]) bulk_load(sbase + L.off_stage, mCumAcc + go, bytes, mbar_stage);
                        if (a.out[V_OCEAN]) bulk_load(sbase + L.off_stage + (unsigned)L.PE * 8u, mCumOc + go, bytes, mbar_stage);
                    }
                    mbar_arrive(mbar_drain);     // compute warps may overwrite the planes
                }
                __syncwarp();
                ENS_TICK(1)
                bar_sync(BAR_STORE, NTH);        // planes of day x+1 are complete (and fenced for the async proxy)
                ENS_TICK(2)                      // waiting for the compute warps
                if (dma_lane) {
                    const unsigned bytes = (unsigned)ncell * 8u;
#pragma unroll
                    for (int p = 0; p < ENS_NPLANE; ++p) {
                        const int v = ENS_PLANE_VAR[p];
                        if (a.out[v] && !(a.dbg & 4)) bulk_store(outp(v, x + 1), sbase + L.plane_off(p) + (p < 2 ? HOWN : 0u), bytes);
                    }
                    if (want_cum) {
                        mbar_wait(mbar_stage, stage_parity);
                        if (a.out[V_ACC]) bulk_store(outp(V_ACC, x + 1), sbase + L.off_stage, bytes);
                        if (a.out[V_OCEAN]) bulk_store(outp(V_OCEAN, x + 1), sbase + L.off_stage + (unsigned)L.PE * 8u, bytes);
                    }
                    bulk_commit();
                    ENS_TICK(3)                  // issue
                }
                stage_parity ^= (unsigned)want_cum;
                __syncwarp();
            }
            continue;
        }

        // =================================================================== compute warps
        bar_sync(BAR_DRAIN, NTH);   // the previous member's bulk stores have read the planes
        // coefficient products the reference forms before touching the arrays, for windT = 0 and 1, as pairs
        if (tid == 0) {
            const MemberCoef mc = a.coef[m];
            double *cf = reinterpret_cast<double *>(smem + L.off_coef);
            cf[0] = mul(mul(0.0, mc.llf), a.k.deltaT); cf[1] = mul(mul(1.0, mc.llf), a.k.deltaT);   // NESOSIM.py:71
            cf[2] = mul(0.0, a.k.deltaT);              cf[3] = mul(1.0, a.k.deltaT);                // NESOSIM.py:94
            cf[4] = mul(mc.neg_wpf_dt, 0.0);           cf[5] = mul(mc.neg_wpf_dt, 1.0);             // NESOSIM.py:119
            cf[6] = mul(mc.wpf_dt, 0.0);               cf[7] = mul(mc.wpf_dt, 1.0);                 // NESOSIM.py:122
            cf[8] = mc.wpt;                            cf[9] = mc.alf;
        }
        // ---- slot 0: genEmptyArrays zeros + the IC split of main (NESOSIM.py:604-609), every cell of the strip.
        for (int i = tid; i < ncell; i += NTC) {
            const int lr = i / nx, c = i - lr * nx;
            const long long o = go_own + i;
            double half = 0.0;
            if (a.ic) {
                double v = a.ic[(long long)m * a.ic_stride + o];
                if (mConc0[o] < a.k.minConc) v = 0.0;
                half = mul(v, 0.5);
            }
            badacc |= out_of_guard(half);
            const unsigned off = HOWN + (unsigned)i * 8u;
            ST(off, half);
            ST(off + PEXB, half);
            const unsigned rem = halo_target(lr, c);
            if (rem) {
                st_cluster(rem, half);
                st_cluster(rem + PEXB, half);
            }
#pragma unroll
            for (int p = PL_DENS; p < ENS_NPLANE; ++p) ST(L.plane_off(p) + (unsigned)i * 8u, 0.0);   // accumulators start at zero
#pragma unroll
            for (int v = 0; v < NVAR; ++v)
                if (a.out[v]) outp(v, 0)[i] = (v == V_H0 || v == V_H1) ? half : 0.0;
        }
        cluster_arrive_release();
        cluster_wait_acquire();

        // state of the owned cells, in registers for the whole season
        double r_h0[KO], r_h1[KO], r_dn[KO], r_adv[KO], r_div[KO], r_lead[KO], r_atm[KO], r_wpl[KO], r_wpg[KO], r_wp[KO];
#pragma unroll
        for (int j = 0; j < KO; ++j) {
            r_h0[j] = LD(HOWN + b_ci[j]);
            r_h1[j] = LD(HOWN + PEXB + b_ci[j]);
            r_dn[j] = r_adv[j] = r_div[j] = r_lead[j] = r_atm[j] = r_wpl[j] = r_wpg[j] = r_wp[j] = 0.0;
        }
        // misfit mode: every owned cell walks its own (day-sorted) sample slots; on an observed day the two layers
        // go to the member's sample array and the cursor moves on (the next slot's day is needed tomorrow at the
        // earliest: its load is never waited for)
        int o_idx[OBS ? KO : 1], o_day[OBS ? KO : 1];
        // (SETS: the set's tables hold the slots of all sets one after the other, the member's row of sample_hh only
        // those of its own set: the row is addressed relative to the set's first slot)
        double2 *const m_samples = !OBS ? nullptr
                                   : SETS ? a.sample_hh + ((long long)m * a.sample_stride - a.obs_slot_base[fset])
                                          : a.sample_hh + (long long)m * a.sample_stride;
        auto obs_take = [&](int j, int slot) {
            if (o_day[j] == slot) {
                m_samples[o_idx[j]] = make_double2(r_h0[j], r_h1[j]);   // snowDepths[slot, 0], snowDepths[slot, 1]
                ++o_idx[j];
                o_day[j] = __ldg(a.obs_day + o_idx[j]);
            }
        };
        if (OBS) {
#pragma unroll
            for (int j = 0; j < KO; ++j) {
                if (SETS)   // the cell's first slot in its member's set (own cells only: flags bit 8+j)
                    o_first[j] = ((flags >> (8 + j)) & 1u)
                                     ? __ldg(a.obs_first + fset * a.obs_first_stride + a.st.ocean_off[k] + tid + j * NTC)
                                     : -1;
                o_idx[j] = o_first[j];
                o_day[j] = o_first[j] >= 0 ? __ldg(a.obs_day + o_idx[j]) : 0x7fffffff;
                obs_take(j, 0);
            }
        }

        // member-independent inputs are requested ahead of their phase: L2 latency never shows
        double2 p01[KR + 1], p23[KR + 1], pfb[KO];
        double pW[KO];
        auto fetch_raw_inputs = [&](int x) {
            if (a.dbg & 1) x = 0;
            const char *base = reinterpret_cast<const char *>(mDA) + ((long long)x * plane + go_raw) * 32;
#pragma unroll
            for (int q = 0; q <= KR; ++q) {
                if ((q < KR) ? (q < nqA) : hasE) {
                    const char *p = base + (size_t)a_c[q] * 4u;
                    p01[q] = ldg_early2(p);
                    p23[q] = ldg_early2(p + 16);
                }
            }
        };
        auto fetch_cell_inputs = [&](int x) {
            if (a.dbg & 1) x = 0;
            const char *bb = reinterpret_cast<const char *>(mDB) + ((long long)x * plane + go_own) * 16;
            const char *bw = reinterpret_cast<const char *>(mW) + ((long long)x * plane + go_own) * 8;
#pragma unroll
            for (int j = 0; j < KO; ++j) {
                if (j < nqB) {
                    pfb[j] = ldg_early2(bb + (size_t)b_ci[j] * 2u);
                    pW[j] = ldg_early(bw + b_ci[j]);
                }
            }
        };
#pragma unroll
        for (int q = 0; q <= KR; ++q) p01[q] = p23[q] = make_double2(0.0, 0.0);
#pragma unroll
        for (int j = 0; j < KO; ++j) { pfb[j] = make_double2(0.0, 0.0); pW[j] = 0.0; }
        if (nqA || hasE) fetch_raw_inputs(0);

        if (TIMING && timing) tlast = clock64();
        for (int x = 0; x < steps; ++x) {
            fetch_cell_inputs(x);   // consumed in B, in flight during A
            if (TIMING && wtiming) tw0 = clock64();

            // ---------------- A: raw advection / divergence.  All loads and arithmetic of the warp's entries first,
            // the tile stores last: nothing in between can alias, so the entries' dependency chains interleave.
            auto phaseA = [&](auto nq_tag, auto edge_tag) {
                constexpr int NQ = decltype(nq_tag)::value;
                constexpr bool EDGE = decltype(edge_tag)::value;      // the warp also has entries in the edge slot
                constexpr int NE = NQ + (EDGE ? 1 : 0);
                double2 o_adv[NE], o_div[NE];
#pragma unroll
                for (int e = 0; e < NE; ++e) {
                    const int q = (e < NQ) ? e : KR;
                    const unsigned ac = a_c[q];
                    const double h0 = LD(ac), h1 = LD(ac + PEXB);
                    double gx0, gy0, gx1, gy1;
                    if (e < NQ) {
                        gx0 = div_const_bare(sub(LD(ac + 8u), LD(ac - 8u)), a.g.two_dx);
                        gy0 = div_const_bare(sub(LD(ac + ROWB), LD(ac - ROWB)), a.g.two_dx);
                        gx1 = div_const_bare(sub(LD(ac + PEXB + 8u), LD(ac + PEXB - 8u)), a.g.two_dx);
                        gy1 = div_const_bare(sub(LD(ac + PEXB + ROWB), LD(ac + PEXB - ROWB)), a.g.two_dx);
                    } else {   // grid edge: one-sided differences there (np.gradient edge_order=1)
                        const unsigned ef = eflags;
                        const unsigned am = (ef & 1u) ? ac : ac - 8u, ap = (ef & 2u) ? ac : ac + 8u;
                        const unsigned au = (ef & 4u) ? ac : ac - ROWB, aw = (ef & 8u) ? ac : ac + ROWB;
                        const bool ex = (ef & 3u) != 0u, ey = (ef & 12u) != 0u;
                        ConstDiv dxx, dyy;
                        dxx.c = ex ? a.g.dx.c : a.g.two_dx.c; dxx.rc = ex ? a.g.dx.rc : a.g.two_dx.rc; dxx.fast = 1;
                        dyy.c = ey ? a.g.dx.c : a.g.two_dx.c; dyy.rc = ey ? a.g.dx.rc : a.g.two_dx.rc; dyy.fast = 1;
                        gx0 = div_const_bare(sub(LD(ap), LD(am)), dxx);
                        gy0 = div_const_bare(sub(LD(aw), LD(au)), dyy);
                        gx1 = div_const_bare(sub(LD(ap + PEXB), LD(am + PEXB)), dxx);
                        gy1 = div_const_bare(sub(LD(aw + PEXB), LD(au + PEXB)), dyy);
                    }
                    o_adv[e] = make_double2(zero_if_nonfinite(adv_term(p01[q].x, p01[q].y, gx0, gy0)),
                                            zero_if_nonfinite(adv_term(p01[q].x, p01[q].y, gx1, gy1)));
                    o_div[e] = make_double2(zero_if_nonfinite(div_term(h0, p23[q].x, p23[q].y)),
                                            zero_if_nonfinite(div_term(h1, p23[q].x, p23[q].y)));
                }
#pragma unroll
                for (int e = 0; e < NE; ++e) {
                    const int q = (e < NQ) ? e : KR;
                    ST2(a_t[q], o_adv[e]);
                    ST2(a_t[q] + L.tile_bytes, o_div[e]);
                }
            };
            auto dispatchA = [&](auto edge_tag) {
#define ENS_A_CASE(n) \
    if constexpr (KR >= n) { if (nqA == n) phaseA(std::integral_constant<int, n>{}, edge_tag); }
                ENS_A_CASE(1) ENS_A_CASE(2) ENS_A_CASE(3) ENS_A_CASE(4) ENS_A_CASE(5) ENS_A_CASE(6)
                if constexpr (decltype(edge_tag)::value) { if (nqA == 0) phaseA(std::integral_constant<int, 0>{}, edge_tag); }
#undef ENS_A_CASE
            };
            if (!hasE) dispatchA(std::false_type{});
            else dispatchA(std::true_type{});
            if (TIMING && wtiming) twA += clock64() - tw0;
            ENS_TICK(0)   // A
            bar_sync(BAR_A, NTC);       // raw tiles complete; nobody in this CTA reads the halo rows of day x any more
            if (tid == 0) {
                // Today's pushes from the neighbours are expected only now, behind the CTA barrier: every thread of this
                // CTA has then finished waiting for YESTERDAY's phase of the halo barrier.  (Armed at the top of the day,
                // a strip that expects no bytes at all -- all-land rows on both sides -- completed today's phase at once,
                // thread 0 could arm and complete the next one, and a slower thread still waiting for yesterday's phase
                // parity saw that parity as the current, incomplete phase: deadlock.)  The pushes themselves cannot
                // arrive earlier: the neighbours wait for this CTA's "done reading" arrival right below.
                mbar_expect_tx(mbar_halo, (unsigned)a.st.halo_tx[k]);
                // (1)
                if (rdone_up) mbar_arrive_remote_relaxed(rdone_up);
                if (rdone_dn) mbar_arrive_remote_relaxed(rdone_dn);
            }
            ENS_TICK(1)

            if (TIMING && wtiming) tw0 = clock64();
            // ---------------- B: owned ocean cells, registers only
            auto phaseB = [&](auto nq_tag) {
                constexpr int NQ = decltype(nq_tag)::value;
#pragma unroll
                for (int j = 0; j < NQ; ++j) {
                    unsigned bq = 0u;
                    double2 sa = make_double2(0.0, 0.0), sd = sa;              // zeros when dynamicsInc == 0 (NESOSIM.py:287-288)
                    if (a.sw.dynamics) {
                        // astropy tap order: rows outer, columns inner, flipped kernel, accumulators start at 0.0;
                        // then smooth_snow's division and fill_nan_no_negative on an ocean cell (NESOSIM.py:276-284)
                        const unsigned ta = b_t[j], td = ta + L.tile_bytes;
                        double a0 = 0.0, a1 = 0.0, d0 = 0.0, d1 = 0.0;
#pragma unroll
                        for (int ii = 0; ii < 3; ++ii)
#pragma unroll
                            for (int jj = 0; jj < 3; ++jj) {
                                const double wgt = a.w[(2 - ii) * 3 + (2 - jj)];
                                const double2 va = LD2(ta + (unsigned)(ii * SXR + jj) * 16u);
                                const double2 vd = LD2(td + (unsigned)(ii * SXR + jj) * 16u);
                                a0 = add(a0, mul(va.x, wgt));
                                a1 = add(a1, mul(va.y, wgt));
                                d0 = add(d0, mul(vd.x, wgt));
                                d1 = add(d1, mul(vd.y, wgt));
                            }
                        // (the raw planes are finite and bounded by the guard, so the sums are finite: the
                        // non-finite -> NaN part of fill_nan_no_negative cannot trigger on an ocean cell)
                        sa = make_double2(div_const_bare(a0, a.conv_div), div_const_bare(a1, a.conv_div));
                        sd = make_double2(div_const_bare(d0, a.conv_div), div_const_bare(d1, a.conv_div));
                    }
                    const double h0 = r_h0[j], h1 = r_h1[j];
                    const double W = pW[j];
                    const double2 fb = pfb[j];
                    const unsigned wsel = (W > LD(L.off_coef + 64u)) ? 8u : 0u;   // windT (NaN > thr is False) picks the pair entry
                    double lead = -mul(mul(mul(LD(L.off_coef + wsel), h0), W), fb.y);
                    double atm = -mul(mul(mul(LD(L.off_coef + 16u + wsel), h0), W), LD(L.off_coef + 72u));
                    double wpl = mul(LD(L.off_coef + 32u + wsel), h0);
                    double wpg = mul(mul(LD(L.off_coef + 48u + wsel), h0), a.k.rho_ratio);
                    double wpn = add(wpl, wpg);
                    if (!a.sw.leadloss) lead = 0.0;
                    if (!a.sw.atmloss) atm = 0.0;
                    if (!a.sw.windpack) wpl = wpg = wpn = 0.0;
                    r_lead[j] = add(r_lead[j], lead);
                    r_atm[j] = add(r_atm[j], atm);
                    r_wpl[j] = add(r_wpl[j], wpl);
                    r_wpg[j] = add(r_wpg[j], wpg);
                    r_wp[j] = add(r_wp[j], wpn);
                    double t0 = add(add(add(add(h0, fb.x), wpl), lead), atm);   // NESOSIM.py:327 before the dynamics terms
                    double t1 = add(h1, wpg);                                  // NESOSIM.py:329
                    r_adv[j] = add(add(r_adv[j], sa.x), sa.y);   // NESOSIM.py:290
                    r_div[j] = add(add(r_div[j], sd.x), sd.y);   // NESOSIM.py:291
                    t0 = add(add(t0, sa.x), sd.x);
                    t1 = add(add(t1, sa.y), sd.y);
                    r_h0[j] = mask_nan(t0, false, true);   // NESOSIM.py:332-333
                    r_h1[j] = mask_nan(t1, false, true);
                    r_dn[j] = density_ocean_flagged(r_h0[j], r_h1[j], a.k, bq);
                    bq |= out_of_guard(r_h0[j]) | out_of_guard(r_h1[j]);
                    badacc |= bq & (flags >> (8 + j));
                }
            };
#define ENS_B_CASE(n) \
    if constexpr (KO >= n) { if (nqB == n) phaseB(std::integral_constant<int, n>{}); }
            ENS_B_CASE(1) ENS_B_CASE(2) ENS_B_CASE(3) ENS_B_CASE(4) ENS_B_CASE(5) ENS_B_CASE(6)
#undef ENS_B_CASE
            if (OBS) {
#pragma unroll
                for (int j = 0; j < KO; ++j) obs_take(j, x + 1);
            }
            if (TIMING && wtiming) twB += clock64() - tw0;
            if ((nqA || hasE) && x + 1 < steps) fetch_raw_inputs(x + 1);   // consumed in the next A
            ENS_TICK(2)   // B compute
            ENS_TICK(3)
            // the bulk stores of day x have finished READING the planes (no CTA barrier: a warp publishes as soon
            // as its own cells are done, overlapping its shared-memory stores with the other warps' arithmetic)
            mbar_wait(mbar_drain, drain_parity);
            drain_parity ^= 1u;
            ENS_TICK(4)   // drain

            // ---------------- publish: planes of day x+1 and the neighbours' halo rows
            bool waited_up = false, waited_dn = false;
            {
#pragma unroll
                for (int j = 0; j < KO; ++j) {
                    if (!((flags >> (8 + j)) & 1u)) continue;
                    const unsigned ci = b_ci[j];
                    ST(HOWN + ci, r_h0[j]);
                    ST(HOWN + PEXB + ci, r_h1[j]);
                    ST(L.plane_off(PL_DENS) + ci, r_dn[j]);
                    ST(L.plane_off(PL_ADV) + ci, r_adv[j]);
                    ST(L.plane_off(PL_DIV) + ci, r_div[j]);
                    ST(L.plane_off(PL_LEAD) + ci, r_lead[j]);
                    ST(L.plane_off(PL_ATM) + ci, r_atm[j]);
                    ST(L.plane_off(PL_WPL) + ci, r_wpl[j]);
                    ST(L.plane_off(PL_WPG) + ci, r_wpg[j]);
                    ST(L.plane_off(PL_WP) + ci, r_wp[j]);
                    if (b_rem[j]) {
                        const bool down = ((flags >> (20 + j)) & 1u) != 0u;
                        // (1): the neighbour this cell is pushed to has finished reading its halo rows of day x
                        if (down && !waited_dn) {
                            mbar_wait(mbar_done_dn, done_parity);
                            waited_dn = true;
                        }
                        if (!down && !waited_up) {
                            mbar_wait(mbar_done_up, done_parity);
                            waited_up = true;
                        }
                        const unsigned rmb = down ? rmbar_dn : rmbar_up;
                        st_async(b_rem[j], r_h0[j], rmb);
                        st_async(b_rem[j] + PEXB, r_h1[j], rmb);
                    }
                }
            }
            // land cells.  Step 0 sees the initial depths; afterwards h is NaN, so every switched-on term is NaN
            // and every switched-off term adds 0 (NESOSIM.py:287-322): closed form, written on the first two days
            // and then left alone in the planes.  The land cells of my halo rows turn NaN the same way; nobody
            // pushes them, so I write them myself.
            if (x <= 1) {
                const MemberCoef mc = a.coef[m];
                // closed-form land values from slot 2 on (slot 1 is computed from the initial depths)
                const double landAdv = a.sw.dynamics ? nan : 0.0, landLead = a.sw.leadloss ? nan : 0.0;
                const double landAtm = a.sw.atmloss ? nan : 0.0, landWp = a.sw.windpack ? nan : 0.0;
                for (int i = tid; i < n_land; i += NTC) {
                    const int code = s_land_code[i], lr = code >> 7, c = code & 127;
                    const unsigned ci = (unsigned)(lr * nx + c) * 8u;
                    double vLead = landLead, vAtm = landAtm, vWpl = landWp, vWpg = landWp, vWp = landWp;
                    if (x == 0) {
                        const long long o = go_own + (long long)lr * nx + c;
                        const double h0 = LD(HOWN + ci);
                        const double W = __ldg(mW + o);
                        const double omc = __ldg(mDB + o).y;
                        const double wt = wind_flag(W, mc.wpt);
                        vLead = add(0.0, a.sw.leadloss ? -mul(mul(mul(mul(mul(wt, mc.llf), a.k.deltaT), h0), W), omc) : 0.0);
                        vAtm = add(0.0, a.sw.atmloss ? atm_loss(wt, h0, W, mc, a.k) : 0.0);
                        double wpl = 0.0, wpg = 0.0, wpn = 0.0;
                        if (a.sw.windpack) wind_packing(wt, h0, mc, a.k, wpl, wpg, wpn);
                        vWpl = add(0.0, wpl);
                        vWpg = add(0.0, wpg);
                        vWp = add(0.0, wpn);
                    }
                    ST(HOWN + ci, nan);
                    ST(HOWN + PEXB + ci, nan);
                    ST(L.plane_off(PL_DENS) + ci, nan);
                    ST(L.plane_off(PL_ADV) + ci, landAdv);
                    ST(L.plane_off(PL_DIV) + ci, landAdv);
                    ST(L.plane_off(PL_LEAD) + ci, vLead);
                    ST(L.plane_off(PL_ATM) + ci, vAtm);
                    ST(L.plane_off(PL_WPL) + ci, vWpl);
                    ST(L.plane_off(PL_WPG) + ci, vWpg);
                    ST(L.plane_off(PL_WP) + ci, vWp);
                }
                for (int i = tid; i < a.st.hland_n[k]; i += NTC) {
                    const int code = a.st.codes[a.st.hland_off[k] + i];
                    const unsigned off = (unsigned)((code >> 7) * nx + (code & 127)) * 8u;
                    ST(off, nan);
                    ST(off + PEXB, nan);
                }
            }
            fence_async_smem();
            ENS_TICK(5)   // publish
            bar_sync(BAR_STORE, NTH);       // planes complete: the DMA warp issues the bulk stores
            ENS_TICK(6)
            mbar_wait(mbar_halo, halo_parity);   // (2): the neighbours' pushes have landed in my halo rows
            halo_parity ^= 1u;
            done_parity ^= 1u;
            ENS_TICK(7)
        }
    }
    if (dma_lane) bulk_wait_all();
    if (badacc & 1u) atomicOr(a.status, 1);
    // nobody leaves while a neighbour may still be pushing into its shared memory or waiting for its arrival
    cluster_arrive_release();
    cluster_wait_acquire();
#undef ENS_TICK
    if (TIMING && timing)
        for (int q = 0; q < (TIMING ? 8 : 1); ++q) a.timing[(long long)blockIdx.x * ENS_NTIMER + (dma_lane ? 8 : 0) + q] = tacc[q];
    if (TIMING && wtiming) {
        a.timing[(long long)blockIdx.x * ENS_NTIMER + 16 + (tid >> 5)] = twA;
        a.timing[(long long)blockIdx.x * ENS_NTIMER + 40 + (tid >> 5)] = twB;
    }
}

// host-side state of this path
struct EnsembleState {
    bool derived_valid = false;
    void *derived = nullptr;           // DA | DB | cumAcc | cumOc
    size_t derived_bytes = 0;
    unsigned short *codes_dev = nullptr;
    StripTables tables;
    bool tables_ready = false;
    size_t smem_bytes = 0;
    int max_clusters = 0;
    int variant = -1;
};

inline void ensemble_release(EnsembleState &e) {
    cudaFree(e.derived);
    cudaFree(e.codes_dev);
    e.derived = nullptr;
    e.codes_dev = nullptr;
    e.derived_bytes = 0;
    e.tables_ready = false;
}

}  // namespace nesosim
