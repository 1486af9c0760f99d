// day_kernels.cuh -- the general (any grid, any member count) day-step path: one launch advances every member
// from slot x to slot x+1.  This is the path `NESOSIM.main` (M=1) and the large grids use; the 100 km ensemble
// has its own season-resident kernel in ensemble_kernel.cuh.
//
// Data flow per output cell (SURVEY.md §3.2): h[x] (2 layers, radius 2) + U,V (radius 2) + P,C,W,mask (point)
//   -> raw adv/div on the tile grown by 1 (calcDynamics, NESOSIM.py:189-222) -> NaN/inf->0
//   -> 3x3 Gaussian (smooth_snow, NESOSIM.py:170-187) -> land mask -> 7 point-wise deltas -> 12 planes of x+1.
// Tiles of TY x TX cells with a 2-cell halo are staged in shared memory; everything else is fused.
#pragma once
#include "cell_math.cuh"

namespace nesosim {

enum Var {
    V_H0 = 0, V_H1, V_DENS, V_ACC, V_OCEAN, V_ADV, V_DIV, V_LEAD, V_ATM, V_WPL, V_WPG, V_WP, NVAR
};

struct Switches {
    int dynamics, leadloss, windpack, atmloss, clim;
};

struct DayArgs {
    int ny, nx;
    const double *P, *C, *W, *U, *V;      // this day's forcing planes (shared by all members)
    const uint8_t *mask;
    const double *prev[NVAR];              // slot x   (prev[V_DENS] unused)
    double *next[NVAR];                    // slot x+1 (NULL: not stored)
    // elements between members: one stride for the two depth layers, one for the ten [T][ny][nx] arrays (the host
    // launches member by member in the rare case where the arrays of one kind do not share a stride)
    long long depth_mstride, plane_mstride;
    const MemberCoef *coef;                // device [M]
    ModelConsts k;
    GradConsts g;
    ConstDiv conv_div;                     // divisor applied after the 3x3 sum
    ConstDiv rho_new;                      // fresh-snow density of this step (200 or the clim value)
    double w[9];                           // 3x3 kernel, row-major
    Switches sw;
    // forcing sets (multi-season batches): member m reads its planes `member_set[m] * set_stride` elements further
    // (2x that for the drift pair) and sits out once `x` reaches its season's step count.  NULL = one shared season.
    const int *member_set, *set_steps;
    long long set_stride;
    int x;
    // per-tile flag "every in-grid cell of this TX x TY tile is land/lake" (NULL: shortcut off for this launch; it is
    // only handed over when slot x was written by this library's own previous step, see day_step_land_tile)
    const uint8_t *tile_land;
};

constexpr int TX = 32;
constexpr int TY = 16;

// Scoring instantiation (SCORE, nesosim_run_season_scores* on the general path): the day kernel as the producer of the
// calibration samples on any grid.  Only the two depth layers are advanced, in a two-slot ring (the nine accumulators
// and density are neither loaded nor stored: h0/h1 of slot x+1 never depend on them), and after pdl_wait every CTA
// copies the observed cells of its tile on day x -- slot x, complete at that point -- into the members' sample rows.
// The entries of one (set, day, tile) are a contiguous run of a CSR table (cell, slot in the member's row); entry i of
// the run belongs to thread i % threads.  sample_last_day_kernel samples each member's last day from its ring slot.
struct SampleArgs {
    const int *begin;          // [sets][T][tiles] + 1 run starts of the (set, day, tile) entry lists
    const int2 *entry;         // (cell, slot)
    double2 *samples;          // [M][stride] {h0, h1}
    long long stride;
    int T, tiles;
    // sample_last_day_kernel only: the depth ring [parity][layer][M][plane] and the members' seasons
    const double *ring;
    long long plane, layer_stride;
    const int *member_set, *set_steps;   // NULL: one shared season of T days
};

// Gradient instantiation (GRAD, nesosim_run_season_score_grads): the scoring build plus the tangent-linear step of the
// two depth layers in GRAD_DIRS parameter directions (windPackFactor, leadLossFactor, atmLossFactor), DESIGN.md §4.1.
// The tangents live in a ring [parity][dir][layer][M][plane] beside the depth ring; slot 0 is zero (the IC does not
// depend on the parameters), so day 0 reads no ring at all.  The tangent samples are [M][dir][stride] {t0, t1}, written
// where the depth samples are.
constexpr int GRAD_DIRS = 3;         // NESOSIM_GRAD_DIRS
struct TangentArgs {
    const double *prev;        // slot x   of direction 0, layer 0, member 0 (dir_stride, layer_stride further: the rest)
    double *next;              // slot x+1
    long long layer_stride, dir_stride;
    double2 *samples;          // [M][GRAD_DIRS][stride] {t0, t1} (stride of SampleArgs)
    const double *ring;        // sample_last_day_grad_kernel only: the ring's parity 0
};

// Row-strip domain decomposition over peer memory (SURVEY.md §8e "Space"; host side: nesosim_strip_* in the ABI).
// This context's grid is one strip of a larger grid, extended by STRIP_GHOST ghost rows towards each neighbouring
// strip.  Only the two depth layers of the ghost rows are ever needed from a neighbour (fused stencil radius 2 of
// calcDynamics + smooth_snow, NESOSIM.py:204-213,184-185), so every strip owns two "mailboxes" (one per side,
// [parity][layer][STRIP_GHOST][nx] doubles, parity = time slot & 1) that its neighbours fill: the day kernel stores the
// new depths of its first / last STRIP_GHOST OWNED rows straight into the neighbour's mailbox (peer memory: NVLink
// between GPUs, plain global memory between strips of one GPU), and the last boundary CTA to finish publishes the
// slot number in the neighbour's flag.  The next day's boundary CTAs wait for their own flag and read the ghost rows
// from the mailbox instead of the (stale) ghost rows of their output array.  No other kernel, copy or collective runs
// between two days; CTAs away from the strip boundary never look at any of this.
constexpr int STRIP_GHOST = 2;

struct StripLink {
    int has_up, has_dn;                       // a neighbouring strip above (rows < 0) / below (rows >= ny)
    int use_mail;                             // 0 on the first step of a season: ghost rows of slot 0 come from the IC
    const double *mail_top, *mail_bot;        // this strip's mailboxes (written by the neighbours)
    double *peer_up_mail, *peer_dn_mail;      // up neighbour's BOTTOM mailbox, down neighbour's TOP mailbox
    const unsigned long long *flag_top, *flag_bot;   // latest slot the neighbour has delivered (epoch in the high word)
    unsigned long long *peer_up_flag, *peer_dn_flag;
    unsigned int *cnt_top, *cnt_bot;          // boundary CTAs done so far (this launch)
    unsigned int expect_top, expect_bot;
    int *timed_out;                           // set when a flag did not arrive within the time limit
    unsigned long long base;                  // epoch << 32: flags only ever grow
    unsigned long long timeout_ns;
};

__device__ __forceinline__ bool strip_top_cta(int y0) { return y0 - 2 < 2 * STRIP_GHOST; }
__device__ __forceinline__ bool strip_bot_cta(int y0, int ny) { return y0 + TY + 2 > ny - 2 * STRIP_GHOST; }

// Programmatic dependent launch: the day kernels of a season are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so day x+1's CTAs may become resident while day x is still
// draining.  Everything that does not depend on day x -- parameters, the forcing and mask of the CTA's cells, the drift
// tile -- is requested before pdl_wait(); yesterday's arrays are only touched after it (it returns once day x has
// completed and its writes are visible).  Without the launch attribute both instructions do nothing.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// 8-byte asynchronous global -> shared copy (no register staging); `valid` false writes 0.0 instead (src-size 0)
__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gmem_src, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int n = valid ? 8 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gmem_src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Raw advection / divergence of both layers (calcDynamics, NESOSIM.py:189-222, then fillMaskAndNaNWithZero) on the tile
// grown by one cell, from the staged depth and raw-drift tiles; zero outside the grid (convolve's boundary='fill').
// The gradient build (GRAD below) runs it twice more per direction: RAW_RECORD is the primal pass that also keeps, in
// `fin`, one bit per raw term of this thread (4 per raw cell it owns: adv0, adv1, div0, div1) telling whether the term
// was finite; RAW_TANGENT runs the same linear stencils on a staged tangent tile and zeroes each term whose primal was
// not finite (zero_if_nonfinite made the primal a constant there).  Same cell-to-thread assignment in every mode.
// RAW_FLAGS (the adjoint's record build) is the primal pass that also writes, for every cell of the tile, the finite bits
// of its four raw terms into s_fin (bits 2..5 of the cell's record byte: adv0, adv1, div0, div1).
enum RawMode { RAW_PRIMAL = 0, RAW_RECORD, RAW_TANGENT, RAW_FLAGS };
template <bool INTERIOR, int DAY_THREADS, int MODE = RAW_PRIMAL>
__device__ __forceinline__ void tile_raw_phase(const DayArgs &a, const int x0, const int y0, double (&s_h)[2][TY + 4][TX + 4],
                                               double (&s_ut)[TY + 4][TX + 4], double (&s_vt)[TY + 4][TX + 4],
                                               double (&s_raw)[4][TY + 2][TX + 2], unsigned *fin = nullptr,
                                               uint8_t *s_fin = nullptr) {
    const int tid = threadIdx.x;
    const int ny = a.ny, nx = a.nx;
    const double dT = a.k.deltaT;
    for (int i = tid; i < (TY + 2) * (TX + 2); i += DAY_THREADS) {
        const int r = i / (TX + 2), c = i - r * (TX + 2);
        const int gy = y0 + r - 1, gx = x0 + c - 1;
        double adv0 = 0.0, adv1 = 0.0, div0 = 0.0, div1 = 0.0;   // zero padding of convolve(boundary='fill')
        unsigned fbits = 0;
        if (INTERIOR || (gy >= 0 && gy < ny && gx >= 0 && gx < nx)) {
            const int sr = r + 1, sc = c + 1;
            const double ut = mul(s_ut[sr][sc], dT), vt = mul(s_vt[sr][sc], dT);   // driftGday*deltaT
            // centred difference with the constant divisor 2.*dx where no cell of the tile is a grid-edge cell
            auto grad = [&](double fm, double fc, double fp, int idx, int n) {
                return INTERIOR ? div_const(sub(fp, fm), a.g.two_dx) : gradient1d(fm, fc, fp, idx, n, a.g);
            };
            const double gxu = grad(mul(s_ut[sr][sc - 1], dT), ut, mul(s_ut[sr][sc + 1], dT), gx, nx);
            const double gyv = grad(mul(s_vt[sr - 1][sc], dT), vt, mul(s_vt[sr + 1][sc], dT), gy, ny);
#pragma unroll
            for (int l = 0; l < 2; ++l) {
                const double h = s_h[l][sr][sc];
                const double gxh = grad(s_h[l][sr][sc - 1], h, s_h[l][sr][sc + 1], gx, nx);
                const double gyh = grad(s_h[l][sr - 1][sc], h, s_h[l][sr + 1][sc], gy, ny);
                double dv, ad;
                const int k = (i - tid) / DAY_THREADS;     // this thread's k-th raw cell
                if (MODE == RAW_TANGENT) {
                    dv = ((*fin >> (4 * k + 2 + l)) & 1u) ? div_term(h, gxu, gyv) : 0.0;
                    ad = ((*fin >> (4 * k + l)) & 1u) ? adv_term(ut, vt, gxh, gyh) : 0.0;
                } else {
                    dv = zero_if_nonfinite(div_term(h, gxu, gyv));
                    ad = zero_if_nonfinite(adv_term(ut, vt, gxh, gyh));
                    if (MODE == RAW_RECORD)
                        *fin |= ((unsigned)nesosim::finite(adv_term(ut, vt, gxh, gyh)) << (4 * k + l)) |
                                ((unsigned)nesosim::finite(div_term(h, gxu, gyv)) << (4 * k + 2 + l));
                    if (MODE == RAW_FLAGS)
                        fbits |= ((unsigned)nesosim::finite(adv_term(ut, vt, gxh, gyh)) << (2 + l)) |
                                 ((unsigned)nesosim::finite(div_term(h, gxu, gyv)) << (4 + l));
                }
                if (l == 0) { adv0 = ad; div0 = dv; } else { adv1 = ad; div1 = dv; }
            }
        }
        if (MODE == RAW_FLAGS && r >= 1 && r <= TY && c >= 1 && c <= TX) s_fin[(r - 1) * TX + (c - 1)] = (uint8_t)fbits;
        s_raw[0][r][c] = adv0;
        s_raw[1][r][c] = adv1;
        s_raw[2][r][c] = div0;
        s_raw[3][r][c] = div1;
    }
}

// What the tangent passes of the gradient build need of a cell's primal step, kept in registers: yesterday's h0 and
// whether fill_nan_no_negative replaced the new h0 / h1 (NaN: non-finite or land; 0: the clamp fired).
struct GradCell {
    double h0;
    bool kill0, kill1;
};

// Record instantiation (REC, nesosim_run_season_score_adjoint): the scoring build writing the depths into a trajectory
// [T][layer][M][plane] (the host points prev/next at slots x and x+1) and one record byte per member-cell-day
// ([T-1][M][plane]): bit 0 kill0, bit 1 kill1 (fill_nan_no_negative replaced the new h0 / h1), bits 2..5 the finite bits
// of the cell's raw terms adv0, adv1, div0, div1 (0 without dynamics) -- what the backward step cannot re-derive.
struct RecArgs {
    uint8_t *flags;            // day x's record bytes [M][plane] (member stride depth_mstride)
};

// 3x3 smoothing of the four raw planes, the point-wise budget terms and the twelve stores of this thread's cells
// (SCORE: the two depth stores only; GRAD: also fills `gc`; REC: also writes the record byte from `s_fin`).
template <bool INTERIOR, bool STRIP, int DAY_THREADS, bool SCORE = false, bool GRAD = false, bool REC = false>
__device__ __forceinline__ void tile_point_phase(const DayArgs &a, const int x0, const int y0, const int m,
                                                 double (&s_h)[2][TY + 4][TX + 4], double (&s_raw)[4][TY + 2][TX + 2],
                                                 const double *h0p, const double *h1p, const MemberCoef &mc,
                                                 const double (&pf_P)[TY / (DAY_THREADS / TX)],
                                                 const double (&pf_C)[TY / (DAY_THREADS / TX)],
                                                 const double (&pf_W)[TY / (DAY_THREADS / TX)],
                                                 const double (&pf_prev)[TY / (DAY_THREADS / TX)][9],
                                                 const bool (&pf_land)[TY / (DAY_THREADS / TX)], const StripLink *sl,
                                                 GradCell *gc = nullptr, const RecArgs *rec = nullptr,
                                                 const uint8_t *s_fin = nullptr) {
    const int tid = threadIdx.x;
    const int ny = a.ny, nx = a.nx;
    const int tx = tid & (TX - 1);
    const int gx = x0 + tx;
    if (!INTERIOR && gx >= nx) return;
#pragma unroll
    for (int rr = 0; rr < TY / (DAY_THREADS / TX); ++rr) {
        const int ty = (tid / TX) + rr * (DAY_THREADS / TX);
        const int gy = y0 + ty;
        if (!INTERIOR && gy >= ny) break;
        const long long o = (long long)gy * nx + gx;
        const bool land = pf_land[rr];

        double adv0 = 0.0, adv1 = 0.0, div0 = 0.0, div1 = 0.0, h0, h1;
        if (a.sw.dynamics) {
            double sm[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const double top = conv3x3(a.w, [&](int ii, int jj) { return s_raw[p][ty + ii][tx + jj]; });
                sm[p] = mask_nan(div_const(top, a.conv_div), land, false);   // NESOSIM.py:276-284
            }
            adv0 = sm[0]; adv1 = sm[1]; div0 = sm[2]; div1 = sm[3];
            h0 = s_h[0][ty + 2][tx + 2];
            h1 = s_h[1][ty + 2][tx + 2];
        } else {
            h0 = h0p[o];
            h1 = h1p[o];
        }

        const double P = pf_P[rr], C = pf_C[rr], W = pf_W[rr];
        const double pd = div_const(P, a.rho_new);           // precipDayT/snowDensityNew (NESOSIM.py:260)
        const double acc = mul(pd, C);                       // NESOSIM.py:263
        const double oc = -mul(pd, sub(1.0, C));             // NESOSIM.py:267
        const double wt = wind_flag(W, mc.wpt);
        const double lead = a.sw.leadloss ? lead_loss(wt, h0, W, C, mc, a.k) : 0.0;
        const double atm = a.sw.atmloss ? atm_loss(wt, h0, W, mc, a.k) : 0.0;
        double wpl = 0.0, wpg = 0.0, wpn = 0.0;
        if (a.sw.windpack) wind_packing(wt, h0, mc, a.k, wpl, wpg, wpn);

        auto prev = [&](int v) { return pf_prev[rr][v - V_ACC]; };
        const long long ip = (long long)m * a.plane_mstride + o, id = (long long)m * a.depth_mstride + o;
        auto store = [&](int v, double val) {       // only the density output is optional
            if (SCORE && v != V_H0 && v != V_H1) return;
            if (v != V_DENS || a.next[v]) a.next[v][(v == V_H0 || v == V_H1) ? id : ip] = val;
        };
        store(V_ACC, add(prev(V_ACC), acc));
        store(V_OCEAN, add(prev(V_OCEAN), oc));
        store(V_ADV, add(add(prev(V_ADV), adv0), adv1));     // NESOSIM.py:290
        store(V_DIV, add(add(prev(V_DIV), div0), div1));     // NESOSIM.py:291
        store(V_LEAD, add(prev(V_LEAD), lead));
        store(V_ATM, add(prev(V_ATM), atm));
        store(V_WPL, add(prev(V_WPL), wpl));
        store(V_WPG, add(prev(V_WPG), wpg));
        store(V_WP, add(prev(V_WP), wpn));

        // NESOSIM.py:327,329 (left to right), then fill_nan_no_negative (332-333)
        double h0n = add(add(add(add(add(add(h0, acc), wpl), lead), atm), adv0), div0);
        double h1n = add(add(add(h1, wpg), adv1), div1);
        if (GRAD) {
            gc[rr].h0 = h0;
            gc[rr].kill0 = !nesosim::finite(h0n) || land || h0n < 0.0;
            gc[rr].kill1 = !nesosim::finite(h1n) || land || h1n < 0.0;
        }
        if (REC) {
            const unsigned k0 = !nesosim::finite(h0n) || land || h0n < 0.0, k1 = !nesosim::finite(h1n) || land || h1n < 0.0;
            const unsigned fb = a.sw.dynamics ? s_fin[ty * TX + tx] : 0u;
            rec->flags[id] = (uint8_t)(fb | k0 | (k1 << 1));
        }
        h0n = mask_nan(h0n, land, true);
        h1n = mask_nan(h1n, land, true);
        store(V_H0, h0n);
        store(V_H1, h1n);
        if (STRIP) {      // first / last owned rows -> the neighbour's mailbox for slot x+1
            const long long par = (long long)((a.x + 1) & 1) * 2 * STRIP_GHOST;
            if (sl->has_up && gy >= STRIP_GHOST && gy < 2 * STRIP_GHOST) {
                const long long mo = (par + (gy - STRIP_GHOST)) * nx + gx;
                sl->peer_up_mail[mo] = h0n;
                sl->peer_up_mail[mo + (long long)STRIP_GHOST * nx] = h1n;
            }
            if (sl->has_dn && gy >= ny - 2 * STRIP_GHOST && gy < ny - STRIP_GHOST) {
                const long long mo = (par + (gy - (ny - 2 * STRIP_GHOST))) * nx + gx;
                sl->peer_dn_mail[mo] = h0n;
                sl->peer_dn_mail[mo + (long long)STRIP_GHOST * nx] = h1n;
            }
        }
        const double rho = a.sw.clim ? density_clim(a.rho_new.c, h0n, h1n, C, land, a.k)
                                     : density_variable(h0n, h1n, land, a.k);
        store(V_DENS, rho);
    }
}

// The tangent of tile_point_phase in direction j (0 windPackFactor, 1 leadLossFactor, 2 atmLossFactor) for this thread's
// cells: the smoothed raw tangents (0 on land), then every point term applied to the tangent, plus -- in the parameter's
// own direction -- the same term of the primal depth with that parameter set to 1; the new tangents are summed in the
// primal's order (acc has no tangent) and zeroed where fill_nan_no_negative replaced the primal value.  `t0p`/`t1p`:
// slot x of this member's tangents (read only without dynamics: with them the staged tile is used).
template <bool INTERIOR, int DAY_THREADS>
__device__ __forceinline__ void tile_tangent_phase(const DayArgs &a, const int x0, const int y0, const int j,
                                                   double (&s_h)[2][TY + 4][TX + 4], double (&s_raw)[4][TY + 2][TX + 2],
                                                   const double *t0p, const double *t1p, double *t0n, double *t1n,
                                                   const MemberCoef &mc, const double (&pf_C)[TY / (DAY_THREADS / TX)],
                                                   const double (&pf_W)[TY / (DAY_THREADS / TX)],
                                                   const bool (&pf_land)[TY / (DAY_THREADS / TX)], const GradCell *gc) {
    const int tid = threadIdx.x;
    const int ny = a.ny, nx = a.nx;
    const int tx = tid & (TX - 1);
    const int gx = x0 + tx;
    if (!INTERIOR && gx >= nx) return;
#pragma unroll
    for (int rr = 0; rr < TY / (DAY_THREADS / TX); ++rr) {
        const int ty = (tid / TX) + rr * (DAY_THREADS / TX);
        const int gy = y0 + ty;
        if (!INTERIOR && gy >= ny) break;
        const long long o = (long long)gy * nx + gx;
        const bool land = pf_land[rr];
        double adv0 = 0.0, adv1 = 0.0, div0 = 0.0, div1 = 0.0, t0, t1;
        if (a.sw.dynamics) {
            double sm[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const double top = conv3x3(a.w, [&](int ii, int jj) { return s_raw[p][ty + ii][tx + jj]; });
                sm[p] = land ? 0.0 : div_const(top, a.conv_div);
            }
            adv0 = sm[0]; adv1 = sm[1]; div0 = sm[2]; div1 = sm[3];
            t0 = s_h[0][ty + 2][tx + 2];
            t1 = s_h[1][ty + 2][tx + 2];
        } else {
            t0 = a.x > 0 ? t0p[o] : 0.0;
            t1 = a.x > 0 ? t1p[o] : 0.0;
        }
        const double W = pf_W[rr], C = pf_C[rr], h0 = gc[rr].h0, dT = a.k.deltaT;
        const double wt = wind_flag(W, mc.wpt);
        MemberCoef one = mc;                 // the coefficients of the parameter's own direction set to 1
        one.neg_wpf_dt = -dT;
        one.wpf_dt = dT;
        one.llf = 1.0;
        one.alf = 1.0;
        double lead = 0.0, atm = 0.0, wpl = 0.0, wpg = 0.0, net;
        if (a.sw.leadloss) {
            lead = lead_loss(wt, t0, W, C, mc, a.k);
            if (j == 1) lead = add(lead, lead_loss(wt, h0, W, C, one, a.k));
        }
        if (a.sw.atmloss) {
            atm = atm_loss(wt, t0, W, mc, a.k);
            if (j == 2) atm = add(atm, atm_loss(wt, h0, W, one, a.k));
        }
        if (a.sw.windpack) {
            wind_packing(wt, t0, mc, a.k, wpl, wpg, net);
            if (j == 0) {
                double l, g;
                wind_packing(wt, h0, one, a.k, l, g, net);
                wpl = add(wpl, l);
                wpg = add(wpg, g);
            }
        }
        const double d0 = add(add(add(add(add(t0, wpl), lead), atm), adv0), div0);
        const double d1 = add(add(add(t1, wpg), adv1), div1);
        t0n[o] = gc[rr].kill0 ? 0.0 : d0;
        t1n[o] = gc[rr].kill1 ? 0.0 : d1;
    }
}

// INTERIOR: the tile with its two-cell halo lies inside the grid and none of its raw-dynamics cells is a grid-edge
// cell, so there are no bounds tests, every difference is centred and the divisor is a launch constant (the
// overwhelming majority of the CTAs on the 25 km and 5 km grids).
template <bool INTERIOR, bool STRIP = false, int DAY_THREADS = 256, bool SCORE = false, bool GRAD = false, bool REC = false>
__device__ __forceinline__ void day_step_body(const DayArgs &a, double (&s_h)[2][TY + 4][TX + 4], double (&s_ut)[TY + 4][TX + 4],
                                              double (&s_vt)[TY + 4][TX + 4], double (&s_raw)[4][TY + 2][TX + 2],
                                              const int bx, const int by, const StripLink *sl = nullptr,
                                              const SampleArgs *sa = nullptr, const TangentArgs *ta = nullptr,
                                              const RecArgs *rec = nullptr, uint8_t *s_fin = nullptr) {
    const int m = blockIdx.z;
    const int x0 = bx * TX, y0 = by * TY;     // (bx, by): the tile (blockIdx, or what a strip / season CTA picked)
    const int tid = threadIdx.x;
    const int ny = a.ny, nx = a.nx;
    const int fset = a.member_set ? a.member_set[m] : 0;
    if (a.set_steps && a.x >= a.set_steps[fset]) {            // this member's season is over (whole CTA)
        pdl_wait();      // a grid whose CTAs all leave early must still order its successor behind its predecessor
        return;
    }
    const long long fo = (long long)fset * a.set_stride;
    const double *aP = a.P + fo, *aC = a.C + fo, *aW = a.W + fo, *aU = a.U + 2 * fo, *aV = a.V + 2 * fo;
    const double *h0p = a.prev[V_H0] + (long long)m * a.depth_mstride;
    const double *h1p = a.prev[V_H1] + (long long)m * a.depth_mstride;

    // The point-wise inputs of this thread's cells (forcing, mask, yesterday's nine accumulators) are requested
    // before anything else: they land while the tiles are staged and the raw dynamics computed, instead of each
    // load waiting in front of its one consumer behind the previous store.  Forcing first (independent of day x) ...
    constexpr int CPT = TY / (DAY_THREADS / TX);   // cells per thread
    const int ptx = tid & (TX - 1), pgx = x0 + ptx;
    double pf_P[CPT], pf_C[CPT], pf_W[CPT], pf_prev[CPT][9];
    bool pf_land[CPT];
    GradCell gc[CPT];          // GRAD only: the primal state the tangent passes need
    unsigned fin = 0;          // GRAD only: finite bits of this thread's primal raw terms (tile_raw_phase)
#pragma unroll
    for (int rr = 0; rr < CPT; ++rr) {
        const int gy = y0 + (tid / TX) + rr * (DAY_THREADS / TX);
        pf_P[rr] = pf_C[rr] = pf_W[rr] = 0.0;
        pf_land[rr] = true;
        if (INTERIOR || (pgx < nx && gy < ny)) {
            const long long o = (long long)gy * nx + pgx;
            pf_P[rr] = __ldg(aP + o);
            pf_C[rr] = __ldg(aC + o);
            pf_W[rr] = __ldg(aW + o);
            pf_land[rr] = is_land(__ldg(a.mask + o));
        }
    }
    // ... and the raw drift tile straight into shared memory (the *deltaT of NESOSIM.py:204,210 is applied where the
    // raw dynamics read it; cells outside the grid are written as 0.0)
    if (a.sw.dynamics) {
        for (int i = tid; i < (TY + 4) * (TX + 4); i += DAY_THREADS) {
            const int r = i / (TX + 4), c = i - r * (TX + 4);
            const int gy = y0 + r - 2, gx = x0 + c - 2;
            const bool in = INTERIOR || (gy >= 0 && gy < ny && gx >= 0 && gx < nx);
            const long long o = in ? (long long)gy * nx + gx : 0;
            cp_async8(&s_ut[r][c], aU + o, in);
            cp_async8(&s_vt[r][c], aV + o, in);
        }
    }
    const MemberCoef mc = a.coef[m];

    pdl_wait();      // ---- from here on yesterday's slot may be read

    if (SCORE) {     // the observed cells of this tile on day x, before any thread of the CTA may leave
        const int *b = sa->begin + ((long long)fset * sa->T + a.x) * sa->tiles + (long long)by * gridDim.x + bx;
        double2 *row = sa->samples + (long long)m * sa->stride;
        for (int i = b[0] + tid; i < b[1]; i += DAY_THREADS) {
            const int2 e = sa->entry[i];
            row[e.y] = make_double2(h0p[e.x], h1p[e.x]);
            if (GRAD) {
#pragma unroll
                for (int j = 0; j < GRAD_DIRS; ++j) {
                    const double *t0 = ta->prev + j * ta->dir_stride + (long long)m * a.depth_mstride;
                    ta->samples[((long long)m * GRAD_DIRS + j) * sa->stride + e.y] =
                        a.x > 0 ? make_double2(t0[e.x], t0[ta->layer_stride + e.x]) : make_double2(0.0, 0.0);
                }
            }
        }
    }

#pragma unroll
    for (int rr = 0; rr < CPT; ++rr) {
        const int gy = y0 + (tid / TX) + rr * (DAY_THREADS / TX);
#pragma unroll
        for (int v = 0; v < 9; ++v) pf_prev[rr][v] = 0.0;
        if (!SCORE && (INTERIOR || (pgx < nx && gy < ny))) {
            const long long ip = (long long)m * a.plane_mstride + (long long)gy * nx + pgx;
#pragma unroll
            for (int v = 0; v < 9; ++v) pf_prev[rr][v] = a.prev[V_ACC + v][ip];
        }
    }

    if (a.sw.dynamics) {
        for (int i = tid; i < (TY + 4) * (TX + 4); i += DAY_THREADS) {
            const int r = i / (TX + 4), c = i - r * (TX + 4);
            const int gy = y0 + r - 2, gx = x0 + c - 2;
            const bool in = INTERIOR || (gy >= 0 && gy < ny && gx >= 0 && gx < nx);
            const long long o = in ? (long long)gy * nx + gx : 0;
            const double *mail = nullptr;      // ghost row of a neighbouring strip: depths come from the mailbox
            int mrow = 0;
            if (STRIP && in && sl->use_mail) {
                if (sl->has_up && gy < STRIP_GHOST) { mail = sl->mail_top; mrow = gy; }
                else if (sl->has_dn && gy >= ny - STRIP_GHOST) { mail = sl->mail_bot; mrow = gy - (ny - STRIP_GHOST); }
            }
            if (STRIP && mail) {
                const long long mo = ((long long)(a.x & 1) * 2 * STRIP_GHOST + mrow) * nx + gx;
                s_h[0][r][c] = __ldcg(mail + mo);
                s_h[1][r][c] = __ldcg(mail + mo + (long long)STRIP_GHOST * nx);
            } else {
                cp_async8(&s_h[0][r][c], h0p + o, in);
                cp_async8(&s_h[1][r][c], h1p + o, in);
            }
        }
        cp_async_wait_all();
        __syncthreads();
        tile_raw_phase<INTERIOR, DAY_THREADS, GRAD ? RAW_RECORD : (REC ? RAW_FLAGS : RAW_PRIMAL)>(a, x0, y0, s_h, s_ut, s_vt,
                                                                                                  s_raw, &fin, s_fin);
        __syncthreads();
    }

    tile_point_phase<INTERIOR, STRIP, DAY_THREADS, SCORE, GRAD, REC>(a, x0, y0, m, s_h, s_raw, h0p, h1p, mc, pf_P, pf_C,
                                                                     pf_W, pf_prev, pf_land, sl, gc, rec, s_fin);
    if (GRAD) {
        // The three tangent passes reuse the tile's shared buffers: the tangent tile of direction j replaces the depth tile,
        // its raw terms the raw terms (the drift tiles stay), so the gradient build needs no more shared memory.
#pragma unroll 1
        for (int j = 0; j < GRAD_DIRS; ++j) {
            const double *t0p = ta->prev + j * ta->dir_stride + (long long)m * a.depth_mstride, *t1p = t0p + ta->layer_stride;
            double *t0n = ta->next + j * ta->dir_stride + (long long)m * a.depth_mstride, *t1n = t0n + ta->layer_stride;
            if (a.sw.dynamics) {
                __syncthreads();      // every thread is done with the previous pass's tiles
                for (int i = tid; i < (TY + 4) * (TX + 4); i += DAY_THREADS) {
                    const int r = i / (TX + 4), c = i - r * (TX + 4);
                    const int gy = y0 + r - 2, gx = x0 + c - 2;
                    const bool in = INTERIOR || (gy >= 0 && gy < ny && gx >= 0 && gx < nx);
                    const long long o = in ? (long long)gy * nx + gx : 0;
                    cp_async8(&s_h[0][r][c], t0p + o, in && a.x > 0);
                    cp_async8(&s_h[1][r][c], t1p + o, in && a.x > 0);
                }
                cp_async_wait_all();
                __syncthreads();
                tile_raw_phase<INTERIOR, DAY_THREADS, RAW_TANGENT>(a, x0, y0, s_h, s_ut, s_vt, s_raw, &fin);
                __syncthreads();
            }
            tile_tangent_phase<INTERIOR, DAY_THREADS>(a, x0, y0, j, s_h, s_raw, t0p, t1p, t0n, t1n, mc, pf_C, pf_W, pf_land, gc);
        }
    }
}

// A tile without a single ocean cell (more than half of the polar grid is land, and it comes in large blocks).  From
// the second step on every depth on land is NaN (fill_nan_no_negative, NESOSIM.py:158-162,332-333), so every term that
// multiplies h0 or passes the land mask is NaN whatever its other operands are -- 0*NaN included, which the reference
// relies on too -- and only snowAcc / snowOcean (NESOSIM.py:263-270, never masked) still need their inputs: 32 B read
// per cell instead of 129, no tiles, no stencils.  Terms whose switch is off add their literal zeros as calcBudget does.
// Only used for a slot this library wrote itself in the same call (x > first_step): a caller-provided slot may hold
// finite depths on land (the IC does), and then the general code below is the reference's arithmetic.
template <int DAY_THREADS>
__device__ __forceinline__ void day_step_land_tile(const DayArgs &a, const int bx, const int by) {
    const int m = blockIdx.z;
    const int fset = a.member_set ? a.member_set[m] : 0;
    if (a.set_steps && a.x >= a.set_steps[fset]) {
        pdl_wait();
        return;
    }
    const long long fo = (long long)fset * a.set_stride;
    const int gx = bx * TX + (threadIdx.x & (TX - 1));
    if (gx >= a.nx) return;
    const double nan = qnan();
    constexpr int CPT = TY / (DAY_THREADS / TX);
    double P[CPT], C[CPT];
#pragma unroll
    for (int rr = 0; rr < CPT; ++rr) {
        const int gy = by * TY + (threadIdx.x / TX) + rr * (DAY_THREADS / TX);
        P[rr] = C[rr] = 0.0;
        if (gy < a.ny) {
            const long long o = (long long)gy * a.nx + gx;
            P[rr] = __ldg(a.P + fo + o);
            C[rr] = __ldg(a.C + fo + o);
        }
    }
    pdl_wait();
#pragma unroll
    for (int rr = 0; rr < CPT; ++rr) {
        const int gy = by * TY + (threadIdx.x / TX) + rr * (DAY_THREADS / TX);
        if (gy >= a.ny) break;
        const long long o = (long long)gy * a.nx + gx;
        const long long ip = (long long)m * a.plane_mstride + o, id = (long long)m * a.depth_mstride + o;
        auto prev = [&](int v) { return a.prev[v][ip]; };
        auto store = [&](int v, double val) {
            if (v != V_DENS || a.next[v]) a.next[v][(v == V_H0 || v == V_H1) ? id : ip] = val;
        };
        const double pacc = prev(V_ACC), poc = prev(V_OCEAN);
        const double pd = div_const(P[rr], a.rho_new);
        store(V_ACC, add(pacc, mul(pd, C[rr])));
        store(V_OCEAN, add(poc, -mul(pd, sub(1.0, C[rr]))));
        store(V_ADV, a.sw.dynamics ? nan : add(add(prev(V_ADV), 0.0), 0.0));
        store(V_DIV, a.sw.dynamics ? nan : add(add(prev(V_DIV), 0.0), 0.0));
        store(V_LEAD, a.sw.leadloss ? nan : add(prev(V_LEAD), 0.0));
        store(V_ATM, a.sw.atmloss ? nan : add(prev(V_ATM), 0.0));
        store(V_WPL, a.sw.windpack ? nan : add(prev(V_WPL), 0.0));
        store(V_WPG, a.sw.windpack ? nan : add(prev(V_WPG), 0.0));
        store(V_WP, a.sw.windpack ? nan : add(prev(V_WP), 0.0));
        store(V_H0, nan);
        store(V_H1, nan);
        store(V_DENS, nan);
    }
}

// The land tile of the scoring build: only its NaN depths are stored (a land tile has no observed cell to sample);
// GRAD: and zero tangents; REC: and the record byte of a land cell (both kills, no finite raw term).
template <int DAY_THREADS, bool GRAD = false, bool REC = false>
__device__ __forceinline__ void day_step_land_depths(const DayArgs &a, const int bx, const int by,
                                                     const TangentArgs *ta = nullptr, const RecArgs *rec = nullptr) {
    const int m = blockIdx.z;
    const int fset = a.member_set ? a.member_set[m] : 0;
    if (a.set_steps && a.x >= a.set_steps[fset]) {
        pdl_wait();
        return;
    }
    const int gx = bx * TX + (threadIdx.x & (TX - 1));
    if (gx >= a.nx) return;
    pdl_wait();
#pragma unroll
    for (int rr = 0; rr < TY / (DAY_THREADS / TX); ++rr) {
        const int gy = by * TY + (threadIdx.x / TX) + rr * (DAY_THREADS / TX);
        if (gy >= a.ny) break;
        const long long id = (long long)m * a.depth_mstride + (long long)gy * a.nx + gx;
        a.next[V_H0][id] = qnan();
        a.next[V_H1][id] = qnan();
        if (REC) rec->flags[id] = 3;
        if (GRAD) {
#pragma unroll
            for (int j = 0; j < GRAD_DIRS; ++j) {
                ta->next[j * ta->dir_stride + id] = 0.0;
                ta->next[j * ta->dir_stride + ta->layer_stride + id] = 0.0;
            }
        }
    }
}

struct TileSmem {
    double h[2][TY + 4][TX + 4];
    double ut[TY + 4][TX + 4];       // raw drift components (multiplied by deltaT where they are read)
    double vt[TY + 4][TX + 4];
    double raw[4][TY + 2][TX + 2];   // adv0, adv1, div0, div1 after the NaN->0 fill
};

template <int DAY_THREADS, bool SCORE = false, bool GRAD = false, bool REC = false>
__device__ __forceinline__ void day_step_tile(const DayArgs &a, TileSmem &sm, const int bx, const int by,
                                              const SampleArgs *sa = nullptr, const TangentArgs *ta = nullptr,
                                              const RecArgs *rec = nullptr, uint8_t *s_fin = nullptr) {
    pdl_launch_dependents();
    if (a.tile_land && a.tile_land[by * ((a.nx + TX - 1) / TX) + bx]) {
        if (SCORE) day_step_land_depths<DAY_THREADS, GRAD, REC>(a, bx, by, ta, rec);
        else day_step_land_tile<DAY_THREADS>(a, bx, by);
        return;
    }
    auto &s_h = sm.h;
    auto &s_ut = sm.ut;
    auto &s_vt = sm.vt;
    auto &s_raw = sm.raw;
    const int x0 = bx * TX, y0 = by * TY;
    const bool interior = x0 >= 2 && y0 >= 2 && x0 + TX + 2 <= a.nx && y0 + TY + 2 <= a.ny;
    if (interior) day_step_body<true, false, DAY_THREADS, SCORE, GRAD, REC>(a, s_h, s_ut, s_vt, s_raw, bx, by, nullptr, sa, ta, rec, s_fin);
    else day_step_body<false, false, DAY_THREADS, SCORE, GRAD, REC>(a, s_h, s_ut, s_vt, s_raw, bx, by, nullptr, sa, ta, rec, s_fin);
}

// Two builds of the same tile code: 256 threads x 2 cells (large grids: fewer, fatter threads) and 512 threads x 1
// cell (small grids, where a day is one wave of CTAs and its length is the dependent chain inside a CTA).
__global__ void __launch_bounds__(256) day_step_kernel(const __grid_constant__ DayArgs a) {
    __shared__ TileSmem sm;
    day_step_tile<256>(a, sm, blockIdx.x, blockIdx.y);
}
__global__ void __launch_bounds__(512, 2) day_step_kernel_512(const __grid_constant__ DayArgs a) {
    __shared__ TileSmem sm;
    day_step_tile<512>(a, sm, blockIdx.x, blockIdx.y);
}

// The scoring builds of the same two shapes (SampleArgs above).
__global__ void __launch_bounds__(256) day_step_score_kernel(const __grid_constant__ DayArgs a,
                                                             const __grid_constant__ SampleArgs s) {
    __shared__ TileSmem sm;
    day_step_tile<256, true>(a, sm, blockIdx.x, blockIdx.y, &s);
}
__global__ void __launch_bounds__(512, 2) day_step_score_kernel_512(const __grid_constant__ DayArgs a,
                                                                    const __grid_constant__ SampleArgs s) {
    __shared__ TileSmem sm;
    day_step_tile<512, true>(a, sm, blockIdx.x, blockIdx.y, &s);
}

// The gradient builds of the same two shapes (TangentArgs above).
__global__ void __launch_bounds__(256) day_step_grad_kernel(const __grid_constant__ DayArgs a,
                                                            const __grid_constant__ SampleArgs s,
                                                            const __grid_constant__ TangentArgs t) {
    __shared__ TileSmem sm;
    day_step_tile<256, true, true>(a, sm, blockIdx.x, blockIdx.y, &s, &t);
}
__global__ void __launch_bounds__(512, 2) day_step_grad_kernel_512(const __grid_constant__ DayArgs a,
                                                                   const __grid_constant__ SampleArgs s,
                                                                   const __grid_constant__ TangentArgs t) {
    __shared__ TileSmem sm;
    day_step_tile<512, true, true>(a, sm, blockIdx.x, blockIdx.y, &s, &t);
}

// The record builds of the same two shapes (RecArgs above).
__global__ void __launch_bounds__(256) day_step_record_kernel(const __grid_constant__ DayArgs a,
                                                              const __grid_constant__ SampleArgs s,
                                                              const __grid_constant__ RecArgs r) {
    __shared__ TileSmem sm;
    __shared__ uint8_t s_fin[TY * TX];
    day_step_tile<256, true, false, true>(a, sm, blockIdx.x, blockIdx.y, &s, nullptr, &r, s_fin);
}
__global__ void __launch_bounds__(512, 2) day_step_record_kernel_512(const __grid_constant__ DayArgs a,
                                                                     const __grid_constant__ SampleArgs s,
                                                                     const __grid_constant__ RecArgs r) {
    __shared__ TileSmem sm;
    __shared__ uint8_t s_fin[TY * TX];
    day_step_tile<512, true, false, true>(a, sm, blockIdx.x, blockIdx.y, &s, nullptr, &r, s_fin);
}

// The last day of every member's season (set_steps[set], or T-1), which no day kernel reads: one CTA per member copies
// its set's entries of that day from the member's ring slot.  A member whose season ended early has not touched its
// ring since (its CTAs leave the later day kernels at once).  GRAD: the tangent samples of that day too.  TRAJ: `ring`
// is the record build's trajectory [T][layer][M][plane].
template <bool GRAD, bool TRAJ = false>
__device__ __forceinline__ void sample_last_day(const SampleArgs &s, const TangentArgs *t) {
    const int m = blockIdx.x;
    const int set = s.member_set ? s.member_set[m] : 0;
    const int day = s.set_steps ? s.set_steps[set] : s.T - 1;
    const double *h0 = s.ring + (long long)(TRAJ ? day : (day & 1)) * 2 * s.layer_stride + (long long)m * s.plane;
    const double *h1 = h0 + s.layer_stride;
    const long long b = ((long long)set * s.T + day) * s.tiles;
    double2 *row = s.samples + (long long)m * s.stride;
    for (int i = s.begin[b] + threadIdx.x; i < s.begin[b + s.tiles]; i += blockDim.x) {
        const int2 e = s.entry[i];
        row[e.y] = make_double2(h0[e.x], h1[e.x]);
        if (GRAD) {
#pragma unroll
            for (int j = 0; j < GRAD_DIRS; ++j) {
                const double *t0 = t->ring + (long long)(day & 1) * GRAD_DIRS * t->dir_stride + j * t->dir_stride +
                                   (long long)m * s.plane;
                t->samples[((long long)m * GRAD_DIRS + j) * s.stride + e.y] =
                    day > 0 ? make_double2(t0[e.x], t0[t->layer_stride + e.x]) : make_double2(0.0, 0.0);
            }
        }
    }
}
__global__ void __launch_bounds__(256) sample_last_day_kernel(const __grid_constant__ SampleArgs s) {
    sample_last_day<false>(s, nullptr);
}
__global__ void __launch_bounds__(256) sample_last_day_grad_kernel(const __grid_constant__ SampleArgs s,
                                                                   const __grid_constant__ TangentArgs t) {
    sample_last_day<true>(s, &t);
}
__global__ void __launch_bounds__(256) sample_last_day_traj_kernel(const __grid_constant__ SampleArgs s) {
    sample_last_day<false, true>(s, nullptr);
}


// Backward day step of the calibration adjoint (nesosim_run_season_score_adjoint, DESIGN.md §4.1): lambda(x) from
// lambda(x+1), day x's record bytes, h0(x) and the day's forcing, as the transpose of the tangent step
// (tile_tangent_phase), then the day's seeds at its sample slots; and each cell's parameter terms mu * term(h0, param = 1)
// into the per-member-cell accumulators.  Order (restated by oracle/score_adjoint.py):
//   mu = kill ? 0 : lambda(x+1);  staged m = mu / divisor on the tile grown by 2 (0 outside the grid);
//   per raw cell r of the tile grown by 1 and layer l, where adv_l(r) was finite: nu = transposed 3x3 sum of m around r,
//   px = (nu * ut) / d_x, py = (nu * vt) / d_y (d = dx on that axis's grid edge, else 2 dx), else 0;
//   per own cell c: lam0 = ((((mu0 + wpl(mu0)) + lead(mu0)) + atm(mu0)) + wpg(mu1)) + dyn0 (terms of a killed layer
//   skipped), lam1 = mu1 + dyn1, dyn = dd - ((px[c-1] - px[c+1] + Ex) + (py[c-1] - py[c+1] + Ey)), E = (last ? p[c] : 0)
//   - (first ? p[c] : 0), dd = -((nud gxu) + (nud gyv)) where div_l(c) was finite.
// Every gate is a select: a killed cell's coefficients may be NaN.
struct AdjArgs {
    const double *lam_in;      // lambda(x+1): layer 0 of member 0 (layer_stride further: layer 1)
    double *lam_out;           // lambda(x)
    long long layer_stride;
    const double *h0;          // trajectory slot x, layer 0 (member stride depth_mstride)
    const uint8_t *flags;      // day x's record bytes [M][plane]
    double *theta;             // [M][GRAD_DIRS][plane] accumulators
    const double2 *seeds;      // [M][stride] dJ/d(h0, h1) at every sample slot
    const int *begin;          // sampling CSR of SampleArgs
    const int2 *entry;
    long long stride;
    int T, tiles;
};

// Forcing build (FORCING, nesosim_run_season_score_adjoint_forcing): per own cell of day x, with mu0 and kill0 as above,
// pd = P / rhoF and X = (((wt llf) dT) h0) W,
//   g_P = kill0 ? 0 : (mu0 C) / rhoF;
//   g_W = kill0 ? 0 : (lead ? mu0 lead_loss(W := 1) : 0) + (atm ? mu0 atm_loss(W := 1) : 0);
//   g_C = (kill0 ? 0 : mu0 pd + (lead ? mu0 X : 0)) + cseed, cseed = the conc seed of the cell's sample slot on day x
//   (0 without one);
// acc[f] += finite(F) ? F g_F : 0 for F = P, W, C, and the three values go to the per-day planes when those are given.
constexpr int FORCING_DIRS = 3;      // NESOSIM_FORCING_DIRS: precip, wind, conc
struct ForcingAdjArgs {
    const double *cseed;       // [M][stride] dJ/dC of the depth observations at every sample slot
    double *acc;               // [M][FORCING_DIRS][plane] accumulators (member stride FORCING_DIRS * depth_mstride)
    double *day[FORCING_DIRS]; // day x's plane of member 0 of each [M][T][plane] per-day output, or NULL
    long long day_mstride;     // T * plane
};

// Drift build (DRIFT, nesosim_run_season_score_adjoint_drift): the raw terms adv_l = -((ut gx(h_l)) + (vt gy(h_l))) and
// div_l = -((h_l gx(ut)) + (h_l gy(vt))) are bilinear in the depth h_l(x) (trajectory slot x) and the drift, so with nu_l
// the transposed 3x3 sum of the staged m_l around a raw cell (as for px / py above) and A_l, D_l the record's finite
// bits of adv_l, div_l:
//   per raw cell r of the tile grown by 1: Qx = qx_0 + qx_1, qx_l = D_l ? (nu_l h_l) / d_x : 0 (Qy alike with d_y);
//   per own cell c: Gx = (A_0 ? nu_0 gx(h_0) : 0) + (A_1 ? nu_1 gx(h_1) : 0) (Gy alike with gy),
//   g_u = -((Gx + ((Qx[c-1] - Qx[c+1]) + Ex)) dT), g_v = -((Gy + ((Qy[c-1] - Qy[c+1]) + Ey)) dT), E as above;
// acc[k] += finite(F) ? F g_F : 0 for F = U, V (the raw drift), and g_u, g_v go to the per-day planes when given.
// Without dynamics both are 0 and nothing is added.  A land tile is not inert here: its cells next to the ocean carry the
// Q of their ocean neighbours, so the drift build takes the land-tile shortcut for lambda alone (lambda = 0, no
// parameter or forcing term, as the plain build) and still forms g_u, g_v on the whole tile.
constexpr int DRIFT_DIRS = 2;        // NESOSIM_DRIFT_DIRS: u, v
struct DriftAdjArgs {
    double *acc;               // [M][DRIFT_DIRS][plane] accumulators (member stride DRIFT_DIRS * depth_mstride)
    double *day;               // day x's [DRIFT_DIRS][plane] of member 0 of the [M][T][DRIFT_DIRS][plane] output, or NULL
    long long day_mstride;     // T * DRIFT_DIRS * plane
};
// What the drift build adds to the shared memory (the layers of h(x) come from AdjArgs::h0, layer_stride apart).
struct DriftSmem {
    double h[2][TY + 2][TX + 2];     // h_0(x), h_1(x) on the tile grown by 1 (0 outside the grid)
    double q[2][TY + 2][TX + 2];     // Qx, Qy
};

// transposed 3x3 sum of the staged plane around (sr, sc)
__device__ __forceinline__ double conv3x3_t(const DayArgs &a, const double (&p)[TY + 4][TX + 4], int sr, int sc) {
    double acc = 0.0;
#pragma unroll
    for (int ii = 0; ii < 3; ++ii)
#pragma unroll
        for (int jj = 0; jj < 3; ++jj) acc = add(acc, mul(p[sr + 1 - ii][sc + 1 - jj], a.w[(2 - ii) * 3 + (2 - jj)]));
    return acc;
}

template <int DAY_THREADS, bool FORCING = false, bool DRIFT = false>
__device__ __forceinline__ void day_step_adjoint(const DayArgs &a, const AdjArgs &j, TileSmem &sm,
                                                 uint8_t (&s_flag)[TY + 4][TX + 4], const ForcingAdjArgs *fa = nullptr,
                                                 double (*s_gc)[TX] = nullptr, const DriftAdjArgs *da = nullptr,
                                                 DriftSmem *ds = nullptr) {
    pdl_launch_dependents();
    const int m = blockIdx.z, bx = blockIdx.x, by = blockIdx.y;
    const int fset = a.member_set ? a.member_set[m] : 0;
    if (a.set_steps && a.x >= a.set_steps[fset]) {
        pdl_wait();
        return;
    }
    const int tid = threadIdx.x, ny = a.ny, nx = a.nx;
    const int x0 = bx * TX, y0 = by * TY;
    const int tx = tid & (TX - 1), gx = x0 + tx;
    constexpr int CPT = TY / (DAY_THREADS / TX);
    const long long ms = (long long)m * a.depth_mstride;
    const double *l0p = j.lam_in + ms, *l1p = j.lam_in + j.layer_stride + ms;
    double *o0p = j.lam_out + ms, *o1p = j.lam_out + j.layer_stride + ms;
    const bool land_tile = a.tile_land && a.tile_land[by * ((nx + TX - 1) / TX) + bx];
    if (land_tile && !(DRIFT && a.sw.dynamics)) {
        // x > 0: every raw term that reads a land depth is NaN, so lambda is 0 on the whole tile and no term is added
        pdl_wait();
        if (gx >= nx) return;
#pragma unroll
        for (int rr = 0; rr < CPT; ++rr) {
            const int gy = y0 + (tid / TX) + rr * (DAY_THREADS / TX);
            if (gy >= ny) break;
            const long long o = (long long)gy * nx + gx;
            o0p[o] = 0.0;
            o1p[o] = 0.0;
            if (FORCING) {
#pragma unroll
                for (int f = 0; f < FORCING_DIRS; ++f)
                    if (fa->day[f]) fa->day[f][(long long)m * fa->day_mstride + o] = 0.0;
            }
            if (DRIFT && da->day) {
                double *d = da->day + (long long)m * da->day_mstride + o;
                d[0] = 0.0;
                d[a.depth_mstride] = 0.0;
            }
        }
        return;
    }
    const long long fo = (long long)fset * a.set_stride;
    const double *aC = a.C + fo, *aW = a.W + fo, *aU = a.U + 2 * fo, *aV = a.V + 2 * fo;
    const uint8_t *fl = j.flags + ms;
    auto &s_m = sm.h;
    auto &s_ut = sm.ut;
    auto &s_vt = sm.vt;
    auto &s_p = sm.raw;       // px0, py0, px1, py1
    // day-x inputs (written before the backward sweep began): record bytes, drift tile, own cells' forcing and h0
    for (int i = tid; i < (TY + 4) * (TX + 4); i += DAY_THREADS) {
        const int r = i / (TX + 4), c = i - r * (TX + 4);
        const int gy = y0 + r - 2, gxx = x0 + c - 2;
        const bool in = gy >= 0 && gy < ny && gxx >= 0 && gxx < nx;
        const long long o = in ? (long long)gy * nx + gxx : 0;
        s_flag[r][c] = in ? fl[o] : (uint8_t)0;
        if (a.sw.dynamics) {
            cp_async8(&s_ut[r][c], aU + o, in);
            cp_async8(&s_vt[r][c], aV + o, in);
        }
    }
    if (DRIFT && a.sw.dynamics) {     // h(x) of the tile grown by 1 (the trajectory is written before the sweep)
        const double *hg = j.h0 + ms;
        for (int i = tid; i < (TY + 2) * (TX + 2); i += DAY_THREADS) {
            const int r = i / (TX + 2), c = i - r * (TX + 2);
            const int gy = y0 + r - 1, gxx = x0 + c - 1;
            const bool in = gy >= 0 && gy < ny && gxx >= 0 && gxx < nx;
            const long long o = in ? (long long)gy * nx + gxx : 0;
            cp_async8(&ds->h[0][r][c], hg + o, in);
            cp_async8(&ds->h[1][r][c], hg + j.layer_stride + o, in);
        }
    }
    double pf_C[CPT], pf_W[CPT], pf_h0[CPT], pf_P[CPT];
#pragma unroll
    for (int rr = 0; rr < CPT; ++rr) {
        const int gy = y0 + (tid / TX) + rr * (DAY_THREADS / TX);
        pf_C[rr] = pf_W[rr] = pf_h0[rr] = pf_P[rr] = 0.0;
        if (gx < nx && gy < ny) {
            const long long o = (long long)gy * nx + gx;
            pf_C[rr] = __ldg(aC + o);
            pf_W[rr] = __ldg(aW + o);
            pf_h0[rr] = j.h0[ms + o];
            if (FORCING) pf_P[rr] = __ldg(a.P + fo + o);
        }
    }
    if (FORCING) {        // the conc seeds of the tile's sample slots on day x (the seed kernel ran before the sweep)
        const int *sb = j.begin + ((long long)fset * j.T + a.x) * j.tiles + (long long)by * gridDim.x + bx;
        for (int i = tid; i < TY * TX; i += DAY_THREADS) s_gc[i / TX][i % TX] = 0.0;
        __syncthreads();
        const double *cs = fa->cseed + (long long)m * j.stride;
        for (int i = sb[0] + tid; i < sb[1]; i += DAY_THREADS) {
            const int2 e = j.entry[i];
            const int cy = e.x / nx;
            s_gc[cy - y0][e.x - cy * nx - x0] = cs[e.y];
        }
    }
    const MemberCoef mc = a.coef[m];
    __syncthreads();      // s_flag is read by other threads than the one that loaded it

    pdl_wait();      // ---- lambda(x+1) and the accumulators may be read from here on

    const double dT = a.k.deltaT;
    if (a.sw.dynamics) {
        for (int i = tid; i < (TY + 4) * (TX + 4); i += DAY_THREADS) {
            const int r = i / (TX + 4), c = i - r * (TX + 4);
            const int gy = y0 + r - 2, gxx = x0 + c - 2;
            double m0 = 0.0, m1 = 0.0;
            if (gy >= 0 && gy < ny && gxx >= 0 && gxx < nx) {
                const long long o = (long long)gy * nx + gxx;
                const unsigned f = s_flag[r][c];
                m0 = (f & 1u) ? 0.0 : div_const(l0p[o], a.conv_div);
                m1 = (f & 2u) ? 0.0 : div_const(l1p[o], a.conv_div);
            }
            s_m[0][r][c] = m0;
            s_m[1][r][c] = m1;
        }
        cp_async_wait_all();
        __syncthreads();
        for (int i = tid; i < (TY + 2) * (TX + 2); i += DAY_THREADS) {
            const int r = i / (TX + 2), c = i - r * (TX + 2);
            const int gy = y0 + r - 1, gxx = x0 + c - 1;
            double p[4] = {0.0, 0.0, 0.0, 0.0};
            double qd[4] = {0.0, 0.0, 0.0, 0.0};    // DRIFT: qx0, qy0, qx1, qy1
            if (gy >= 0 && gy < ny && gxx >= 0 && gxx < nx) {
                const int sr = r + 1, sc = c + 1;
                const unsigned f = s_flag[sr][sc];
                const double ut = mul(s_ut[sr][sc], dT), vt = mul(s_vt[sr][sc], dT);
                const bool ex = gxx == 0 || gxx == nx - 1, ey = gy == 0 || gy == ny - 1;
                ConstDiv dxd, dyd;
                dxd.c = ex ? a.g.dx.c : a.g.two_dx.c;
                dxd.rc = ex ? a.g.dx.rc : a.g.two_dx.rc;
                dyd.c = ey ? a.g.dx.c : a.g.two_dx.c;
                dyd.rc = ey ? a.g.dx.rc : a.g.two_dx.rc;
                dxd.fast = dyd.fast = a.g.dx.fast & a.g.two_dx.fast;
#pragma unroll
                for (int l = 0; l < 2; ++l) {
                    const bool fa_l = (f >> (2 + l)) & 1u, fd_l = DRIFT && ((f >> (4 + l)) & 1u);
                    if (fa_l || fd_l) {
                        const double nu = conv3x3_t(a, s_m[l], sr, sc);
                        if (fa_l) {
                            p[2 * l] = div_const(mul(nu, ut), dxd);
                            p[2 * l + 1] = div_const(mul(nu, vt), dyd);
                        }
                        if (fd_l) {
                            const double nh = mul(nu, ds->h[l][r][c]);
                            qd[2 * l] = div_const(nh, dxd);
                            qd[2 * l + 1] = div_const(nh, dyd);
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) s_p[q][r][c] = p[q];
            if (DRIFT) {
                ds->q[0][r][c] = add(qd[0], qd[2]);
                ds->q[1][r][c] = add(qd[1], qd[3]);
            }
        }
        __syncthreads();
    }

    if (gx < nx) {
        MemberCoef one = mc;
        one.neg_wpf_dt = -dT;
        one.wpf_dt = dT;
        one.llf = 1.0;
        one.alf = 1.0;
#pragma unroll
        for (int rr = 0; rr < CPT; ++rr) {
            const int ty = (tid / TX) + rr * (DAY_THREADS / TX);
            const int gy = y0 + ty;
            if (gy >= ny) break;
            const long long o = (long long)gy * nx + gx;
            const unsigned f = s_flag[ty + 2][tx + 2];
            if (DRIFT) {
                double g[DRIFT_DIRS] = {0.0, 0.0};
                if (a.sw.dynamics) {
                    const int sr = ty + 2, sc = tx + 2, pr = ty + 1, pc = tx + 1;
                    double ax[2] = {0.0, 0.0}, ay[2] = {0.0, 0.0};
#pragma unroll
                    for (int l = 0; l < 2; ++l) {
                        if ((f >> (2 + l)) & 1u) {
                            const double (&h)[TY + 2][TX + 2] = ds->h[l];
                            const double nu = conv3x3_t(a, s_m[l], sr, sc);
                            ax[l] = mul(nu, gradient1d(h[pr][pc - 1], h[pr][pc], h[pr][pc + 1], gx, nx, a.g));
                            ay[l] = mul(nu, gradient1d(h[pr - 1][pc], h[pr][pc], h[pr + 1][pc], gy, ny, a.g));
                        }
                    }
                    const double (&qx)[TY + 2][TX + 2] = ds->q[0];
                    const double (&qy)[TY + 2][TX + 2] = ds->q[1];
                    const bool fx = gx == 0, lx = gx == nx - 1, fy = gy == 0, ly = gy == ny - 1;
                    const double ex = sub(lx ? qx[pr][pc] : 0.0, fx ? qx[pr][pc] : 0.0);
                    const double ey = sub(ly ? qy[pr][pc] : 0.0, fy ? qy[pr][pc] : 0.0);
                    g[0] = -mul(add(add(ax[0], ax[1]), add(sub(qx[pr][pc - 1], qx[pr][pc + 1]), ex)), dT);
                    g[1] = -mul(add(add(ay[0], ay[1]), add(sub(qy[pr - 1][pc], qy[pr + 1][pc]), ey)), dT);
                    const double F[DRIFT_DIRS] = {s_ut[sr][sc], s_vt[sr][sc]};
#pragma unroll
                    for (int k = 0; k < DRIFT_DIRS; ++k) {
                        double *t = da->acc + ((long long)m * DRIFT_DIRS + k) * a.depth_mstride + o;
                        *t = add(*t, nesosim::finite(F[k]) ? mul(F[k], g[k]) : 0.0);
                    }
                }
                if (da->day) {
                    double *d = da->day + (long long)m * da->day_mstride + o;
                    d[0] = g[0];
                    d[a.depth_mstride] = g[1];
                }
                if (land_tile) {     // lambda and the other terms as the land-tile shortcut above
                    o0p[o] = 0.0;
                    o1p[o] = 0.0;
                    if (FORCING) {
#pragma unroll
                        for (int fi = 0; fi < FORCING_DIRS; ++fi)
                            if (fa->day[fi]) fa->day[fi][(long long)m * fa->day_mstride + o] = 0.0;
                    }
                    continue;
                }
            }
            const bool k0 = f & 1u, k1 = (f >> 1) & 1u;
            const double mu0 = k0 ? 0.0 : l0p[o], mu1 = k1 ? 0.0 : l1p[o];
            const double W = pf_W[rr], C = pf_C[rr], h0 = pf_h0[rr];
            const double wt = wind_flag(W, mc.wpt);
            double a0 = mu0, wl, wg, wn;
            if (!k0) {
                if (a.sw.windpack) { wind_packing(wt, mu0, mc, a.k, wl, wg, wn); a0 = add(a0, wl); }
                if (a.sw.leadloss) a0 = add(a0, lead_loss(wt, mu0, W, C, mc, a.k));
                if (a.sw.atmloss) a0 = add(a0, atm_loss(wt, mu0, W, mc, a.k));
            }
            if (!k1 && a.sw.windpack) { wind_packing(wt, mu1, mc, a.k, wl, wg, wn); a0 = add(a0, wg); }
            double lam0 = a0, lam1 = mu1;
            if (a.sw.dynamics) {
                const int sr = ty + 2, sc = tx + 2, pr = ty + 1, pc = tx + 1;
                const double gxu = gradient1d(mul(s_ut[sr][sc - 1], dT), mul(s_ut[sr][sc], dT), mul(s_ut[sr][sc + 1], dT), gx, nx, a.g);
                const double gyv = gradient1d(mul(s_vt[sr - 1][sc], dT), mul(s_vt[sr][sc], dT), mul(s_vt[sr + 1][sc], dT), gy, ny, a.g);
                const bool fx = gx == 0, lx = gx == nx - 1, fy = gy == 0, ly = gy == ny - 1;
                double dyn[2];
#pragma unroll
                for (int l = 0; l < 2; ++l) {
                    double dd = 0.0;
                    if ((f >> (4 + l)) & 1u) dd = div_term(conv3x3_t(a, s_m[l], sr, sc), gxu, gyv);
                    const double (&px)[TY + 2][TX + 2] = s_p[2 * l];
                    const double (&py)[TY + 2][TX + 2] = s_p[2 * l + 1];
                    const double ex = sub(lx ? px[pr][pc] : 0.0, fx ? px[pr][pc] : 0.0);
                    const double ey = sub(ly ? py[pr][pc] : 0.0, fy ? py[pr][pc] : 0.0);
                    const double sx = add(sub(px[pr][pc - 1], px[pr][pc + 1]), ex);
                    const double sy = add(sub(py[pr - 1][pc], py[pr + 1][pc]), ey);
                    dyn[l] = sub(dd, add(sx, sy));
                }
                lam0 = add(lam0, dyn[0]);
                lam1 = add(lam1, dyn[1]);
            }
            o0p[o] = lam0;
            o1p[o] = lam1;
            // parameter terms (windPackFactor: both layers' terms first), in day order per cell
            double s0 = 0.0, s1 = 0.0;
            if (a.sw.windpack) {
                wind_packing(wt, h0, one, a.k, wl, wg, wn);
                s0 = k0 ? 0.0 : mul(mu0, wl);
                s1 = k1 ? 0.0 : mul(mu1, wg);
            }
            const double th[GRAD_DIRS] = {
                add(s0, s1),
                (a.sw.leadloss && !k0) ? mul(mu0, lead_loss(wt, h0, W, C, one, a.k)) : 0.0,
                (a.sw.atmloss && !k0) ? mul(mu0, atm_loss(wt, h0, W, one, a.k)) : 0.0};
#pragma unroll
            for (int d = 0; d < GRAD_DIRS; ++d) {
                double *t = j.theta + ((long long)m * GRAD_DIRS + d) * a.depth_mstride + o;
                *t = add(*t, th[d]);
            }
            if (FORCING) {
                const double P = pf_P[rr];
                const double gP = k0 ? 0.0 : div_const(mul(mu0, C), a.rho_new);
                const double wl1 = a.sw.leadloss ? mul(mu0, lead_loss(wt, h0, 1.0, C, mc, a.k)) : 0.0;
                const double wa1 = a.sw.atmloss ? mul(mu0, atm_loss(wt, h0, 1.0, mc, a.k)) : 0.0;
                const double gW = k0 ? 0.0 : add(wl1, wa1);
                const double X = mul(mul(mul(mul(wt, mc.llf), dT), h0), W);
                const double sC = add(mul(mu0, div_const(P, a.rho_new)), a.sw.leadloss ? mul(mu0, X) : 0.0);
                const double gC = add(k0 ? 0.0 : sC, s_gc[ty][tx]);
                const double F[FORCING_DIRS] = {P, W, C}, g[FORCING_DIRS] = {gP, gW, gC};
#pragma unroll
                for (int f = 0; f < FORCING_DIRS; ++f) {
                    if (fa->day[f]) fa->day[f][(long long)m * fa->day_mstride + o] = g[f];
                    double *t = fa->acc + ((long long)m * FORCING_DIRS + f) * a.depth_mstride + o;
                    *t = add(*t, nesosim::finite(F[f]) ? mul(F[f], g[f]) : 0.0);
                }
            }
        }
    }
    if (DRIFT && land_tile) return;     // (CTA-uniform) no sample slot on a land tile
    __syncthreads();       // the tile's lambda(x) is stored: add the day's seeds at its sample slots
    const int *b = j.begin + ((long long)fset * j.T + a.x) * j.tiles + (long long)by * gridDim.x + bx;
    const double2 *sd = j.seeds + (long long)m * j.stride;
    for (int i = b[0] + tid; i < b[1]; i += DAY_THREADS) {
        const int2 e = j.entry[i];
        const double2 v = sd[e.y];
        o0p[e.x] = add(o0p[e.x], v.x);
        o1p[e.x] = add(o1p[e.x], v.y);
    }
}

// The two CTA shapes of the general path.
__global__ void __launch_bounds__(256) day_step_adjoint_kernel(const __grid_constant__ DayArgs a,
                                                               const __grid_constant__ AdjArgs j) {
    __shared__ TileSmem sm;
    __shared__ uint8_t s_flag[TY + 4][TX + 4];
    day_step_adjoint<256>(a, j, sm, s_flag);
}
__global__ void __launch_bounds__(512, 2) day_step_adjoint_kernel_512(const __grid_constant__ DayArgs a,
                                                                      const __grid_constant__ AdjArgs j) {
    __shared__ TileSmem sm;
    __shared__ uint8_t s_flag[TY + 4][TX + 4];
    day_step_adjoint<512>(a, j, sm, s_flag);
}

// The forcing builds of the same two shapes (ForcingAdjArgs above).
__global__ void __launch_bounds__(256) day_step_adjoint_forcing_kernel(const __grid_constant__ DayArgs a,
                                                                       const __grid_constant__ AdjArgs j,
                                                                       const __grid_constant__ ForcingAdjArgs fa) {
    __shared__ TileSmem sm;
    __shared__ uint8_t s_flag[TY + 4][TX + 4];
    __shared__ double s_gc[TY][TX];
    day_step_adjoint<256, true>(a, j, sm, s_flag, &fa, s_gc);
}
__global__ void __launch_bounds__(512, 2) day_step_adjoint_forcing_kernel_512(const __grid_constant__ DayArgs a,
                                                                              const __grid_constant__ AdjArgs j,
                                                                              const __grid_constant__ ForcingAdjArgs fa) {
    __shared__ TileSmem sm;
    __shared__ uint8_t s_flag[TY + 4][TX + 4];
    __shared__ double s_gc[TY][TX];
    day_step_adjoint<512, true>(a, j, sm, s_flag, &fa, s_gc);
}

// The drift builds (DriftAdjArgs above), without and with the forcing terms, in the same two shapes.  Their tiles do
// not fit the 48 KB of static shared memory, so they take it dynamically: sizeof(AdjDriftSmem<FORCING>) bytes, which
// the host allows with cudaFuncAttributeMaxDynamicSharedMemorySize.
template <bool FORCING>
struct AdjDriftSmem {
    TileSmem sm;
    DriftSmem d;
    double gc[FORCING ? TY : 1][TX];
    uint8_t flag[TY + 4][TX + 4];
};
template <int DAY_THREADS, bool FORCING>
__device__ __forceinline__ void day_step_adjoint_drift(const DayArgs &a, const AdjArgs &j, const ForcingAdjArgs *fa,
                                                       const DriftAdjArgs &da) {
    extern __shared__ __align__(16) unsigned char adj_drift_smem[];
    AdjDriftSmem<FORCING> &s = *reinterpret_cast<AdjDriftSmem<FORCING> *>(adj_drift_smem);
    day_step_adjoint<DAY_THREADS, FORCING, true>(a, j, s.sm, s.flag, fa, FORCING ? s.gc : nullptr, &da, &s.d);
}
__global__ void __launch_bounds__(256) day_step_adjoint_drift_kernel(const __grid_constant__ DayArgs a,
                                                                     const __grid_constant__ AdjArgs j,
                                                                     const __grid_constant__ DriftAdjArgs da) {
    day_step_adjoint_drift<256, false>(a, j, nullptr, da);
}
__global__ void __launch_bounds__(512, 2) day_step_adjoint_drift_kernel_512(const __grid_constant__ DayArgs a,
                                                                            const __grid_constant__ AdjArgs j,
                                                                            const __grid_constant__ DriftAdjArgs da) {
    day_step_adjoint_drift<512, false>(a, j, nullptr, da);
}
__global__ void __launch_bounds__(256) day_step_adjoint_forcing_drift_kernel(const __grid_constant__ DayArgs a,
                                                                             const __grid_constant__ AdjArgs j,
                                                                             const __grid_constant__ ForcingAdjArgs fa,
                                                                             const __grid_constant__ DriftAdjArgs da) {
    day_step_adjoint_drift<256, true>(a, j, &fa, da);
}
__global__ void __launch_bounds__(512, 2) day_step_adjoint_forcing_drift_kernel_512(
    const __grid_constant__ DayArgs a, const __grid_constant__ AdjArgs j, const __grid_constant__ ForcingAdjArgs fa,
    const __grid_constant__ DriftAdjArgs da) {
    day_step_adjoint_drift<512, true>(a, j, &fa, da);
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Wait until *flag >= want (system-scope acquire: the neighbour may be another GPU).  Bounded: a strip whose neighbour
// never delivers raises `timed_out` and carries on with whatever the mailbox holds; the host reports the error.
__device__ __forceinline__ void strip_wait(const unsigned long long *flag, unsigned long long want, const StripLink &s) {
    if (*(volatile int *)s.timed_out) return;
    const unsigned long long t0 = globaltimer_ns();
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
        if (v >= want) return;
        if (globaltimer_ns() - t0 > s.timeout_ns) { atomicExch(s.timed_out, 1); return; }
        __nanosleep(200);
    }
}

__device__ __forceinline__ void strip_signal(unsigned int *cnt, unsigned int expect, unsigned long long *peer_flag,
                                             unsigned long long value) {
    if (atomicAdd(cnt, 1u) == expect - 1u) {     // every boundary CTA of this side has fenced its mailbox stores
        atomicExch(cnt, 0u);
        __threadfence_system();
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(peer_flag), "l"(value) : "memory");
    }
}

// The day step of one strip (M = 1, dynamics on).  CTAs whose tile (with its halo) stays clear of the ghost rows and
// of the rows a neighbour needs run exactly the code of day_step_kernel.
template <int DAY_THREADS>
__device__ __forceinline__ void day_step_strip(const DayArgs &a, const StripLink &s) {
    // CTAs start roughly in blockIdx order, so the tile rows are dealt boundary first -- top, bottom, second, second to
    // last, ... -- and the rows a neighbour waits for leave in the first wave of the launch instead of its last
    const int ty = blockIdx.y, nty = gridDim.y;
    const int by = (ty & 1) ? nty - 1 - (ty >> 1) : (ty >> 1);
    const int y0 = by * TY;
    const bool top = s.has_up && strip_top_cta(y0), bot = s.has_dn && strip_bot_cta(y0, a.ny);
    __shared__ TileSmem sm;
    if (!top && !bot) {
        day_step_tile<DAY_THREADS>(a, sm, blockIdx.x, by);
        return;
    }
    if (s.use_mail) {
        if (threadIdx.x == 0) {
            if (top) strip_wait(s.flag_top, s.base + (unsigned long long)a.x, s);
            if (bot) strip_wait(s.flag_bot, s.base + (unsigned long long)a.x, s);
        }
        __syncthreads();
    }
    // Only now may the next day's CTAs take SM slots: every CTA of this launch that depends on another strip has what it
    // needs, so this launch finishes on its own and nothing resident is waiting on a kernel that cannot be scheduled
    // (several strips sharing one GPU would otherwise deadlock on slots held by early-launched, waiting grids).
    pdl_launch_dependents();
    day_step_body<false, true, DAY_THREADS>(a, sm.h, sm.ut, sm.vt, sm.raw, blockIdx.x, by, &s);
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long v = s.base + (unsigned long long)a.x + 1ull;
        if (top) strip_signal(s.cnt_top, s.expect_top, s.peer_up_flag, v);
        if (bot) strip_signal(s.cnt_bot, s.expect_bot, s.peer_dn_flag, v);
    }
}

__global__ void __launch_bounds__(256)
day_step_strip_kernel(const __grid_constant__ DayArgs a, const __grid_constant__ StripLink s) { day_step_strip<256>(a, s); }
__global__ void __launch_bounds__(512, 2)
day_step_strip_kernel_512(const __grid_constant__ DayArgs a, const __grid_constant__ StripLink s) { day_step_strip<512>(a, s); }

// Slot 0 of every array: zeros (genEmptyArrays, NESOSIM.py:350-376) and the initial-condition split of main
// (NESOSIM.py:604-609): IC[conc<minConc]=0; h[0,0]=h[0,1]=IC*0.5.
struct InitArgs {
    long long plane;
    const double *ic;         // NULL -> zero depth
    long long ic_stride;      // 0 (shared) or plane (per member)
    const double *conc0;      // first day's concentration
    const int *member_set;    // forcing set of each member (NULL: one shared season)
    long long set_stride;     // elements between the sets' concentration stacks
    double minConc;
    double *slot0[NVAR];
    long long stride[NVAR];
};

__global__ void init_slot0_kernel(const __grid_constant__ InitArgs a) {
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= a.plane) return;
    const int m = blockIdx.y;
    double half = 0.0;
    if (a.ic) {
        double v = a.ic[(long long)m * a.ic_stride + o];
        if (__ldg(a.conc0 + (a.member_set ? a.member_set[m] * a.set_stride : 0) + o) < a.minConc) v = 0.0;
        half = mul(v, 0.5);
    }
#pragma unroll
    for (int v = 0; v < NVAR; ++v)
        if (a.slot0[v]) a.slot0[v][(long long)m * a.stride[v] + o] = (v == V_H0 || v == V_H1) ? half : 0.0;
}

// ------------------------------------------------------------------ smooth_snow, standalone (both branches)

// flags: bit0 NaN present, bit1 +inf present, bit2 -inf present  (np.isnan(arr.sum()), see oracle)
__global__ void scan_nonfinite_kernel(const double *in, long long n, int *flags) {
    int f = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double v = in[i];
        if (v != v) f |= 1;
        else if (v == __longlong_as_double(0x7ff0000000000000LL)) f |= 2;
        else if (v == __longlong_as_double(0xfff0000000000000LL)) f |= 4;
    }
    f = __reduce_or_sync(0xffffffffu, f);
    if ((threadIdx.x & 31) == 0 && f) atomicOr(flags, f);
}

struct SmoothArgs {
    const double *in;
    double *out;
    int ny, nx;
    double w[9];
    ConstDiv div;
    const int *flags;
};

__global__ void smooth_kernel(const __grid_constant__ SmoothArgs a) {
    const int gx = blockIdx.x * blockDim.x + threadIdx.x;
    const int gy = blockIdx.y * blockDim.y + threadIdx.y;
    if (gx >= a.nx || gy >= a.ny) return;
    const int fl = *a.flags;
    const bool interp = (fl & 1) || ((fl & 6) == 6);
    auto fetch = [&](int ii, int jj) {
        const int r = gy + ii - 1, c = gx + jj - 1;
        return (r >= 0 && r < a.ny && c >= 0 && c < a.nx) ? a.in[(long long)r * a.nx + c] : 0.0;
    };
    double res;
    if (!interp) {
        res = div_const(conv3x3(a.w, fetch), a.div);
    } else {
        double top = 0.0, bot = 0.0;
#pragma unroll
        for (int ii = 0; ii < 3; ++ii)
#pragma unroll
            for (int jj = 0; jj < 3; ++jj) {
                const double val = fetch(ii, jj);
                const double ker = a.w[(2 - ii) * 3 + (2 - jj)];
                if (val == val) {
                    top = add(top, mul(val, ker));
                    bot = add(bot, ker);
                }
            }
        res = (bot == 0.0) ? a.in[(long long)gy * a.nx + gx] : __ddiv_rn(top, bot);
    }
    a.out[(long long)gy * a.nx + gx] = res;
}

// ------------------------------------------------------------------ final products (OutputSnowModelFinal, utils.py:161-179)

// np.around(x, 4): multiply by 10**4, round half to even, divide -- three fp64 operations, then the float32 cast
// the NetCDF variable applies on assignment.
__device__ __forceinline__ float around4_f32(double x) {
    return __double2float_rn(__ddiv_rn(rint(__dmul_rn(x, 10000.0)), 10000.0));
}

struct FinalArgs {
    const double *depths, *density, *conc, *precip, *wind;
    long long plane, n;          // cells per day, cells in all (days*plane)
    long long forcing_days;      // conc/precip/wind repeat with this period (members sharing one forcing)
    double ice_conc_mask;
    float *snow_depth, *snow_volume, *snow_density, *ice_conc, *precip_out, *wind_out;
};

__global__ void final_products_kernel(const __grid_constant__ FinalArgs a) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
        const long long t = i / a.plane, c = i - t * a.plane;
        const double h0 = a.depths[(2 * t) * a.plane + c], h1 = a.depths[(2 * t + 1) * a.plane + c];
        const long long fi = (t % a.forcing_days) * a.plane + c;
        const double C = a.conc[fi];
        double vol = add(h0, h1);                       // snowDepths[:, 0]+snowDepths[:, 1]   (NESOSIM.py:654)
        double depth = __ddiv_rn(vol, C);               // .../iceConcDays  (0/0 and x/0 are data, masked below)
        double dens = a.density ? a.density[i] : 0.0;
        const bool masked = a.ice_conc_mask > 0.0 && C < a.ice_conc_mask;   // NaN < m is False
        if (masked) vol = depth = dens = qnan();
        double cc = C;
        if (a.ice_conc_mask > 0.0 && C < 0.15) cc = qnan();
        if (a.snow_volume) a.snow_volume[i] = around4_f32(vol);
        if (a.snow_depth) a.snow_depth[i] = around4_f32(depth);
        if (a.snow_density) a.snow_density[i] = around4_f32(dens);
        if (a.ice_conc) a.ice_conc[i] = around4_f32(cc);
        if (a.precip_out) a.precip_out[i] = around4_f32(a.precip[fi]);
        if (a.wind_out) a.wind_out[i] = around4_f32(a.wind[fi]);
    }
}

// ------------------------------------------------------------------ per-function kernels (known-answer tests)

__global__ void op_dynamics_kernel(const double *drift, const double *h, int ny, int nx, double deltaT,
                                   GradConsts g, double *adv, double *dv) {
    const int gx = blockIdx.x * blockDim.x + threadIdx.x;
    const int gy = blockIdx.y * blockDim.y + threadIdx.y;
    if (gx >= nx || gy >= ny) return;
    const long long plane = (long long)ny * nx, o = (long long)gy * nx + gx;
    const double *U = drift, *V = drift + plane;
    auto ut = [&](int r, int c) { return mul(U[(long long)r * nx + c], deltaT); };
    auto vt = [&](int r, int c) { return mul(V[(long long)r * nx + c], deltaT); };
    const int xm = max(gx - 1, 0), xp = min(gx + 1, nx - 1), ym = max(gy - 1, 0), yp = min(gy + 1, ny - 1);
    const double gxu = gradient1d(ut(gy, xm), ut(gy, gx), ut(gy, xp), gx, nx, g);
    const double gyv = gradient1d(vt(ym, gx), vt(gy, gx), vt(yp, gx), gy, ny, g);
    for (int l = 0; l < 2; ++l) {
        const double *hl = h + l * plane;
        const double hc = hl[o];
        const double gxh = gradient1d(hl[(long long)gy * nx + xm], hc, hl[(long long)gy * nx + xp], gx, nx, g);
        const double gyh = gradient1d(hl[(long long)ym * nx + gx], hc, hl[(long long)yp * nx + gx], gy, ny, g);
        dv[l * plane + o] = zero_if_nonfinite(div_term(hc, gxu, gyv));
        adv[l * plane + o] = zero_if_nonfinite(adv_term(ut(gy, gx), vt(gy, gx), gxh, gyh));
    }
}

__global__ void op_wind_terms_kernel(const double *h0, const double *W, const double *C, long long n,
                                     MemberCoef mc, ModelConsts k, double *lead, double *atm, double *wpl,
                                     double *wpg, double *wpn) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double wt = wind_flag(W[i], mc.wpt);
    if (lead) lead[i] = lead_loss(wt, h0[i], W[i], C[i], mc, k);
    if (atm) atm[i] = atm_loss(wt, h0[i], W[i], mc, k);
    double l, g_, nnet;
    wind_packing(wt, h0[i], mc, k, l, g_, nnet);
    if (wpl) wpl[i] = l;
    if (wpg) wpg[i] = g_;
    if (wpn) wpn[i] = nnet;
}

__global__ void op_fill_zero_kernel(double *a, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = zero_if_nonfinite(a[i]);
}

__global__ void op_fill_nan_kernel(double *a, const uint8_t *mask, long long n, int neg_to_zero) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = mask_nan(a[i], is_land(mask[i]), neg_to_zero != 0);
}

__global__ void op_density_kernel(const double *h, const uint8_t *mask, long long n, ModelConsts k, double *rho) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rho[i] = density_variable(h[i], h[n + i], is_land(mask[i]), k);
}

}  // namespace nesosim
