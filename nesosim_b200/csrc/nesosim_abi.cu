// nesosim_abi.cu -- C ABI (include/nesosim_b200.h) over the sm_100a kernels.  No torch, no CPU fallback.
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nesosim_b200.h"
#include "day_kernels.cuh"
#include "ensemble_kernel.cuh"
#include "drain_kernels.cuh"

using namespace nesosim;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char *what) {
    return fail(NESOSIM_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                                            \
    do {                                                    \
        cudaError_t e_ = (call);                            \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

// Decide whether div_const()'s 3-operation path is provably exact for divisor c (see cell_math.cuh).
// With c = B*2^e, B a 53-bit integer significand, x/c can only come within 3*2^-107 (relative to its binade) of
// a rounding midpoint if |A*2^k - M*B| is tiny for some dividend significand A and odd M (k = 53 or 54).  When
// B has t trailing zero bits that quantity is a non-zero multiple of 2^t, so t >= 8 already rules it out with
// a wide margin; this covers every grid spacing (dx, 2*dx are integers below 2^29 metres) and the fresh-snow
// density.  Divisors with a full significand (the Gaussian kernel sum) go through check_full_divisor().
bool check_full_divisor(double c);

ConstDiv const_div_host(double c) {
    ConstDiv d;
    d.c = c;
    d.rc = 1.0 / c;
    d.fast = 0;
    if (!(std::fabs(c) >= 1e-100 && std::fabs(c) <= 1e100)) return d;
    if (c == 1.0) { d.fast = 1; return d; }
    int e;
    const double mant = std::frexp(std::fabs(c), &e);             // [0.5, 1)
    const unsigned long long B = (unsigned long long)std::ldexp(mant, 53);
    const int tz = __builtin_ctzll(B);
    d.fast = (tz >= 8) ? 1 : (check_full_divisor(c) ? 1 : 0);
    return d;
}

// Exhaustive check for a divisor with an arbitrary significand B (odd part up to 53 bits): the only dividends
// whose quotient can lie within 2^-105 of a midpoint are those with |A*2^k - M*B| <= LIM for an odd M, i.e.
// A = (N * inv(2^k) mod B') solutions for |N| <= LIM -- a handful of significands per binade relation.  Each
// candidate (and its neighbours) is run through the same three operations on the host (fma is exact in glibc)
// and compared with the IEEE quotient.  Any mismatch disables the fast path for this divisor.
unsigned long long mulmod(unsigned long long a, unsigned long long b, unsigned long long m) {
    return (unsigned long long)(((unsigned __int128)a * b) % m);
}
unsigned long long powmod(unsigned long long a, unsigned long long e, unsigned long long m) {
    unsigned long long r = 1 % m;
    a %= m;
    while (e) {
        if (e & 1) r = mulmod(r, a, m);
        a = mulmod(a, a, m);
        e >>= 1;
    }
    return r;
}
long long egcd_inv(long long a, long long m) {   // inverse of a mod m, gcd(a,m)=1
    __int128 t = 0, nt = 1, r = m, nr = a % m;
    while (nr != 0) {
        __int128 q = r / nr;
        __int128 tmp = t - q * nt; t = nt; nt = tmp;
        tmp = r - q * nr; r = nr; nr = tmp;
    }
    if (t < 0) t += m;
    return (long long)t;
}
bool fast_div_matches(double x, double c, double rc) {
    const double q0 = x * rc;
    const double r = std::fma(-c, q0, x);
    const double q = std::fma(r, rc, q0);
    return q == x / c;
}
bool check_full_divisor(double c) {
    int e;
    const double mant = std::frexp(std::fabs(c), &e);
    unsigned long long B = (unsigned long long)std::ldexp(mant, 53);   // [2^52, 2^53)
    const int tz = __builtin_ctzll(B);
    const unsigned long long Bodd = B >> tz;
    if (Bodd == 1) return true;
    const double rc = 1.0 / c;
    const int LIM = 64;
    for (int k = 53; k <= 54; ++k) {
        // A * 2^k == N (mod Bodd)  ->  A == N * inv(2^k) (mod Bodd)
        const unsigned long long p2 = powmod(2, (unsigned long long)k, Bodd);
        const unsigned long long inv = (unsigned long long)egcd_inv((long long)p2, (long long)Bodd);
        for (int N = -LIM; N <= LIM; ++N) {
            if (N == 0) continue;
            const unsigned long long Nm = (N > 0) ? (unsigned long long)N % Bodd : Bodd - ((unsigned long long)(-N) % Bodd);
            unsigned long long A0 = mulmod(Nm % Bodd, inv, Bodd);
            // all A in [2^52, 2^53) congruent to A0 mod Bodd (Bodd may be much smaller than 2^52 only when
            // tz is large, which const_div_host() already accepted; cap the walk)
            unsigned long long first = A0 + ((((1ULL << 52) > A0) ? ((1ULL << 52) - A0 + Bodd - 1) / Bodd : 0) * Bodd);
            int walked = 0;
            for (unsigned long long A = first; A < (1ULL << 53) && walked < 4096; A += Bodd, ++walked) {
                for (int d = -1; d <= 1; ++d) {
                    const double x = (double)(A + d);
                    for (int s = -2; s <= 2; ++s) {
                        const double xs = std::ldexp(x, s);
                        if (!fast_div_matches(xs, c, rc) || !fast_div_matches(-xs, c, rc)) return false;
                    }
                }
            }
        }
    }
    return true;
}

// device-side resources of nesosim_run_season_host (host_path.inl), cached across calls
struct HostPath {
    double *forcing = nullptr;      // [P|C|W][T][plane] + drift [T][2][plane] + rho_clim [T]
    double *ic = nullptr;
    double *outbuf[2] = {nullptr, nullptr};
    size_t outbuf_bytes = 0;        // bytes of each of the two output staging buffers
    cudaStream_t compute = nullptr, copy = nullptr;
    cudaEvent_t done[2] = {nullptr, nullptr}, drained[2] = {nullptr, nullptr};
    cudaEvent_t shared_ready = nullptr;   // member 0's snowAcc / snowOcean have reached the host
    size_t ic_elems = 0;
    // compacted drain (drain_kernels.cuh): packed records on the device (one buffer per output buffer), a ring of pinned
    // host slots the chunks land in, the cell lists of the mask, one "land cells not constant" counter per chunk
    double *packed[2] = {nullptr, nullptr};
    size_t packed_bytes = 0;
    double *ring = nullptr;               // pinned
    size_t ring_bytes = 0;
    std::vector<cudaEvent_t> arrived;     // one per ring slot
    int *cells_dev = nullptr;             // ocean list, then land list
    int n_ocean = -1, n_land = 0;
    std::vector<int> ocean_idx, land_idx;
    unsigned long long *chunk_flags = nullptr;   // device
    size_t chunk_flags_n = 0;
};


}  // namespace

// A season-resident launch whose operand-range flag has not been looked at yet (asynchronous mode, nesosim_set_async).
struct PendingSeason {
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, done = nullptr;   // around the kernel; after the flag's copy to the host
    int *flag_host = nullptr;                                    // pinned
    const double *ic_dev = nullptr;
    int ic_per_member = 0, m0 = 0, mcount = 0;
    nesosim_outputs out;
    std::vector<nesosim_member_params> params;                   // of the whole context (the rerun uploads them again)
    cudaStream_t stream = nullptr;
};

struct nesosim_ctx {
    nesosim_config cfg;
    long long plane;
    uint8_t *mask_dev = nullptr;
    std::vector<uint8_t> mask_host;
    MemberCoef *coef_dev = nullptr;
    const double *P = nullptr, *C = nullptr, *W = nullptr, *UV = nullptr, *rho_clim = nullptr;
    std::vector<double> rho_clim_host;
    double *scratch = nullptr;      // lazily allocated state for outputs the caller did not ask for
    HostPath hp;
    int *flags_dev = nullptr;
    long long launches = 0;
    ModelConsts k;
    GradConsts g;
    ConstDiv conv_div, rho_fresh_div;
    EnsembleState ens;              // season-resident ensemble path (ensemble_kernel.cuh)
    cudaEvent_t ens_ev[2] = {nullptr, nullptr};   // around the season kernel, on its own stream
    double ens_kernel_ms = 0.0;     // device time of every season-kernel launch so far ...
    long long ens_kernel_launches = 0;   // ... and their number (bench.py: roofline of the dominant kernel)
    int n_sets = 1;                 // forcing sets (nesosim_set_forcing_sets); 1 = plain season
    int *member_set_dev = nullptr, *set_steps_dev = nullptr;
    std::vector<int> set_days;      // days of every forcing set (empty: one shared forcing)
    int ens_status = 0;             // flag read back from the last season-resident launch (1 = rerun needed)
    struct {                        // observations of the calibration driver (nesosim_set_observations)
        bool ready = false;
        int *first = nullptr, *day = nullptr;            // sample slots: first slot of every owned cell, day of every slot
        double2 *samples = nullptr;                      // [M][stride] {h0, h1} at every slot (written by the season kernel)
        long long stride = 0;
        double *val = nullptr, *sigma = nullptr;         // per observation: value, error, sample slot, day, cell, index
        int *o_slot = nullptr, *o_day = nullptr, *o_cell = nullptr, *src = nullptr;   // among its set's input observations
        int *kind_begin = nullptr;                       // [sets][NESOSIM_OBS_KINDS+1] every set's observations, by kind
        long long row_len = 0;                           // the largest number of input observations of one set
        bool depth_only = true;                          // every observation is depth with sigma 1 (misfit can report it)
        // nesosim_set_observations_sets: the tables of every set one after the other; set_days = the forcing layout they
        // were compiled against (empty: plain observations of one shared forcing)
        std::vector<int> set_days;
        long long first_stride = 0;                      // entries of one set's `first` table
        int *slot_base = nullptr;                        // [sets] the set's first slot in `day`
        // footprints (nesosim_set_observations_fp): every set's footprints one set after the other, each set's
        // stable-partitioned by kind; the points of footprint q are [fp_begin[q], fp_begin[q+1]) of the pt_* tables
        long long n_fp = 0;                              // footprints registered (0: point observations only)
        long long fp_row_len = 0;                        // the largest number of input footprints of one set
        long long *fp_begin = nullptr;                   // [n_fp+1]
        int *fp_kind = nullptr, *fp_src = nullptr;       // per footprint: kind, index among its set's input footprints
        double *fp_val = nullptr, *fp_sigma = nullptr;   // per footprint: observed value, error
        int *fp_kind_begin = nullptr;                    // [sets][NESOSIM_OBS_KINDS+1] every set's footprints, by kind
        int *pt_slot = nullptr, *pt_day = nullptr, *pt_cell = nullptr;   // per footprint point: sample slot, day, cell,
        double *pt_w = nullptr;                          // weight
        double *fp_mean = nullptr;                       // [M][max(1, fp_row_len)] footprint means in table order
        // compiled for the general path (nesosim_set_path(ctx, 1)): owners are the row-major ocean-cell indices, the
        // samples are filled by day_step_score_kernel (SampleArgs in day_kernels.cuh) from a two-slot depth ring
        bool general = false;
        int *smp_begin = nullptr;                        // [sets][T][tiles] + 1 run starts of the sampling entries
        int2 *smp_entry = nullptr;                       // (cell, slot in the member's row)
        int smp_tiles = 0;                               // day-kernel tiles of the grid
        double *ring = nullptr;                          // [parity 2][layer 2][M][plane]
        // nesosim_run_season_score_grads (allocated by its first call, freed with the observations): the tangent ring
        // [parity 2][GRAD_DIRS][layer 2][M][plane], the tangent samples [M][GRAD_DIRS][stride] and the footprint mean
        // derivatives [M][GRAD_DIRS][max(1, fp_row_len)]
        double *tring = nullptr;
        double2 *tsamples = nullptr;
        double *fp_dmean = nullptr;
        // nesosim_run_season_score_adjoint: the seed contributions of every sample slot, slot-major ([sets][stride] + 1
        // run starts; item (q, p): point observation q of kind -1-p when p < 0, else point p of footprint q), built at
        // registration and uploaded by the first adjoint call, which also allocates the adjoint state: the trajectory
        // [T][layer][M][plane], the record bytes [T-1][M][plane], the lambda ring [parity][layer][M][plane], the theta
        // accumulators [M][GRAD_DIRS][plane], the seeds [M][stride] and the footprint coefficients [M][fp_row_len]
        std::vector<int> adj_begin_h;
        std::vector<int2> adj_item_h;
        int *adj_begin = nullptr;
        int2 *adj_item = nullptr;
        double *traj = nullptr, *lam = nullptr, *theta_acc = nullptr, *fp_coef = nullptr;
        uint8_t *rec_flags = nullptr;
        double2 *seeds = nullptr;
        // nesosim_run_season_score_adjoint_forcing: the conc seeds [M][stride] and the scale accumulators
        // [M][FORCING_DIRS][plane], allocated by the first forcing call
        double *cseed = nullptr, *forcing_acc = nullptr;
        // nesosim_run_season_score_adjoint_drift: the drift scale accumulators [M][DRIFT_DIRS][plane], allocated by the
        // first drift call
        double *drift_acc = nullptr;
    } obs;
    bool async_mode = false;        // nesosim_set_async: run_season never synchronises; flags are resolved by nesosim_sync
    std::vector<PendingSeason> pending;
    int *flag_pool = nullptr;       // pinned host slots the pending seasons' flags are copied into
    unsigned flag_next = 0;
    std::vector<nesosim_member_params> last_params;
    long long ens_reruns = 0;
    uint8_t *tile_land_dev = nullptr;   // per day-kernel tile: no ocean cell inside (day_step_land_tile)
    bool land_shortcut = true;
    bool pdl = true;                // programmatic dependent launch of the day kernels (NESOSIM_PDL=0 turns it off)
    int day_variant = 256;          // threads per CTA of the day kernel (256 x 2 cells or 512 x 1 cell)
    int path = 0;                   // 0 auto, 1 general per-day launches, 2 season-resident ensemble kernel
    int last_path = 0;              // which path the last run_season used (1 or 2)
    int hp_last_compact = 0;        // nesosim_run_season_host: did the last call use the compacted drain?
    long long hp_full_chunks = 0;   // blocks of a compacted drain that had to be copied in full (land cells not constant)
    long long hp_blocks_packed = 0, hp_blocks_plain = 0;   // last compacted drain: (member, array) blocks sent packed / copied whole
    // row-strip domain decomposition over peer memory (nesosim_strip_*; StripLink in day_kernels.cuh)
    struct {
        bool on = false;
        int has_up = 0, has_dn = 0;
        char *block = nullptr;      // [mail_top | mail_bot | flags[2] | cnt[2] | timed_out], one cudaMalloc (IPC-exportable)
        char *peer_up = nullptr, *peer_dn = nullptr;   // the neighbours' blocks (same layout: every strip has this nx)
        bool ipc_up = false, ipc_dn = false;           // opened with cudaIpcOpenMemHandle (to be closed)
        unsigned long long epoch = 0;
        double timeout_s = 5.0;
    } strip;
};

namespace {

int upload_coef(nesosim_ctx *ctx, const nesosim_member_params *p, cudaStream_t st) {
    const int M = ctx->cfg.n_members;
    std::vector<MemberCoef> h(M);
    for (int m = 0; m < M; ++m) {
        h[m].llf = p[m].leadLossFactor;
        h[m].alf = p[m].atmLossFactor;
        h[m].wpt = p[m].windPackThresh;
        h[m].neg_wpf_dt = (-p[m].windPackFactor) * ctx->cfg.deltaT;
        h[m].wpf_dt = p[m].windPackFactor * ctx->cfg.deltaT;
    }
    // pageable source: the copy is staged before the call returns, so the vector may die afterwards
    CU(cudaMemcpyAsync(ctx->coef_dev, h.data(), sizeof(MemberCoef) * M, cudaMemcpyHostToDevice, st));
    return NESOSIM_OK;
}

int ensure_scratch(nesosim_ctx *ctx) {
    if (ctx->scratch) return NESOSIM_OK;
    const size_t n = (size_t)NVAR * 2 * ctx->cfg.n_members * ctx->plane;
    CU(cudaMalloc(&ctx->scratch, n * sizeof(double)));
    CU(cudaMemset(ctx->scratch, 0, n * sizeof(double)));
    return NESOSIM_OK;
}

double *out_base(const nesosim_outputs *o, int v) {
    switch (v) {
        case V_H0: case V_H1: return o->snowDepths;
        case V_DENS: return o->density;
        case V_ACC: return o->snowAcc;
        case V_OCEAN: return o->snowOcean;
        case V_ADV: return o->snowAdv;
        case V_DIV: return o->snowDiv;
        case V_LEAD: return o->snowLead;
        case V_ATM: return o->snowAtm;
        case V_WPL: return o->snowWindPackLoss;
        case V_WPG: return o->snowWindPackGain;
        case V_WP: return o->snowWindPack;
    }
    return nullptr;
}

// pointer to variable v, time slot t, member 0, plus the member stride
// (`o` already points at the first member of the range being run; `m0` only offsets the internal scratch)
void slot_ptr(const nesosim_ctx *ctx, const nesosim_outputs *o, int v, int t, int m0, double **ptr, long long *stride) {
    double *base = out_base(o, v);
    const long long plane = ctx->plane;
    if (base) {
        if (v == V_H0 || v == V_H1) {
            *ptr = base + ((long long)t * 2 + (v == V_H1 ? 1 : 0)) * plane;
            *stride = o->depth_member_stride;
        } else {
            *ptr = base + (long long)t * plane;
            *stride = o->plane_member_stride;
        }
    } else {
        *ptr = ctx->scratch ? ctx->scratch + (((long long)v * 2 + (t & 1)) * ctx->cfg.n_members + m0) * plane : nullptr;
        *stride = plane;
    }
}

bool any_missing(const nesosim_outputs *o) {
    for (int v = 0; v < NVAR; ++v)
        if (v != V_DENS && !out_base(o, v)) return true;
    return false;
}

int check_outputs(const nesosim_ctx *ctx, const nesosim_outputs *o) {
    if (!o) return fail(NESOSIM_ERR_ARG, "outputs struct is NULL");
    const long long T = ctx->cfg.num_days, plane = ctx->plane;
    if (ctx->cfg.n_members > 1) {
        if (o->snowDepths && o->depth_member_stride < T * 2 * plane)
            return fail(NESOSIM_ERR_ARG, "depth_member_stride smaller than T*2*ny*nx");
        if (o->plane_member_stride < T * plane) {
            for (int v = 2; v < NVAR; ++v)
                if (out_base(o, v)) return fail(NESOSIM_ERR_ARG, "plane_member_stride smaller than T*ny*nx");
        }
    }
    return NESOSIM_OK;
}

// Layout of a strip's exchange block (nesosim_strip_setup): two mailboxes of [parity 2][layer 2][STRIP_GHOST][nx]
// doubles, then the two flags, the two CTA counters and the time-out mark.
// Day kernels are launched with programmatic stream serialization (see pdl_wait in day_kernels.cuh): the next day's
// CTAs may start their day-independent prologue while this day's last CTAs finish.
template <typename... KArgs, typename... Args>
cudaError_t launch_day_kernel_smem(void (*kern)(KArgs...), dim3 grid, int threads, size_t smem, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}
template <typename... KArgs, typename... Args>
cudaError_t launch_day_kernel(void (*kern)(KArgs...), dim3 grid, int threads, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

void obs_release(nesosim_ctx *ctx) {
    auto &ob = ctx->obs;
    cudaFree(ob.first); cudaFree(ob.day); cudaFree(ob.val); cudaFree(ob.sigma); cudaFree(ob.samples);
    cudaFree(ob.o_slot); cudaFree(ob.o_day); cudaFree(ob.o_cell); cudaFree(ob.src);
    cudaFree(ob.kind_begin); cudaFree(ob.slot_base);
    cudaFree(ob.fp_begin); cudaFree(ob.fp_kind); cudaFree(ob.fp_src); cudaFree(ob.fp_val); cudaFree(ob.fp_sigma);
    cudaFree(ob.fp_kind_begin); cudaFree(ob.pt_slot); cudaFree(ob.pt_day); cudaFree(ob.pt_cell); cudaFree(ob.pt_w);
    cudaFree(ob.fp_mean);
    cudaFree(ob.smp_begin); cudaFree(ob.smp_entry); cudaFree(ob.ring);
    cudaFree(ob.tring); cudaFree(ob.tsamples); cudaFree(ob.fp_dmean);
    cudaFree(ob.adj_begin); cudaFree(ob.adj_item); cudaFree(ob.traj); cudaFree(ob.lam); cudaFree(ob.theta_acc);
    cudaFree(ob.fp_coef); cudaFree(ob.rec_flags); cudaFree(ob.seeds); cudaFree(ob.cseed); cudaFree(ob.forcing_acc);
    cudaFree(ob.drift_acc);
    ob = {};
}

void strip_release(nesosim_ctx *ctx) {
    if (ctx->strip.ipc_up && ctx->strip.peer_up) cudaIpcCloseMemHandle(ctx->strip.peer_up);
    if (ctx->strip.ipc_dn && ctx->strip.peer_dn) cudaIpcCloseMemHandle(ctx->strip.peer_dn);
    cudaFree(ctx->strip.block);
    ctx->strip.block = ctx->strip.peer_up = ctx->strip.peer_dn = nullptr;
    ctx->strip.ipc_up = ctx->strip.ipc_dn = false;
    ctx->strip.on = false;
}

size_t strip_mail_bytes(int nx) { return (size_t)2 * 2 * STRIP_GHOST * nx * sizeof(double); }
size_t strip_block_bytes(int nx) { return 2 * strip_mail_bytes(nx) + 2 * sizeof(unsigned long long) + 4 * sizeof(unsigned int); }

void strip_link(const nesosim_ctx *ctx, int x, dim3 grid, StripLink *s) {
    const int nx = ctx->cfg.nx, ny = ctx->cfg.ny;
    const size_t mb = strip_mail_bytes(nx);
    auto mail = [&](char *blk, int side) { return (double *)(blk + side * mb); };
    auto flag = [&](char *blk, int side) { return (unsigned long long *)(blk + 2 * mb) + side; };
    char *blk = ctx->strip.block;
    unsigned int *cnt = (unsigned int *)(blk + 2 * mb + 2 * sizeof(unsigned long long));
    s->has_up = ctx->strip.has_up;
    s->has_dn = ctx->strip.has_dn;
    s->use_mail = x > 0;
    s->mail_top = mail(blk, 0);
    s->mail_bot = mail(blk, 1);
    s->flag_top = flag(blk, 0);
    s->flag_bot = flag(blk, 1);
    s->peer_up_mail = ctx->strip.peer_up ? mail(ctx->strip.peer_up, 1) : nullptr;
    s->peer_up_flag = ctx->strip.peer_up ? flag(ctx->strip.peer_up, 1) : nullptr;
    s->peer_dn_mail = ctx->strip.peer_dn ? mail(ctx->strip.peer_dn, 0) : nullptr;
    s->peer_dn_flag = ctx->strip.peer_dn ? flag(ctx->strip.peer_dn, 0) : nullptr;
    s->cnt_top = cnt;
    s->cnt_bot = cnt + 1;
    s->timed_out = (int *)(cnt + 2);
    unsigned top_rows = 0, bot_rows = 0;         // tile rows in each boundary set: same predicates as the kernel
    for (unsigned by = 0; by < grid.y; ++by) {
        const int y0 = (int)by * TY;
        if (y0 - 2 < 2 * STRIP_GHOST) ++top_rows;
        if (y0 + TY + 2 > ny - 2 * STRIP_GHOST) ++bot_rows;
    }
    s->expect_top = top_rows * grid.x;
    s->expect_bot = bot_rows * grid.x;
    s->base = ctx->strip.epoch << 32;
    s->timeout_ns = (unsigned long long)(ctx->strip.timeout_s * 1e9);
}

// Returns false when the arrays of one kind (depth layers / plane arrays) do not share one member stride (some outputs
// given by the caller, others in the internal scratch): such a step is launched member by member.
bool fill_day_args(nesosim_ctx *ctx, int x, const double *P, const double *C, const double *W, const double *U,
                   const double *V, double rho_new, const nesosim_outputs *o, int m0, bool land_ok, DayArgs &a) {
    bool uniform = true;
    a.depth_mstride = a.plane_mstride = -1;
    a.tile_land = (land_ok && ctx->land_shortcut) ? ctx->tile_land_dev : nullptr;
    a.ny = ctx->cfg.ny;
    a.nx = ctx->cfg.nx;
    a.P = P; a.C = C; a.W = W; a.U = U; a.V = V;
    a.mask = ctx->mask_dev;
    for (int v = 0; v < NVAR; ++v) {
        double *pp, *np_;
        long long ps, ns;
        slot_ptr(ctx, o, v, x, m0, &pp, &ps);
        slot_ptr(ctx, o, v, x + 1, m0, &np_, &ns);
        a.prev[v] = pp;
        a.next[v] = np_;
        if (v == V_DENS && !o->density) continue;        // never read, not stored
        long long &want = (v == V_H0 || v == V_H1) ? a.depth_mstride : a.plane_mstride;
        if (want < 0) want = ns;
        else if (want != ns) uniform = false;
    }
    if (!o->density) a.next[V_DENS] = nullptr;
    a.coef = ctx->coef_dev + m0;
    a.k = ctx->k;
    a.g = ctx->g;
    a.conv_div = ctx->conv_div;
    a.rho_new = ctx->cfg.density_clim ? const_div_host(rho_new) : ctx->rho_fresh_div;
    std::memcpy(a.w, ctx->cfg.conv_weights, sizeof(a.w));
    a.sw = Switches{ctx->cfg.dynamicsInc == 1, ctx->cfg.leadlossInc == 1, ctx->cfg.windpackInc == 1,
                    ctx->cfg.atmlossInc == 1, ctx->cfg.density_clim != 0};
    a.member_set = ctx->member_set_dev ? ctx->member_set_dev + m0 : nullptr;
    a.set_steps = ctx->set_steps_dev;
    a.set_stride = (long long)ctx->cfg.num_days * ctx->plane;
    a.x = x;
    return uniform;
}

int launch_day(nesosim_ctx *ctx, int x, const double *P, const double *C, const double *W, const double *U,
               const double *V, double rho_new, const nesosim_outputs *o, int m0, int mcount, cudaStream_t st,
               bool strip_step = false, bool land_ok = false) {
    // Programmatic launch only behind one of this library's own day kernels of the same call (x > first_step, which is
    // what land_ok says too): the part of a day kernel that runs before griddepcontrol.wait reads forcing, mask and
    // coefficients, and whatever the caller enqueued before the first step (a kernel producing those) must be complete
    // and visible -- an ordinary launch guarantees that.
    const bool pdl = ctx->pdl && land_ok;
    DayArgs a;
    if (!fill_day_args(ctx, x, P, C, W, U, V, rho_new, o, m0, land_ok, a) && mcount > 1) {
        for (int mm = 0; mm < mcount; ++mm) {            // mixed strides: one member per launch, pointers pre-offset
            nesosim_outputs om = *o;
            double **ptrs[] = {&om.snowDepths, &om.density, &om.snowAcc, &om.snowOcean, &om.snowAdv, &om.snowDiv, &om.snowLead,
                               &om.snowAtm, &om.snowWindPackLoss, &om.snowWindPackGain, &om.snowWindPack};
            for (size_t i = 0; i < sizeof(ptrs) / sizeof(ptrs[0]); ++i)
                if (*ptrs[i]) *ptrs[i] += (long long)mm * (i == 0 ? o->depth_member_stride : o->plane_member_stride);
            int rc = launch_day(ctx, x, P, C, W, U, V, rho_new, &om, m0 + mm, 1, st, strip_step, land_ok);
            if (rc) return rc;
        }
        return NESOSIM_OK;
    }
    dim3 grid((a.nx + TX - 1) / TX, (a.ny + TY - 1) / TY, mcount);
    const bool stripped = strip_step && ctx->strip.on && a.sw.dynamics && (ctx->strip.has_up || ctx->strip.has_dn);
    if (stripped) {
        StripLink s;
        strip_link(ctx, x, grid, &s);
        if (ctx->day_variant == 512) CU(launch_day_kernel(day_step_strip_kernel_512, grid, 512, st, pdl, a, s));
        else CU(launch_day_kernel(day_step_strip_kernel, grid, 256, st, pdl, a, s));
    } else if (ctx->day_variant == 512) {
        CU(launch_day_kernel(day_step_kernel_512, grid, 512, st, pdl, a));
    } else {
        CU(launch_day_kernel(day_step_kernel, grid, 256, st, pdl, a));
    }
    ctx->launches++;
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

int launch_init(nesosim_ctx *ctx, const double *ic, int ic_per_member, const double *conc0,
                const nesosim_outputs *o, int m0, int mcount, cudaStream_t st) {
    InitArgs a;
    a.plane = ctx->plane;
    a.ic = (ic && ic_per_member) ? ic + (long long)m0 * ctx->plane : ic;
    a.ic_stride = ic_per_member ? ctx->plane : 0;
    a.conc0 = conc0;
    a.member_set = ctx->member_set_dev ? ctx->member_set_dev + m0 : nullptr;
    a.set_stride = (long long)ctx->cfg.num_days * ctx->plane;
    a.minConc = ctx->cfg.minConc;
    for (int v = 0; v < NVAR; ++v) {
        double *p;
        long long s;
        slot_ptr(ctx, o, v, 0, m0, &p, &s);
        a.slot0[v] = p;
        a.stride[v] = s;
    }
    if (!o->density) a.slot0[V_DENS] = nullptr;
    dim3 grid((unsigned)((ctx->plane + 255) / 256), mcount);
    init_slot0_kernel<<<grid, 256, 0, st>>>(a);
    ctx->launches++;
    CU(cudaGetLastError());
    return NESOSIM_OK;
}


// ------------------------------------------------------------------ season-resident ensemble path (host side)

// Build variants of the season kernel: NTC compute threads (+ one DMA warp), KR raw-list entries and KO owned
// ocean cells per compute thread.  A variant fits a strip decomposition when every strip's lists fit KR*NTC and
// KO*NTC; fewer threads mean more registers per thread (65536 / (NTC+32)).  Order = preference.
struct EnsVariant {
    const char *name;
    int ntc, kr, ko;
    void (*kernel)(const EnsArgs);
    void (*kernel_timing)(const EnsArgs);
    void (*kernel_sets)(const EnsArgs);    // members on different forcing sets (nesosim_set_forcing_sets)
    void (*kernel_obs)(const EnsArgs);     // misfit mode: observations reduced inside the kernel (nesosim_run_season_misfit)
    void (*kernel_obs_sets)(const EnsArgs);   // misfit mode on forcing sets (nesosim_set_observations_sets)
};
#define ENS_V(ntc, kr, ko) \
    {"t" #ntc "r" #kr "o" #ko, ntc, kr, ko, ensemble_season_kernel<ntc, kr, ko, false, false>, ensemble_season_kernel<ntc, kr, ko, true, false>, \
     ensemble_season_kernel<ntc, kr, ko, false, true>, ensemble_season_kernel<ntc, kr, ko, false, false, true>, \
     ensemble_season_kernel<ntc, kr, ko, false, true, true>}
const EnsVariant *ens_variants(int *n) {
    static const EnsVariant v[] = {
        ENS_V(352, 3, 2), ENS_V(224, 4, 3), ENS_V(480, 2, 2), ENS_V(608, 2, 1), ENS_V(480, 2, 1), ENS_V(736, 2, 1), ENS_V(352, 6, 5),
    };
    *n = (int)(sizeof(v) / sizeof(v[0]));
    return v;
}

constexpr size_t ENS_SMEM_CAP = 227 * 1024;

// Cut the grid into `cl` row strips with balanced work and compile the mask into the per-strip cell lists the
// kernel walks.  A strip must satisfy the bulk-copy rules (16-byte aligned start, 16-byte multiple size), hold
// at least ENS_MIN_ROWS rows (its top two and bottom two rows are its neighbours' halos) and fit shared memory.
// Returns false if no such cut exists for this cluster size.
bool try_strip_tables(nesosim_ctx *ctx, int cl, int cap_raw, int cap_ocean, int cap_edge, StripTables &t,
                      std::vector<unsigned short> &codes, size_t &smem_bytes, double &day_cost) {
    const int ny = ctx->cfg.ny, nx = ctx->cfg.nx;
    const std::vector<uint8_t> &mask = ctx->mask_host;
    auto land = [&](int r, int c) { const uint8_t m = mask[(size_t)r * nx + c]; return m > 10 || m < 1; };
    if (ny < ENS_MIN_ROWS * cl) return false;
    // per-row ocean count and count of cells with an ocean cell in their 3x3 neighbourhood
    std::vector<int> oc(ny, 0), dil(ny, 0);
    for (int r = 0; r < ny; ++r)
        for (int c = 0; c < nx; ++c) {
            oc[r] += !land(r, c);
            bool near = false;
            for (int rr = std::max(r - 1, 0); rr <= std::min(r + 1, ny - 1) && !near; ++rr)
                for (int cc = std::max(c - 1, 0); cc <= std::min(c + 1, nx - 1); ++cc)
                    if (!land(rr, cc)) { near = true; break; }
            dil[r] += near;
        }
    std::vector<long long> coc(ny + 1, 0), cdil(ny + 1, 0);
    for (int r = 0; r < ny; ++r) { coc[r + 1] = coc[r] + oc[r]; cdil[r + 1] = cdil[r] + dil[r]; }
    const int max_rows_smem = [&] {   // tallest strip whose tiles fit in shared memory (land list sized generously)
        int best = 0;
        for (int rows = ENS_MIN_ROWS; rows <= ny; ++rows)
            if (ens_layout(rows, nx, rows * nx).total <= ENS_SMEM_CAP) best = rows;
        return best;
    }();
    auto strip_cost = [&](int ra, int rb) -> double {   // < 0: not allowed
        const int rows = rb - ra;
        if (rows < ENS_MIN_ROWS || rows > max_rows_smem) return -1.0;
        if (((long long)rows * nx) % 2 || ((long long)ra * nx) % 2) return -1.0;
        const long long ocean = coc[rb] - coc[ra];
        const long long raw = cdil[std::min(rb + 1, ny)] - cdil[std::max(ra - 1, 0)];   // (upper bound of the list length)
        if (ocean > cap_ocean || raw > cap_raw) return -1.0;
        // relative cost per day: the dynamics phase scales with the raw-list length, the budget phase with the owned
        // ocean cells, the bulk stores with the strip's cells.  NESOSIM_ENS_COST="w_raw,w_ocean,w_cells" overrides
        // the weights (tuning aid).
        double w[3] = {1.0, 0.3, 0.0};
        if (const char *env = getenv("NESOSIM_ENS_COST")) sscanf(env, "%lf,%lf,%lf", &w[0], &w[1], &w[2]);
        return w[0] * raw + w[1] * ocean + w[2] * rows * nx;
    };
    const double INF = 1e300;
    std::vector<std::vector<double>> best(cl + 1, std::vector<double>(ny + 1, INF));
    std::vector<std::vector<int>> from(cl + 1, std::vector<int>(ny + 1, -1));
    best[0][0] = 0.0;
    for (int k = 1; k <= cl; ++k)
        for (int r = ENS_MIN_ROWS * k; r <= ny; ++r)
            for (int q = ENS_MIN_ROWS * (k - 1); q <= r - ENS_MIN_ROWS; ++q) {
                if (best[k - 1][q] >= INF) continue;
                const double c = strip_cost(q, r);
                if (c < 0) continue;
                const double v = std::max(best[k - 1][q], c);
                if (v < best[k][r]) { best[k][r] = v; from[k][r] = q; }
            }
    if (best[cl][ny] >= INF) return false;
    t = StripTables{};
    t.cluster = cl;
    for (int k = cl, r = ny; k >= 1; --k) { t.row0[k] = r; r = from[k][r]; }
    t.row0[0] = 0;
    // NESOSIM_ENS_ROWS="r1,r2,...": put the cl-1 interior strip boundaries at these rows (tests of the halo protocol on
    // masks with all-land rows at a boundary); ignored unless it names a valid cut for this cluster size
    if (const char *env = getenv("NESOSIM_ENS_ROWS")) {
        std::vector<int> rows;
        for (const char *q = env; *q;) {
            char *end;
            const long v = strtol(q, &end, 10);
            if (end == q) break;
            rows.push_back((int)v);
            q = (*end == ',') ? end + 1 : end;
        }
        if ((int)rows.size() == cl - 1) {
            rows.insert(rows.begin(), 0);
            rows.push_back(ny);
            bool ok = true;
            for (int k = 0; k < cl && ok; ++k) ok = rows[k] < rows[k + 1] && strip_cost(rows[k], rows[k + 1]) >= 0;
            if (!ok) return false;
            for (int k = 0; k <= cl; ++k) t.row0[k] = rows[k];
        }
    }
    codes.clear();
    int max_ocean = 0, max_raw = 0, max_rows = 0, max_land = 0, max_edge = 0;
    for (int k = 0; k < cl; ++k) {
        const int ra = t.row0[k], rb = t.row0[k + 1];
        std::vector<unsigned short> ri, re, ocl, la;
        for (int r = std::max(ra - 1, 0); r <= std::min(rb, ny - 1); ++r)
            for (int c = 0; c < nx; ++c) {
                bool needed = false;   // some ocean cell of this strip has (r,c) in its 3x3 neighbourhood
                for (int rr = std::max(r - 1, ra); rr <= std::min(r + 1, rb - 1) && !needed; ++rr)
                    for (int cc = std::max(c - 1, 0); cc <= std::min(c + 1, nx - 1); ++cc)
                        if (!land(rr, cc)) { needed = true; break; }
                if (!needed) continue;
                const bool edge = (r == 0 || r == ny - 1 || c == 0 || c == nx - 1);
                (edge ? re : ri).push_back((unsigned short)(r * 128 + c));
            }
        for (int r = ra; r < rb; ++r)
            for (int c = 0; c < nx; ++c) (land(r, c) ? la : ocl).push_back((unsigned short)((r - ra) * 128 + c));
        auto append = [&](const std::vector<unsigned short> &v, int &off, int &n) {
            while (codes.size() % 8) codes.push_back(0);
            off = (int)codes.size();
            n = (int)v.size();
            codes.insert(codes.end(), v.begin(), v.end());
        };
        t.raw_int_n[k] = (int)ri.size();
        ri.insert(ri.end(), re.begin(), re.end());           // interior entries first, then the edge entries
        append(ri, t.raw_off[k], t.raw_n[k]);
        append(ocl, t.ocean_off[k], t.ocean_n[k]);
        append(la, t.land_off[k], t.land_n[k]);
        // the four halo rows (two above, two below; inside the grid and owned by a neighbour strip): their land
        // cells, as (row of the extended plane)*128 + col, and the bytes their ocean cells receive per day
        std::vector<unsigned short> hl;
        int halo_ocean = 0;
        for (int hr = 0; hr < 4; ++hr) {
            const int r = hr < 2 ? ra - 2 + hr : rb + (hr - 2);
            if ((hr < 2 && k == 0) || (hr >= 2 && k == cl - 1)) continue;
            const int ext_row = r - (ra - 2);
            for (int c = 0; c < nx; ++c) {
                if (land(r, c)) hl.push_back((unsigned short)(ext_row * 128 + c));
                else ++halo_ocean;
            }
        }
        append(hl, t.hland_off[k], t.hland_n[k]);
        t.halo_tx[k] = halo_ocean * 16;
        max_raw = std::max(max_raw, t.raw_int_n[k]);
        max_edge = std::max(max_edge, t.raw_n[k] - t.raw_int_n[k]);
        max_rows = std::max(max_rows, rb - ra);
        max_land = std::max(max_land, (int)la.size());
        max_ocean = std::max(max_ocean, (int)ocl.size());
    }
    codes.push_back(0);
    t.rows_alloc = max_rows;
    t.raw_max = max_raw;
    t.ocean_max = max_ocean;
    t.land_alloc = max_land;
    smem_bytes = ens_layout(max_rows, nx, max_land).total;
    if (smem_bytes > ENS_SMEM_CAP) return false;
    if (max_edge > cap_edge) return false;   // (one edge entry per thread)
    day_cost = best[cl][ny];
    return true;
}

int max_active_clusters(const EnsVariant *v, int cl, size_t smem_bytes) {
    if (cudaFuncSetAttribute((const void *)v->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    if (cl > 8) cudaFuncSetAttribute((const void *)v->kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cfg.blockDim = dim3(v->ntc + 32);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.gridDim = dim3(cl * 64);
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, (const void *)v->kernel, &cfg) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// Choose the cluster size (CTAs per member) and the build variant: every size whose strips fit in shared memory is
// costed as rounds(members / co-resident clusters) x (heaviest strip + fixed per-day overhead), the cheapest wins;
// the variant is the first in preference order whose per-thread capacities hold the strips' lists.
int build_strip_tables(nesosim_ctx *ctx) {
    EnsembleState &e = ctx->ens;
    if (e.tables_ready) return NESOSIM_OK;
    int forced = 0;
    if (const char *env = getenv("NESOSIM_ENS_CLUSTER")) forced = atoi(env);
    const char *forced_var = getenv("NESOSIM_ENS_VARIANT");
    int nv;
    const EnsVariant *vars = ens_variants(&nv);
    std::vector<unsigned short> best_codes;
    double best_time = 1e300;
    for (int vi = 0; vi < nv; ++vi) {
        if (forced_var && *forced_var && strcmp(forced_var, vars[vi].name)) continue;
        bool found = false;
        for (int cl = 2; cl <= ENS_MAX_CLUSTER; ++cl) {
            if (forced && cl != forced) continue;
            StripTables t;
            std::vector<unsigned short> codes;
            size_t smem = 0;
            double day_cost = 0;
            if (!try_strip_tables(ctx, cl, vars[vi].kr * vars[vi].ntc, vars[vi].ko * vars[vi].ntc, vars[vi].ntc, t, codes, smem, day_cost)) continue;
            const int ncl = max_active_clusters(&vars[vi], cl, smem);
            if (ncl < 1) continue;
            const int rounds = (ctx->cfg.n_members + ncl - 1) / ncl;
            const double time = rounds * (day_cost + 1500.0);   // heaviest strip + fixed barrier overhead per day
            if (time < best_time) {
                best_time = time;
                e.tables = t;
                e.smem_bytes = smem;
                e.max_clusters = ncl;
                e.variant = vi;
                best_codes.swap(codes);
                found = true;
            }
        }
        if (found) break;   // variants are listed in order of preference: the first one that fits wins
    }
    if (best_time >= 1e300) return fail(NESOSIM_ERR_ARG, "grid does not fit the season-resident kernel's shared-memory strips");
    CU(cudaMalloc(&e.codes_dev, best_codes.size() * sizeof(unsigned short)));
    CU(cudaMemcpy(e.codes_dev, best_codes.data(), best_codes.size() * sizeof(unsigned short), cudaMemcpyHostToDevice));
    e.tables.codes = e.codes_dev;
    e.tables_ready = true;
    return NESOSIM_OK;
}

// The kernel keeps a whole member on one cluster of 2..8 CTAs: rows of at most 96 columns, strips that fit in
// shared memory, 16-byte aligned planes for the bulk stores.
bool ensemble_eligible(nesosim_ctx *ctx, int first_step, int num_steps, const nesosim_outputs *out, const char **why) {
    const nesosim_config &c = ctx->cfg;
    if (ctx->strip.on) { *why = "strip of a decomposed grid"; return false; }
    if (c.nx > ENS_MAX_NX) { *why = "nx > 96"; return false; }
    if (c.nx < 3) { *why = "nx < 3"; return false; }
    if (c.ny < 2 * ENS_MIN_ROWS) { *why = "ny < 8"; return false; }
    if (c.ny > 511) { *why = "ny > 511 (cell codes are row*128+col in 16 bits)"; return false; }
    if (((long long)c.ny * c.nx) % 2) { *why = "odd number of cells (bulk stores need 16-byte aligned planes)"; return false; }
    if (c.density_clim) { *why = "densityType='clim'"; return false; }
    if (first_step != 0 || num_steps != c.num_days - 1) { *why = "partial season"; return false; }
    for (int v = 0; v < NVAR; ++v)
        if (out_base(out, v) && ((uintptr_t)out_base(out, v) % 16)) { *why = "output array not 16-byte aligned"; return false; }
    if ((out->depth_member_stride % 2) || (out->plane_member_stride % 2)) { *why = "odd member stride"; return false; }
    if (!(ctx->g.dx.fast && ctx->g.two_dx.fast && ctx->conv_div.fast)) { *why = "a divisor without the exact fast-division proof"; return false; }
    if (!(c.dx >= 1.0 && c.dx <= 536870912.0)) { *why = "dx outside [1, 2^29] m"; return false; }
    for (int i = 0; i < 9; ++i) {
        const double w = std::fabs(c.conv_weights[i]);
        if (!(w == 0.0 || (w >= 9.5367431640625e-07 && w <= 1048576.0))) { *why = "kernel weight outside [2^-20, 2^20]"; return false; }
    }
    if (!(std::fabs(c.conv_divisor) >= 9.5367431640625e-07 && std::fabs(c.conv_divisor) <= 1048576.0)) { *why = "kernel divisor outside [2^-20, 2^20]"; return false; }
    if (build_strip_tables(ctx) != NESOSIM_OK) { *why = "no strip decomposition fits"; return false; }
    return true;
}

struct ObsDevice {                      // misfit mode: device arrays of the sample slots (see EnsArgs)
    const int *first = nullptr, *day = nullptr;
    double2 *sample_hh = nullptr;
    long long sample_stride = 0;
    long long first_stride = 0;         // forcing sets: per-set tables
    const int *slot_base = nullptr;
};

int run_ensemble(nesosim_ctx *ctx, const double *ic_dev, int ic_per_member, const nesosim_outputs *out, int m0,
                 int mcount, cudaStream_t st, const ObsDevice *obs = nullptr) {
    const nesosim_config &c = ctx->cfg;
    const long long plane = ctx->plane;
    const int steps = c.num_days - 1;
    EnsembleState &e = ctx->ens;
    const size_t cells = (size_t)steps * plane * ctx->n_sets;
    const size_t need = cells * (2 + 1 + 1) * sizeof(double2);
    if (e.derived_bytes < need) {
        cudaFree(e.derived);
        e.derived = nullptr;
        e.derived_bytes = 0;
        CU(cudaMalloc(&e.derived, need));
        e.derived_bytes = need;
    }
    double2 *DA = (double2 *)e.derived, *DB = DA + 2 * cells;
    double *cumAcc = (double *)(DB + cells), *cumOc = cumAcc + cells;
    // member-independent pre-pass: part of the season, recomputed on every call
    DeriveArgs d;
    d.ny = c.ny; d.nx = c.nx; d.steps = steps; d.T = c.num_days; d.sets = ctx->n_sets;
    d.P = ctx->P; d.C = ctx->C; d.UV = ctx->UV;
    d.DA = DA; d.DB = DB; d.cumAcc = cumAcc; d.cumOc = cumOc;
    d.k = ctx->k; d.g = ctx->g; d.rho_new = ctx->rho_fresh_div;
    d.status = ctx->flags_dev;
    CU(cudaMemsetAsync(ctx->flags_dev, 0, sizeof(int), st));
    dim3 blk(32, 8), grid((c.nx + 31) / 32, (c.ny + 7) / 8, steps * ctx->n_sets);
    derive_pointwise_kernel<<<grid, blk, 0, st>>>(d);
    derive_scan_kernel<<<(unsigned)((plane * ctx->n_sets + 63) / 64), 64, 0, st>>>(DB, cumAcc, cumOc, plane, steps, ctx->n_sets);
    ctx->launches += 2;
    CU(cudaGetLastError());

    int nv_;
    const EnsVariant *v = &ens_variants(&nv_)[e.variant];
    const int cl = e.tables.cluster;
    const bool dbg_timing = getenv("NESOSIM_ENS_TIMING") != nullptr;   // debug aid: per-phase cycle totals to stderr
    void (*kernel)(const EnsArgs) = obs ? (ctx->member_set_dev ? v->kernel_obs_sets : v->kernel_obs)
                                        : ctx->member_set_dev ? v->kernel_sets : (dbg_timing ? v->kernel_timing : v->kernel);
    CU(cudaFuncSetAttribute((const void *)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e.smem_bytes));
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cfg.blockDim = dim3(v->ntc + 32);
    cfg.dynamicSmemBytes = e.smem_bytes;
    cfg.stream = st;
    int max_clusters = e.max_clusters;
    if (max_clusters < 1) return fail(NESOSIM_ERR_CUDA, "no cluster of this size fits on the device");
    if (const char *envc = getenv("NESOSIM_ENS_CLUSTERS")) max_clusters = std::max(1, std::min(max_clusters, atoi(envc)));
    const int ncl = std::min(max_clusters, mcount);

    EnsArgs a;
    a.ny = c.ny; a.nx = c.nx; a.T = c.num_days; a.M = mcount;
    a.DA = DA; a.DB = DB; a.cumAcc = cumAcc; a.cumOc = cumOc;
    a.W = ctx->W;
    a.ic = (ic_dev && ic_per_member) ? ic_dev + (long long)m0 * plane : ic_dev;
    a.ic_stride = ic_per_member ? plane : 0;
    a.conc0 = ctx->C;
    a.member_set = ctx->member_set_dev ? ctx->member_set_dev + m0 : nullptr;
    a.set_steps = ctx->set_steps_dev;
    for (int vv = 0; vv < NVAR; ++vv) {
        double *base = out_base(out, vv);
        a.out[vv] = base ? base + (vv == V_H1 ? plane : 0) : nullptr;
        a.mstride[vv] = (vv == V_H0 || vv == V_H1) ? out->depth_member_stride : out->plane_member_stride;
    }
    a.coef = ctx->coef_dev + m0;
    a.k = ctx->k; a.g = ctx->g; a.conv_div = ctx->conv_div;
    std::memcpy(a.w, c.conv_weights, sizeof(a.w));
    a.sw = Switches{c.dynamicsInc == 1, c.leadlossInc == 1, c.windpackInc == 1, c.atmlossInc == 1, 0};
    a.st = e.tables;
    a.status = ctx->flags_dev;
    a.obs_first = obs ? obs->first : nullptr;
    a.obs_day = obs ? obs->day : nullptr;
    a.sample_hh = obs ? obs->sample_hh : nullptr;
    a.sample_stride = obs ? obs->sample_stride : 0;
    a.obs_first_stride = obs ? obs->first_stride : 0;
    a.obs_slot_base = obs ? obs->slot_base : nullptr;
    a.dbg = getenv("NESOSIM_ENS_DBG") ? atoi(getenv("NESOSIM_ENS_DBG")) : 0;
    a.timing = nullptr;
    if (dbg_timing && !ctx->member_set_dev && !obs) {
        CU(cudaMalloc(&a.timing, sizeof(long long) * ENS_NTIMER * ncl * cl));
        CU(cudaMemset(a.timing, 0, sizeof(long long) * ENS_NTIMER * ncl * cl));
    }
    cfg.gridDim = dim3(ncl * cl);
    if (!ctx->ens_ev[0]) {
        CU(cudaEventCreate(&ctx->ens_ev[0]));
        CU(cudaEventCreate(&ctx->ens_ev[1]));
    }
    CU(cudaEventRecord(ctx->ens_ev[0], st));
    CU(cudaLaunchKernelEx(&cfg, kernel, a));
    CU(cudaEventRecord(ctx->ens_ev[1], st));
    ctx->launches++;
    CU(cudaGetLastError());
    // The kernel only carries the fast divisions; if an operand left their proven range the season is redone by
    // the general kernels (run_members looks at ens_status).  Reading the flag needs the stream to finish.
    if (ctx->async_mode && !dbg_timing && !obs) {
        // Asynchronous mode: the flag travels to pinned host memory behind the kernel and is looked at by nesosim_sync
        // (or by a later call, without waiting).  The launch keeps its own pair of timing events.
        PendingSeason p;
        p.ev0 = ctx->ens_ev[0];
        p.ev1 = ctx->ens_ev[1];
        ctx->ens_ev[0] = ctx->ens_ev[1] = nullptr;
        CU(cudaEventCreateWithFlags(&p.done, cudaEventDisableTiming));
        p.flag_host = ctx->flag_pool + (ctx->flag_next++ % 256);      // (at most 64 seasons are ever pending)
        *p.flag_host = 0;
        CU(cudaMemcpyAsync(p.flag_host, ctx->flags_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(p.done, st));
        p.ic_dev = ic_dev; p.ic_per_member = ic_per_member; p.m0 = m0; p.mcount = mcount; p.out = *out;
        p.params = ctx->last_params;
        p.stream = st;
        ctx->pending.push_back(std::move(p));
        ctx->ens_status = 0;
        return NESOSIM_OK;
    }
    CU(cudaMemcpyAsync(&ctx->ens_status, ctx->flags_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ens_ev[0], ctx->ens_ev[1]) == cudaSuccess) {
            ctx->ens_kernel_ms += ms;
            ctx->ens_kernel_launches++;
        }
    }
    if (dbg_timing && !ctx->member_set_dev && !obs) {
        std::vector<long long> h(ENS_NTIMER * ncl * cl);
        CU(cudaMemcpy(h.data(), a.timing, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        cudaFree(a.timing);
        static const char *names[12] = {"A", "barA", "Bcompute", "clwait1", "drain", "publish", "barStore", "halowait",
                                        "dma:drain", "dma:arrive", "dma:wait_compute", "dma:issue"};
        const double days = (double)(c.num_days - 1) * ((mcount + ncl - 1) / ncl);
        for (int kk = 0; kk < cl; ++kk) {
            fprintf(stderr, "[ens timing] %s cluster=%d x %d smem=%zu strip %d rows %d ocean %d land %d raw %d | cycles/day:", v->name, cl,
                    ncl, e.smem_bytes, kk, e.tables.row0[kk + 1] - e.tables.row0[kk], e.tables.ocean_n[kk], e.tables.land_n[kk],
                    e.tables.raw_n[kk]);
            for (int q = 0; q < 12; ++q) fprintf(stderr, " %s=%.0f", names[q], h[kk * ENS_NTIMER + q] / days);
            fprintf(stderr, "\n[ens timing]   strip %d per-warp A:", kk);
            for (int w = 0; w < v->ntc / 32 && w < 24; ++w) fprintf(stderr, " %.0f", h[kk * ENS_NTIMER + 16 + w] / days);
            fprintf(stderr, "\n[ens timing]   strip %d per-warp B:", kk);
            for (int w = 0; w < v->ntc / 32 && w < 24; ++w) fprintf(stderr, " %.0f", h[kk * ENS_NTIMER + 40 + w] / days);
            fprintf(stderr, "\n");
        }
    }
    return NESOSIM_OK;
}

int run_members(nesosim_ctx *ctx, const double *ic_dev, int ic_per_member, const nesosim_outputs *out, int m0,
                int mcount, int first_step, int num_steps, cudaStream_t st);

void pending_release(PendingSeason &p) {
    if (p.ev0) cudaEventDestroy(p.ev0);
    if (p.ev1) cudaEventDestroy(p.ev1);
    if (p.done) cudaEventDestroy(p.done);
    p.ev0 = p.ev1 = p.done = nullptr;
    p.flag_host = nullptr;
}

// Look at the flags of the asynchronous season launches that have finished (`block`: wait for all of them).  A season
// whose operands left the fast divisions' range is redone by the general kernels here, as the synchronous mode does
// inside nesosim_run_season.  Returns the number of seasons redone through *redone.
int resolve_pending(nesosim_ctx *ctx, bool block, int *redone) {
    size_t keep = 0;
    for (size_t i = 0; i < ctx->pending.size(); ++i) {
        PendingSeason &p = ctx->pending[i];
        cudaError_t e = block ? cudaEventSynchronize(p.done) : cudaEventQuery(p.done);
        if (e == cudaErrorNotReady) {
            cudaGetLastError();
            if (keep != i) ctx->pending[keep] = std::move(p);
            ++keep;
            continue;
        }
        if (e != cudaSuccess) return cuda_fail(e, "waiting for an asynchronous season");
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.ev0, p.ev1) == cudaSuccess) {
            ctx->ens_kernel_ms += ms;
            ctx->ens_kernel_launches++;
        }
        const int flag = *p.flag_host;
        if (flag) {
            ctx->ens_reruns++;
            if (redone) ++*redone;
            const int saved = ctx->path;
            ctx->path = 1;
            int rc = upload_coef(ctx, p.params.data(), p.stream);
            if (!rc) rc = run_members(ctx, p.ic_dev, p.ic_per_member, &p.out, p.m0, p.mcount, 0, -1, p.stream);
            ctx->path = saved;
            if (rc) return rc;
            CU(cudaStreamSynchronize(p.stream));
        }
        pending_release(p);
    }
    ctx->pending.resize(keep);
    return NESOSIM_OK;
}

// Steps first_step .. first_step+num_steps-1 for members [m0, m0+mcount); `out` addresses member m0.
int run_members(nesosim_ctx *ctx, const double *ic_dev, int ic_per_member, const nesosim_outputs *out, int m0,
                int mcount, int first_step, int num_steps, cudaStream_t st) {
    const int T = ctx->cfg.num_days;
    if (num_steps < 0) num_steps = T - 1 - first_step;
    if (first_step < 0 || first_step + num_steps > T - 1) return fail(NESOSIM_ERR_ARG, "step range outside the season");
    int rc;
    const char *why = "";
    const bool can_ens = ensemble_eligible(ctx, first_step, num_steps, out, &why);
    if (ctx->path == 2 && !can_ens)
        return fail(NESOSIM_ERR_ARG, std::string("season-resident ensemble path not applicable: ") + why);
    if (ctx->path != 1 && can_ens) {
        ctx->last_path = 2;
        rc = run_ensemble(ctx, ic_dev, ic_per_member, out, m0, mcount, st);
        if (rc || !ctx->ens_status) return rc;
        ctx->ens_reruns++;          // fall through: redo these members with the general kernels
    }
    ctx->last_path = 1;
    if (any_missing(out) && (rc = ensure_scratch(ctx))) return rc;
    if (first_step == 0 && (rc = launch_init(ctx, ic_dev, ic_per_member, ctx->C, out, m0, mcount, st))) return rc;
    const long long plane = ctx->plane;
    if (ctx->strip.on) {
        if ((ctx->strip.has_up && !ctx->strip.peer_up) || (ctx->strip.has_dn && !ctx->strip.peer_dn))
            return fail(NESOSIM_ERR_STATE, "strip neighbours are not connected (nesosim_strip_connect*)");
        if (first_step == 0) ctx->strip.epoch++;       // every strip counts its seasons the same way: flags only grow
    }
    for (int x = first_step; x < first_step + num_steps; ++x) {
        const double rho = ctx->cfg.density_clim ? ctx->rho_clim_host[x] : ctx->cfg.snowDensityFresh;
        rc = launch_day(ctx, x, ctx->P + x * plane, ctx->C + x * plane, ctx->W + x * plane,
                        ctx->UV + (long long)x * 2 * plane, ctx->UV + ((long long)x * 2 + 1) * plane, rho, out,
                        m0, mcount, st, true, x > first_step);
        if (rc) return rc;
    }
    return NESOSIM_OK;
}

}  // namespace

extern "C" {

int nesosim_abi_version(void) { return NESOSIM_ABI_VERSION; }
const char *nesosim_last_error(void) { return g_err.c_str(); }

int nesosim_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int nesosim_create(const nesosim_config *cfg, const uint8_t *region_mask_host, nesosim_ctx **out) {
    if (!cfg || !region_mask_host || !out) return fail(NESOSIM_ERR_ARG, "NULL argument");
    if (cfg->ny < 2 || cfg->nx < 2) return fail(NESOSIM_ERR_ARG, "ny and nx must be >= 2 (np.gradient needs two points)");
    if (cfg->num_days < 2) return fail(NESOSIM_ERR_ARG, "num_days must be >= 2");
    if (cfg->n_members < 1 || cfg->n_members > 65535) return fail(NESOSIM_ERR_ARG, "n_members must be in [1, 65535]");
    if (!(cfg->dx > 0) || !(cfg->deltaT > 0)) return fail(NESOSIM_ERR_ARG, "dx and deltaT must be positive");
    if (!(cfg->conv_divisor != 0)) return fail(NESOSIM_ERR_ARG, "conv_divisor must be non-zero");
    if (nesosim_device_count() <= cfg->device || cfg->device < 0)
        return fail(NESOSIM_ERR_CUDA, "no such CUDA device (this library has no CPU path)");
    CU(cudaSetDevice(cfg->device));
    nesosim_ctx *ctx = new (std::nothrow) nesosim_ctx();
    if (!ctx) return fail(NESOSIM_ERR_NOMEM, "out of host memory");
    ctx->cfg = *cfg;
    ctx->plane = (long long)cfg->ny * cfg->nx;
    ctx->mask_host.assign(region_mask_host, region_mask_host + (size_t)cfg->ny * cfg->nx);
    ctx->k = ModelConsts{cfg->deltaT, cfg->snowDensityFresh, cfg->snowDensityOld,
                         cfg->snowDensityFresh / cfg->snowDensityOld, cfg->minSnowD, cfg->minConc};
    ctx->g.dx = const_div_host(cfg->dx);
    ctx->g.two_dx = const_div_host(2. * cfg->dx);
    ctx->conv_div = const_div_host(cfg->conv_divisor);
    ctx->rho_fresh_div = const_div_host(cfg->snowDensityFresh);
    cudaError_t e = cudaMalloc(&ctx->mask_dev, ctx->plane);
    if (e == cudaSuccess) e = cudaMemcpy(ctx->mask_dev, region_mask_host, ctx->plane, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->coef_dev, sizeof(MemberCoef) * cfg->n_members);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->flags_dev, sizeof(int));
    // day-kernel tiles without an ocean cell (land: code > 10, lakes: code < 1; fill_nan_no_negative, NESOSIM.py:158-162)
    const int tgx = (cfg->nx + TX - 1) / TX, tgy = (cfg->ny + TY - 1) / TY;
    std::vector<uint8_t> tl((size_t)tgx * tgy, 1);
    for (int y = 0; y < cfg->ny; ++y)
        for (int x = 0; x < cfg->nx; ++x) {
            const uint8_t c = region_mask_host[(size_t)y * cfg->nx + x];
            if (!(c > 10 || c < 1)) tl[(size_t)(y / TY) * tgx + x / TX] = 0;
        }
    if (e == cudaSuccess) e = cudaMalloc(&ctx->tile_land_dev, tl.size());
    if (e == cudaSuccess) e = cudaMemcpy(ctx->tile_land_dev, tl.data(), tl.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        nesosim_destroy(ctx);
        return cuda_fail(e, "nesosim_create allocation");
    }
    // CTA shape and land shortcut by the number of CTAs per day (measured on a B200, tools/general_timing.py,
    // profiles/r01_general_path_variants*.jsonl): a day of one wave or less is as long as the dependent chain inside one
    // CTA -- 512 threads x 1 cell shorten it when an SM holds a single CTA (100 km: 8.2 -> 7.7 us/day); with about two
    // CTAs per SM 256 threads x 2 cells are faster (25 km: 9.5 vs 12.4 us/day); with many waves throughput counts and
    // the two shapes tie (5 km: 171 us/day).  The land-tile shortcut is looked up before the programmatic-launch wait,
    // so it costs nothing on the chain and is on whenever there is more than one CTA per SM.
    {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
        const long long ctas = (long long)tgx * tgy * cfg->n_members;
        if (ctas <= sms) { ctx->day_variant = 512; ctx->land_shortcut = false; }
        else if (ctas >= 8LL * sms) { ctx->day_variant = 512; ctx->land_shortcut = true; }
        else { ctx->day_variant = 256; ctx->land_shortcut = true; }
    }
    // development switches for A/B timing (both settings of each produce identical values)
    if (const char *v = std::getenv("NESOSIM_DAY_THREADS")) ctx->day_variant = std::atoi(v) == 512 ? 512 : 256;
    if (const char *v = std::getenv("NESOSIM_LAND_SHORTCUT")) ctx->land_shortcut = std::atoi(v) != 0;
    if (const char *v = std::getenv("NESOSIM_PDL")) ctx->pdl = std::atoi(v) != 0;
    *out = ctx;
    return NESOSIM_OK;
}

int nesosim_destroy(nesosim_ctx *ctx) {
    if (!ctx) return NESOSIM_OK;
    cudaSetDevice(ctx->cfg.device);
    ensemble_release(ctx->ens);
    for (auto &p : ctx->pending) {
        if (p.done) cudaEventSynchronize(p.done);
        pending_release(p);
    }
    ctx->pending.clear();
    if (ctx->flag_pool) cudaFreeHost(ctx->flag_pool);
    obs_release(ctx);
    for (int i = 0; i < 2; ++i)
        if (ctx->ens_ev[i]) cudaEventDestroy(ctx->ens_ev[i]);
    strip_release(ctx);
    cudaFree(ctx->tile_land_dev);
    cudaFree(ctx->mask_dev);
    cudaFree(ctx->coef_dev);
    cudaFree(ctx->scratch);
    cudaFree(ctx->flags_dev);
    cudaFree(ctx->member_set_dev);
    cudaFree(ctx->set_steps_dev);
    cudaFree(ctx->hp.forcing);
    cudaFree(ctx->hp.ic);
    for (int i = 0; i < 2; ++i) {
        cudaFree(ctx->hp.outbuf[i]);
        if (ctx->hp.done[i]) cudaEventDestroy(ctx->hp.done[i]);
        if (ctx->hp.drained[i]) cudaEventDestroy(ctx->hp.drained[i]);
    }
    if (ctx->hp.shared_ready) cudaEventDestroy(ctx->hp.shared_ready);
    for (int i = 0; i < 2; ++i) cudaFree(ctx->hp.packed[i]);
    if (ctx->hp.ring) cudaFreeHost(ctx->hp.ring);
    for (cudaEvent_t e : ctx->hp.arrived) cudaEventDestroy(e);
    cudaFree(ctx->hp.cells_dev);
    cudaFree(ctx->hp.chunk_flags);
    if (ctx->hp.compute) cudaStreamDestroy(ctx->hp.compute);
    if (ctx->hp.copy) cudaStreamDestroy(ctx->hp.copy);
    delete ctx;
    return NESOSIM_OK;
}

int nesosim_set_forcing(nesosim_ctx *ctx, const double *precip_dev, const double *conc_dev,
                        const double *wind_dev, const double *drift_dev, const double *rho_clim_dev) {
    if (!ctx || !precip_dev || !conc_dev || !wind_dev || !drift_dev) return fail(NESOSIM_ERR_ARG, "NULL forcing pointer");
    if (ctx->cfg.density_clim && !rho_clim_dev) return fail(NESOSIM_ERR_ARG, "density_clim=1 needs rho_clim");
    CU(cudaSetDevice(ctx->cfg.device));
    ctx->P = precip_dev; ctx->C = conc_dev; ctx->W = wind_dev; ctx->UV = drift_dev; ctx->rho_clim = rho_clim_dev;
    ctx->rho_clim_host.clear();
    if (ctx->cfg.density_clim) {
        ctx->rho_clim_host.resize(ctx->cfg.num_days);
        CU(cudaMemcpy(ctx->rho_clim_host.data(), rho_clim_dev, sizeof(double) * ctx->cfg.num_days, cudaMemcpyDeviceToHost));
    }
    ctx->ens.derived_valid = false;
    ctx->n_sets = 1;
    ctx->set_days.clear();
    cudaFree(ctx->member_set_dev);
    cudaFree(ctx->set_steps_dev);
    ctx->member_set_dev = ctx->set_steps_dev = nullptr;
    return NESOSIM_OK;
}

int nesosim_set_forcing_sets(nesosim_ctx *ctx, int n_sets, const double *precip_dev, const double *conc_dev,
                             const double *wind_dev, const double *drift_dev, const int32_t *member_set_host,
                             const int32_t *set_days_host) {
    if (!ctx || !member_set_host || !set_days_host || n_sets < 1) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (ctx->cfg.density_clim) return fail(NESOSIM_ERR_ARG, "forcing sets support densityType='variable' only");
    int rc = nesosim_set_forcing(ctx, precip_dev, conc_dev, wind_dev, drift_dev, nullptr);
    if (rc) return rc;
    const int M = ctx->cfg.n_members, T = ctx->cfg.num_days;
    std::vector<int> steps(n_sets);
    for (int s = 0; s < n_sets; ++s) {
        if (set_days_host[s] < 2 || set_days_host[s] > T) return fail(NESOSIM_ERR_ARG, "set_days must be in [2, num_days]");
        steps[s] = set_days_host[s] - 1;
    }
    for (int m = 0; m < M; ++m)
        if (member_set_host[m] < 0 || member_set_host[m] >= n_sets) return fail(NESOSIM_ERR_ARG, "member_set entry outside [0, n_sets)");
    CU(cudaMalloc(&ctx->member_set_dev, sizeof(int) * M));
    CU(cudaMalloc(&ctx->set_steps_dev, sizeof(int) * n_sets));
    CU(cudaMemcpy(ctx->member_set_dev, member_set_host, sizeof(int) * M, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->set_steps_dev, steps.data(), sizeof(int) * n_sets, cudaMemcpyHostToDevice));
    ctx->n_sets = n_sets;
    ctx->set_days.assign(set_days_host, set_days_host + n_sets);
    return NESOSIM_OK;
}

int nesosim_run_season(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                       int ic_per_member, const nesosim_outputs *out, int first_step, int num_steps,
                       void *stream) {
    if (!ctx || !params_host) return fail(NESOSIM_ERR_ARG, "NULL argument");
    if (!ctx->P) return fail(NESOSIM_ERR_STATE, "nesosim_set_forcing has not been called");
    int rc = check_outputs(ctx, out);
    if (rc) return rc;
    CU(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    if (ctx->async_mode) {
        ctx->last_params.assign(params_host, params_host + ctx->cfg.n_members);
        if ((rc = resolve_pending(ctx, ctx->pending.size() >= 64, nullptr))) return rc;   // finished ones only, unless the list is long
    }
    if ((rc = upload_coef(ctx, params_host, st))) return rc;
    return run_members(ctx, ic_dev, ic_per_member, out, 0, ctx->cfg.n_members, first_step, num_steps, st);
}

}  // extern "C"

// Epilogue of the misfit mode: one CTA per member.  The sample {h0, h1} of an observation's slot gives the model value of
// its kind: depth over ice (h0+h1)/iceConc of that day and cell (what main writes as snow depth, NESOSIM.py:654), volume
// h0+h1, or the bulk density densityCalc(h0, h1) (NESOSIM.py:458-473).  The terms ((model - observed)/sigma)^2 of a kind
// are summed in a fixed order over that kind's contiguous range of observations (observation i of the range belongs to
// thread i % 256, threads are combined by shuffles, warps one after the other): each kind's sum is formed exactly as if
// it had been registered alone.  SETS: member m is scored against the observations of its forcing set member_set[m], on
// that set's concentration stack, exactly as for its season on its own.
struct MisfitArgs {
    const double2 *samples;         // [M][stride]
    long long stride;
    const int *obs_slot, *obs_day, *obs_cell, *src;
    const double *obs_val, *sigma;
    const int *kind_begin;          // [sets][NESOSIM_OBS_KINDS+1]
    const double *conc;             // [T][plane] (SETS: [sets][T][plane])
    long long plane;
    ModelConsts k;
    double *chi2;                   // [M][n_kinds]
    long long *count;               // same shape, or NULL
    int n_kinds;                    // kinds reported: NESOSIM_OBS_KINDS, or 1 (depth only, nesosim_run_season_misfit)
    double *model;                  // [M][model_stride]: the model value at every observation's input index, or NULL
    long long model_stride;
    const int *member_set;          // SETS only
    long long conc_set_stride;      // SETS only: T * plane
    // footprint stage (nesosim_run_season_scores_fp), skipped when fp_chi2 is NULL: the footprint means of
    // footprint_mean_kernel scored per kind exactly as the point observations
    const double *fp_mean;          // [M][fp_stride] in table order within the member's set
    long long fp_stride;
    const double *fp_val, *fp_sigma;
    const int *fp_kind_begin;       // [sets][NESOSIM_OBS_KINDS+1]
    double *fp_chi2;                // [M][NESOSIM_OBS_KINDS] or NULL
    long long *fp_count;            // same shape, or NULL
};

// The fixed-order block total of the thread partial sums (acc, cnt): shuffle-down tree per warp, then the 8 warps one
// after the other; thread 0 gets the result.  Ends with a barrier, so red / redc can be reused at once.
__device__ __forceinline__ void block_total(double acc, long long cnt, double *red, long long *redc, double *total,
                                            long long *total_count) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        acc = add(acc, __shfl_down_sync(0xffffffffu, acc, off));
        cnt += __shfl_down_sync(0xffffffffu, cnt, off);
    }
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = acc; redc[threadIdx.x >> 5] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        long long n = 0;
        for (int w = 0; w < 8; ++w) { t = add(t, red[w]); n += redc[w]; }
        *total = t;
        if (total_count) *total_count = n;
    }
    __syncthreads();
}

// Gradient stage of the epilogue (misfit_finish_grad_kernel, nesosim_run_season_score_grads): the tangent samples give
// each observation's derivative dv in GRAD_DIRS directions (density_tangent for density), NaN where v is not finite;
// per kind and direction the terms 2 r (dv / sigma) of the observations chi2 counts are summed in chi2's order.
struct MisfitGrad {
    const double2 *tsamples;        // [M][GRAD_DIRS][stride] {t0, t1}
    double *grad;                   // [M][NESOSIM_OBS_KINDS][GRAD_DIRS]
    double *jac;                    // [M][GRAD_DIRS][jac_stride] at the input index, or NULL
    long long jac_stride;
    const double *fp_dmean;         // [M][GRAD_DIRS][fp_stride] footprint mean derivatives (footprint_mean_grad_kernel)
    double *fp_grad;                // [M][NESOSIM_OBS_KINDS][GRAD_DIRS] (read only with the footprint stage)
};

// d(densityCalc)/dtheta at a sample from the primal quotient q and den = h0 + h1 (quotient rule), 0 where a clamp set q
__device__ __forceinline__ double density_tangent(double h0, double h1, double t0, double t1, const ModelConsts &k) {
    const double den = add(h0, h1);
    const double q = div_ieee(add(mul(h0, k.rhoFresh), mul(h1, k.rhoOld)), den);
    if (q > k.rhoOld || q < k.rhoFresh) return 0.0;
    return div_ieee(sub(add(mul(t0, k.rhoFresh), mul(t1, k.rhoOld)), mul(q, add(t0, t1))), den);
}

__device__ __forceinline__ double obs_tangent(int kind, double2 h, double2 t, double C, const ModelConsts &k) {
    if (kind == NESOSIM_OBS_DEPTH) return div_ieee(add(t.x, t.y), C);
    if (kind == NESOSIM_OBS_VOLUME) return add(t.x, t.y);
    return density_tangent(h.x, h.y, t.x, t.y, k);
}

template <bool SETS, bool GRAD>
__device__ __forceinline__ void misfit_finish(const MisfitArgs &a, const MisfitGrad *g) {
    const int m = blockIdx.x;
    const double2 *samp = a.samples + (long long)m * a.stride;
    const int set = SETS ? a.member_set[m] : 0;
    const int *kb = a.kind_begin + set * (NESOSIM_OBS_KINDS + 1);
    const double *conc = SETS ? a.conc + (long long)set * a.conc_set_stride : a.conc;
    double *model = a.model ? a.model + (long long)m * a.model_stride : nullptr;
    __shared__ double red[8];
    __shared__ long long redc[8];
    for (int kind = 0; kind < a.n_kinds; ++kind) {
        const long long i0 = kb[kind], n_obs = (long long)kb[kind + 1] - i0;
        double acc = 0.0, gacc[GRAD_DIRS] = {0.0, 0.0, 0.0};
        long long cnt = 0;
        for (long long i = threadIdx.x; i < n_obs; i += 256) {
            const long long q = i0 + i;
            const double2 h = samp[a.obs_slot[q]];
            double v;
            if (kind == NESOSIM_OBS_DEPTH) v = div_ieee(add(h.x, h.y), __ldg(conc + (long long)a.obs_day[q] * a.plane + a.obs_cell[q]));
            else if (kind == NESOSIM_OBS_VOLUME) v = add(h.x, h.y);
            else v = density_variable(h.x, h.y, false, a.k);
            if (model) model[a.src[q]] = v;
            double dv[GRAD_DIRS];
            if (GRAD) {
                const double C = kind == NESOSIM_OBS_DEPTH ? __ldg(conc + (long long)a.obs_day[q] * a.plane + a.obs_cell[q]) : 1.0;
#pragma unroll
                for (int j = 0; j < GRAD_DIRS; ++j) {
                    const double2 t = g->tsamples[((long long)m * GRAD_DIRS + j) * a.stride + a.obs_slot[q]];
                    dv[j] = nesosim::finite(v) ? obs_tangent(kind, h, t, C, a.k) : nesosim::qnan();
                    if (g->jac) g->jac[((long long)m * GRAD_DIRS + j) * g->jac_stride + a.src[q]] = dv[j];
                }
            }
            const double r = div_ieee(sub(v, a.obs_val[q]), a.sigma[q]);   // sigma 1: exact, r = model - observed
            if (nesosim::finite(r)) {
                acc = add(acc, mul(r, r));
                ++cnt;
                if (GRAD) {
#pragma unroll
                    for (int j = 0; j < GRAD_DIRS; ++j) gacc[j] = add(gacc[j], mul(mul(2.0, r), div_ieee(dv[j], a.sigma[q])));
                }
            }
        }
        block_total(acc, cnt, red, redc, a.chi2 + (long long)m * a.n_kinds + kind,
                    a.count ? a.count + (long long)m * a.n_kinds + kind : nullptr);
        if (GRAD) {
#pragma unroll
            for (int j = 0; j < GRAD_DIRS; ++j)
                block_total(gacc[j], 0, red, redc, g->grad + ((long long)m * NESOSIM_OBS_KINDS + kind) * GRAD_DIRS + j, nullptr);
        }
    }
    if (!a.fp_chi2) return;
    // footprints: the same fixed order over each kind's range of the set's footprint table
    const int *fkb = a.fp_kind_begin + set * (NESOSIM_OBS_KINDS + 1);
    const double *mean = a.fp_mean + (long long)m * a.fp_stride - fkb[0];   // indexed by table position
    for (int kind = 0; kind < NESOSIM_OBS_KINDS; ++kind) {
        const long long i0 = fkb[kind], n_fp = (long long)fkb[kind + 1] - i0;
        double acc = 0.0, gacc[GRAD_DIRS] = {0.0, 0.0, 0.0};
        long long cnt = 0;
        for (long long i = threadIdx.x; i < n_fp; i += 256) {
            const long long q = i0 + i;
            const double r = div_ieee(sub(mean[q], a.fp_val[q]), a.fp_sigma[q]);
            if (nesosim::finite(r)) {
                acc = add(acc, mul(r, r));
                ++cnt;
                if (GRAD) {
#pragma unroll
                    for (int j = 0; j < GRAD_DIRS; ++j) {
                        const double dm = g->fp_dmean[((long long)m * GRAD_DIRS + j) * a.fp_stride - fkb[0] + q];
                        gacc[j] = add(gacc[j], mul(mul(2.0, r), div_ieee(dm, a.fp_sigma[q])));
                    }
                }
            }
        }
        block_total(acc, cnt, red, redc, a.fp_chi2 + (long long)m * NESOSIM_OBS_KINDS + kind,
                    a.fp_count ? a.fp_count + (long long)m * NESOSIM_OBS_KINDS + kind : nullptr);
        if (GRAD) {
#pragma unroll
            for (int j = 0; j < GRAD_DIRS; ++j)
                block_total(gacc[j], 0, red, redc, g->fp_grad + ((long long)m * NESOSIM_OBS_KINDS + kind) * GRAD_DIRS + j, nullptr);
        }
    }
}

template <bool SETS>
__global__ void __launch_bounds__(256) misfit_finish_kernel(const __grid_constant__ MisfitArgs a) {
    misfit_finish<SETS, false>(a, nullptr);
}
template <bool SETS>
__global__ void __launch_bounds__(256) misfit_finish_grad_kernel(const __grid_constant__ MisfitArgs a,
                                                                 const __grid_constant__ MisfitGrad g) {
    misfit_finish<SETS, true>(a, &g);
}

// Footprint means: one warp per (member, footprint).  The model value of every point is formed with exactly the
// operator of misfit_finish_kernel (depth (h0+h1)/iceConc, volume h0+h1, density densityCalc).  Point j of the
// footprint (in input order, land points dropped at registration) belongs to lane j % 32, which adds w*v to sw and w to
// s in order, skipping non-finite v; lane 0 collects both with the shuffle-down tree 16, 8, 4, 2, 1, and the mean is
// sw / s (NaN when no point was finite: 0/0).  Each lane keeps FP_UNROLL points' loads in flight: a monthly regional
// mean has tens of thousands of points.  A block is one warp: footprints differ in size by orders of magnitude, and a
// finished warp's slot is refilled at once instead of waiting for the longest warp of its block.  The point tables do
// not depend on the member, so the warps of every member on the same footprint (adjacent blocks: block = footprint *
// M + member) read them from L2.  Warps past the set's footprint count write the NaN padding of the caller's model row.
struct FootprintArgs {
    const double2 *samples;         // [M][stride]
    long long stride;
    const long long *begin;         // [n_fp+1]
    const int *kind, *src;
    const int *pt_slot, *pt_day, *pt_cell;
    const double *pt_w;
    const int *kind_begin;          // [sets][NESOSIM_OBS_KINDS+1]
    const double *conc;             // [T][plane] (SETS: [sets][T][plane])
    long long plane;
    ModelConsts k;
    int n_members;
    long long row_len;              // footprints per member row (the largest set's)
    double *mean;                   // [M][mean_stride] in table order within the set
    long long mean_stride;
    double *model;                  // [M][model_stride] at the input index within the set, or NULL
    long long model_stride;
    const int *member_set;          // SETS only
    long long conc_set_stride;      // SETS only
};
constexpr int FP_UNROLL = 8;
// GRAD (footprint_mean_grad_kernel): lane l also adds w*dv of the same points, in the same order, for every direction,
// and the same tree gives the derivative of the mean, sdw / s (NaN where the mean is not finite).
struct FootprintGrad {
    const double2 *tsamples;        // [M][GRAD_DIRS][stride]
    double *dmean;                  // [M][GRAD_DIRS][mean_stride] in table order within the set
    double *jac;                    // [M][GRAD_DIRS][jac_stride] at the input index within the set, or NULL
    long long jac_stride;
};
// ADJ (footprint_mean_adj_kernel, nesosim_run_season_score_adjoint): lane 0 also writes the footprint's seed
// coefficient b = (((2 r) fw[kind]) / sigma) / s, NaN where r is not finite (the footprint is not counted).
struct FootprintAdj {
    double *coef;                   // [M][mean_stride] in table order within the set
    const double *val, *sigma;      // the footprint table's values and errors
    double fw[NESOSIM_OBS_KINDS];
};
template <bool SETS, bool GRAD, bool ADJ = false>
__device__ __forceinline__ void footprint_mean(const FootprintArgs &a, const FootprintGrad *fg, const FootprintAdj *fa = nullptr) {
    const int m = (int)(blockIdx.x % (unsigned)a.n_members);
    const long long g = blockIdx.x / (unsigned)a.n_members;
    const int lane = threadIdx.x;
    if (g >= a.row_len) return;
    const int set = SETS ? a.member_set[m] : 0;
    const int *kb = a.kind_begin + set * (NESOSIM_OBS_KINDS + 1);
    double *model = a.model ? a.model + (long long)m * a.model_stride : nullptr;
    if (g >= (long long)kb[NESOSIM_OBS_KINDS] - kb[0]) {          // padding of a set with fewer footprints
        if (model && lane == 0) model[g] = nesosim::qnan();
        if (GRAD && fg->jac && lane == 0)
            for (int j = 0; j < GRAD_DIRS; ++j) fg->jac[((long long)m * GRAD_DIRS + j) * fg->jac_stride + g] = nesosim::qnan();
        return;
    }
    const long long q = kb[0] + g;
    const int kind = a.kind[q];
    const double2 *samp = a.samples + (long long)m * a.stride;
    const double *conc = SETS ? a.conc + (long long)set * a.conc_set_stride : a.conc;
    const long long p1 = a.begin[q + 1];
    double sw = 0.0, s = 0.0, sdw[GRAD_DIRS] = {0.0, 0.0, 0.0};
    for (long long p = a.begin[q] + lane; p < p1; p += 32 * FP_UNROLL) {
        double2 h[FP_UNROLL];
        double w[FP_UNROLL], c[FP_UNROLL];
#pragma unroll
        for (int u = 0; u < FP_UNROLL; ++u) {
            const long long pp = p + 32 * u;
            if (pp < p1) {
                h[u] = samp[__ldg(a.pt_slot + pp)];
                w[u] = __ldg(a.pt_w + pp);
                c[u] = kind == NESOSIM_OBS_DEPTH ? __ldg(conc + (long long)__ldg(a.pt_day + pp) * a.plane + __ldg(a.pt_cell + pp)) : 1.0;
            }
        }
#pragma unroll
        for (int u = 0; u < FP_UNROLL; ++u) {
            if (p + 32 * u < p1) {
                double v;
                if (kind == NESOSIM_OBS_DEPTH) v = div_ieee(add(h[u].x, h[u].y), c[u]);
                else if (kind == NESOSIM_OBS_VOLUME) v = add(h[u].x, h[u].y);
                else v = density_variable(h[u].x, h[u].y, false, a.k);
                if (nesosim::finite(v)) {
                    sw = add(sw, mul(w[u], v));
                    s = add(s, w[u]);
                    if (GRAD) {
                        const int slot = __ldg(a.pt_slot + p + 32 * u);
#pragma unroll
                        for (int j = 0; j < GRAD_DIRS; ++j) {
                            const double2 t = fg->tsamples[((long long)m * GRAD_DIRS + j) * a.stride + slot];
                            sdw[j] = add(sdw[j], mul(w[u], obs_tangent(kind, h[u], t, c[u], a.k)));
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        sw = add(sw, __shfl_down_sync(0xffffffffu, sw, off));
        s = add(s, __shfl_down_sync(0xffffffffu, s, off));
        if (GRAD) {
#pragma unroll
            for (int j = 0; j < GRAD_DIRS; ++j) sdw[j] = add(sdw[j], __shfl_down_sync(0xffffffffu, sdw[j], off));
        }
    }
    if (lane == 0) {
        const double v = div_ieee(sw, s);
        a.mean[(long long)m * a.mean_stride + g] = v;
        if (model) model[a.src[q]] = v;
        if (ADJ) {
            const double r = div_ieee(sub(v, fa->val[q]), fa->sigma[q]);
            fa->coef[(long long)m * a.mean_stride + g] =
                nesosim::finite(r) ? div_ieee(div_ieee(mul(mul(2.0, r), fa->fw[kind]), fa->sigma[q]), s) : nesosim::qnan();
        }
        if (GRAD) {
            for (int j = 0; j < GRAD_DIRS; ++j) {
                const double dm = nesosim::finite(v) ? div_ieee(sdw[j], s) : nesosim::qnan();
                fg->dmean[((long long)m * GRAD_DIRS + j) * a.mean_stride + g] = dm;
                if (fg->jac) fg->jac[((long long)m * GRAD_DIRS + j) * fg->jac_stride + a.src[q]] = dm;
            }
        }
    }
}
template <bool SETS>
__global__ void __launch_bounds__(32) footprint_mean_kernel(const __grid_constant__ FootprintArgs a) {
    footprint_mean<SETS, false>(a, nullptr);
}
template <bool SETS>
__global__ void __launch_bounds__(32) footprint_mean_grad_kernel(const __grid_constant__ FootprintArgs a,
                                                                 const __grid_constant__ FootprintGrad fg) {
    footprint_mean<SETS, true>(a, &fg);
}
template <bool SETS>
__global__ void __launch_bounds__(32) footprint_mean_adj_kernel(const __grid_constant__ FootprintArgs a,
                                                                const __grid_constant__ FootprintAdj fa) {
    footprint_mean<SETS, false, true>(a, nullptr, &fa);
}

// Seeds of the adjoint: one thread per (member, sample slot) sums dJ/d(h0, h1) from 0.0 over the slot's items in table
// order -- the point observations chi2 counts, in chi2's order, then the kept footprint points with finite v, in
// footprint input order -- each adding a * dv/d(h0, h1): a = ((2 r) w[kind]) / sigma for a point, b * w_p for a
// footprint point; depth (a/C, a/C), volume (a, a), density ((a (rhoF - q)) / den, (a (rhoO - q)) / den), 0 at a clamp.
struct SeedArgs {
    const double2 *samples;
    double2 *seeds;                 // [M][stride]
    long long stride;
    const int *begin;               // [sets][stride] + 1
    const int2 *item;
    const int *obs_day, *obs_cell;
    const double *obs_val, *sigma;
    const double *fp_coef;          // [M][fp_stride]
    long long fp_stride;
    const int *fp_kind, *fp_kind_begin, *pt_day, *pt_cell;
    const double *pt_w;
    const double *conc;             // [sets][T][plane]
    long long plane, conc_set_stride;
    const int *member_set;
    ModelConsts k;
    double w[NESOSIM_OBS_KINDS];
};
__device__ __forceinline__ void seed_partials(int kind, double2 h, double C, double a, const ModelConsts &k, double &g0,
                                              double &g1) {
    if (kind == NESOSIM_OBS_DEPTH) {
        g0 = g1 = div_ieee(a, C);
    } else if (kind == NESOSIM_OBS_VOLUME) {
        g0 = g1 = a;
    } else {
        const double den = add(h.x, h.y);
        const double q = div_ieee(add(mul(h.x, k.rhoFresh), mul(h.y, k.rhoOld)), den);
        if (q > k.rhoOld || q < k.rhoFresh) {
            g0 = g1 = 0.0;
        } else {
            g0 = div_ieee(mul(a, sub(k.rhoFresh, q)), den);
            g1 = div_ieee(mul(a, sub(k.rhoOld, q)), den);
        }
    }
}
// FORCING (adjoint_seed_forcing_kernel): also `cseed` [M][stride] = dJ/dC at the slot, summed from 0.0 in the same item
// order over the depth items alone: -((a v) / C) with v = (h0 + h1) / C (dv/dC = -v/C).
template <bool FORCING>
__device__ __forceinline__ void adjoint_seed(const SeedArgs &a, double *cseed) {
    const long long sl = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int m = blockIdx.y;
    if (sl >= a.stride) return;
    const int set = a.member_set ? a.member_set[m] : 0;
    const double *conc = a.conc + (long long)set * a.conc_set_stride;
    const double2 h = a.samples[(long long)m * a.stride + sl];
    const long long b = (long long)set * a.stride + sl;
    double s0 = 0.0, s1 = 0.0, cs = 0.0;
    for (int i = a.begin[b]; i < a.begin[b + 1]; ++i) {
        const int2 it = a.item[i];
        int kind;
        double av, v, C = 1.0;
        if (it.y < 0) {
            const int q = it.x;
            kind = -1 - it.y;
            if (kind == NESOSIM_OBS_DEPTH) {
                C = __ldg(conc + (long long)a.obs_day[q] * a.plane + a.obs_cell[q]);
                v = div_ieee(add(h.x, h.y), C);
            } else if (kind == NESOSIM_OBS_VOLUME) v = add(h.x, h.y);
            else v = density_variable(h.x, h.y, false, a.k);
            const double r = div_ieee(sub(v, a.obs_val[q]), a.sigma[q]);
            if (!nesosim::finite(r)) continue;
            av = div_ieee(mul(mul(2.0, r), a.w[kind]), a.sigma[q]);
        } else {
            const int q = it.x, p = it.y;
            kind = a.fp_kind[q];
            const double bc = a.fp_coef[(long long)m * a.fp_stride + q - a.fp_kind_begin[set * (NESOSIM_OBS_KINDS + 1)]];
            if (!nesosim::finite(bc)) continue;
            if (kind == NESOSIM_OBS_DEPTH) {
                C = __ldg(conc + (long long)a.pt_day[p] * a.plane + a.pt_cell[p]);
                v = div_ieee(add(h.x, h.y), C);
            } else if (kind == NESOSIM_OBS_VOLUME) v = add(h.x, h.y);
            else v = density_variable(h.x, h.y, false, a.k);
            if (!nesosim::finite(v)) continue;
            av = mul(bc, a.pt_w[p]);
        }
        double g0, g1;
        seed_partials(kind, h, C, av, a.k, g0, g1);
        s0 = add(s0, g0);
        s1 = add(s1, g1);
        if (FORCING && kind == NESOSIM_OBS_DEPTH) cs = add(cs, -div_ieee(mul(av, v), C));
    }
    a.seeds[(long long)m * a.stride + sl] = make_double2(s0, s1);
    if (FORCING) cseed[(long long)m * a.stride + sl] = cs;
}
__global__ void __launch_bounds__(256) adjoint_seed_kernel(const __grid_constant__ SeedArgs a) {
    adjoint_seed<false>(a, nullptr);
}
__global__ void __launch_bounds__(256) adjoint_seed_forcing_kernel(const __grid_constant__ SeedArgs a, double *cseed) {
    adjoint_seed<true>(a, cseed);
}

// lambda at each member's last slot L (set_steps, or T-1): 0, plus the seeds of day L at its sample slots.
struct AdjInitArgs {
    double *lam;                    // ring [parity][layer][M][plane]
    long long plane, layer_stride;
    const double2 *seeds;
    long long stride;
    const int *begin;
    const int2 *entry;
    int T, tiles;
    const int *member_set, *set_steps;
};
// FORCING (adjoint_init_forcing_kernel): also the per-day planes of days L..T-1 (0, and g_C(L) = 0 + cseed at day L's
// sample slots; no backward kernel writes these days) and the conc accumulator's first term, C(L) g_C(L).
struct ForcingInitArgs {
    const double *cseed;            // [M][stride]
    double *acc;                    // [M][FORCING_DIRS][plane], zeroed
    double *day[FORCING_DIRS];      // [M][T][plane] or NULL
    const double *conc;             // [sets][T][plane]
};
template <bool FORCING>
__device__ __forceinline__ void adjoint_init(const AdjInitArgs &a, const ForcingInitArgs *fi) {
    const int m = blockIdx.x;
    const int set = a.member_set ? a.member_set[m] : 0;
    const int L = a.set_steps ? a.set_steps[set] : a.T - 1;
    double *l0 = a.lam + (long long)(L & 1) * 2 * a.layer_stride + (long long)m * a.plane, *l1 = l0 + a.layer_stride;
    for (long long i = threadIdx.x; i < a.plane; i += blockDim.x) l0[i] = l1[i] = 0.0;
    if (FORCING) {
        for (int f = 0; f < FORCING_DIRS; ++f) {
            if (!fi->day[f]) continue;
            double *d = fi->day[f] + ((long long)m * a.T + L) * a.plane;
            for (long long i = threadIdx.x; i < (long long)(a.T - L) * a.plane; i += blockDim.x) d[i] = 0.0;
        }
    }
    __syncthreads();
    const long long b = ((long long)set * a.T + L) * a.tiles;
    const double2 *sd = a.seeds + (long long)m * a.stride;
    for (int i = a.begin[b] + threadIdx.x; i < a.begin[b + a.tiles]; i += blockDim.x) {
        const int2 e = a.entry[i];
        l0[e.x] = add(l0[e.x], sd[e.y].x);
        l1[e.x] = add(l1[e.x], sd[e.y].y);
        if (FORCING) {
            const double g = add(0.0, fi->cseed[(long long)m * a.stride + e.y]);
            const double C = __ldg(fi->conc + ((long long)set * a.T + L) * a.plane + e.x);
            if (fi->day[2]) fi->day[2][((long long)m * a.T + L) * a.plane + e.x] = g;
            double *t = fi->acc + ((long long)m * FORCING_DIRS + 2) * a.plane + e.x;
            *t = add(*t, nesosim::finite(C) ? mul(C, g) : 0.0);
        }
    }
}
__global__ void __launch_bounds__(256) adjoint_init_kernel(const __grid_constant__ AdjInitArgs a) {
    adjoint_init<false>(a, nullptr);
}
__global__ void __launch_bounds__(256) adjoint_init_forcing_kernel(const __grid_constant__ AdjInitArgs a,
                                                                   const __grid_constant__ ForcingInitArgs fi) {
    adjoint_init<true>(a, &fi);
}

// One CTA per member: theta_grad[m][j] = the fixed-order sum of the accumulators over the cells (cell i to thread
// i % 256, block_total), and ic_grad = (lambda0(0) + lambda1(0)) * 0.5, 0 where conc[0] < minConc.
struct AdjFinishArgs {
    const double *theta_acc;        // [M][GRAD_DIRS][plane]
    const double *lam0;             // ring slot 0, layer 0 (layer_stride further: layer 1)
    long long plane, layer_stride;
    const double *conc0;            // first day's concentration of set 0 (set_stride further: the next set)
    long long set_stride;
    const int *member_set;
    double minConc;
    double *theta_grad;             // [M][GRAD_DIRS]
    double *ic_grad;                // [M][plane]
};
// FORCING (adjoint_finish_forcing_kernel): also the scale fields (the accumulators) and their totals, each summed over
// the cells in the same fixed order as theta_grad.
struct ForcingFinishArgs {
    const double *acc;              // [M][FORCING_DIRS][plane]
    double *scale_grad;             // [M][FORCING_DIRS][plane]
    double *scale_total;            // [M][FORCING_DIRS]
};
// DRIFT (adjoint_finish_drift_kernel, adjoint_finish_forcing_drift_kernel): also the drift scale fields and totals in
// the same order, and 0 in the per-day drift planes of the member's days L..T-1 (no backward kernel writes those).
struct DriftFinishArgs {
    const double *acc;              // [M][DRIFT_DIRS][plane]
    double *scale_grad;             // [M][DRIFT_DIRS][plane]
    double *scale_total;            // [M][DRIFT_DIRS]
    double *day;                    // [M][T][DRIFT_DIRS][plane] or NULL
    const int *set_steps;           // NULL: one shared season of T days
    int T;
};
template <bool FORCING, bool DRIFT = false>
__device__ __forceinline__ void adjoint_finish(const AdjFinishArgs &a, const ForcingFinishArgs *ff,
                                               const DriftFinishArgs *df = nullptr) {
    const int m = blockIdx.x;
    __shared__ double red[8];
    __shared__ long long redc[8];
    for (int j = 0; j < GRAD_DIRS; ++j) {
        const double *t = a.theta_acc + ((long long)m * GRAD_DIRS + j) * a.plane;
        double acc = 0.0;
        for (long long i = threadIdx.x; i < a.plane; i += 256) acc = add(acc, t[i]);
        block_total(acc, 0, red, redc, a.theta_grad + (long long)m * GRAD_DIRS + j, nullptr);
    }
    if (FORCING) {
        for (int f = 0; f < FORCING_DIRS; ++f) {
            const long long o = ((long long)m * FORCING_DIRS + f) * a.plane;
            double acc = 0.0;
            for (long long i = threadIdx.x; i < a.plane; i += 256) {
                const double v = ff->acc[o + i];
                ff->scale_grad[o + i] = v;
                acc = add(acc, v);
            }
            block_total(acc, 0, red, redc, ff->scale_total + (long long)m * FORCING_DIRS + f, nullptr);
        }
    }
    if (DRIFT) {
        for (int k = 0; k < DRIFT_DIRS; ++k) {
            const long long o = ((long long)m * DRIFT_DIRS + k) * a.plane;
            double acc = 0.0;
            for (long long i = threadIdx.x; i < a.plane; i += 256) {
                const double v = df->acc[o + i];
                df->scale_grad[o + i] = v;
                acc = add(acc, v);
            }
            block_total(acc, 0, red, redc, df->scale_total + (long long)m * DRIFT_DIRS + k, nullptr);
        }
        if (df->day) {
            const int L = df->set_steps ? df->set_steps[a.member_set ? a.member_set[m] : 0] : df->T - 1;
            double *d = df->day + ((long long)m * df->T + L) * DRIFT_DIRS * a.plane;
            for (long long i = threadIdx.x; i < (long long)(df->T - L) * DRIFT_DIRS * a.plane; i += 256) d[i] = 0.0;
        }
    }
    const double *c0 = a.conc0 + (a.member_set ? a.member_set[m] * a.set_stride : 0);
    const double *l0 = a.lam0 + (long long)m * a.plane, *l1 = l0 + a.layer_stride;
    for (long long i = threadIdx.x; i < a.plane; i += 256)
        a.ic_grad[(long long)m * a.plane + i] = __ldg(c0 + i) < a.minConc ? 0.0 : mul(add(l0[i], l1[i]), 0.5);
}
__global__ void __launch_bounds__(256) adjoint_finish_kernel(const __grid_constant__ AdjFinishArgs a) {
    adjoint_finish<false>(a, nullptr);
}
__global__ void __launch_bounds__(256) adjoint_finish_forcing_kernel(const __grid_constant__ AdjFinishArgs a,
                                                                     const __grid_constant__ ForcingFinishArgs ff) {
    adjoint_finish<true>(a, &ff);
}
__global__ void __launch_bounds__(256) adjoint_finish_drift_kernel(const __grid_constant__ AdjFinishArgs a,
                                                                   const __grid_constant__ DriftFinishArgs df) {
    adjoint_finish<false, true>(a, nullptr, &df);
}
__global__ void __launch_bounds__(256) adjoint_finish_forcing_drift_kernel(const __grid_constant__ AdjFinishArgs a,
                                                                           const __grid_constant__ ForcingFinishArgs ff,
                                                                           const __grid_constant__ DriftFinishArgs df) {
    adjoint_finish<true, true>(a, &ff, &df);
}

// Observations compiled against the strip tables (host side).  One season's tables: every observation mapped to its
// owner (strip, index in the strip's ocean list), sorted by owner and day; `first` has list_end+1 entries, sample
// slots are the distinct (cell, day) pairs per owning cell in day order with one sentinel behind every cell's run --
// observations of different kinds at one cell and day share a slot.  The observations are then stable-partitioned by
// kind (kind_begin: NESOSIM_OBS_KINDS+1 entries per set), so each kind's sub-sequence is the one a registration of that
// kind alone gets.  Several seasons (forcing sets) are appended one after the other: a set's `first` entries and o_slot
// count from the set's first slot, so each set's tables are exactly those its season would get on its own (the caller
// moves `first` to absolute slots for the season kernel; o_slot stays the slot in the member's row of samples).
struct ObsPoint { int owner, day, cell, kind, src; double val, sigma; };
struct ObsTables {
    std::vector<int> first, slot_day, o_slot, o_day, o_cell, o_src, kind_begin;
    std::vector<double> o_val, o_sigma;
};

// position of every ocean cell in the concatenated code lists (ocean_off[k] + idx), -1 on land; list_end = the lists' end
std::vector<int> obs_owners(nesosim_ctx *ctx, int *list_end) {
    const StripTables &t = ctx->ens.tables;
    const int nx = ctx->cfg.nx;
    std::vector<int> owner((size_t)ctx->cfg.ny * nx, -1);
    *list_end = 0;
    for (int k = 0; k < t.cluster; ++k) {
        int idx = 0;
        for (int r = t.row0[k]; r < t.row0[k + 1]; ++r)
            for (int col = 0; col < nx; ++col) {
                const uint8_t m = ctx->mask_host[(size_t)r * nx + col];
                if (!(m > 10 || m < 1)) owner[(size_t)r * nx + col] = t.ocean_off[k] + idx++;
            }
        *list_end = std::max(*list_end, t.ocean_off[k] + idx);
    }
    return owner;
}

// General path: the owner of an ocean cell is its index among the ocean cells in row-major order -- monotone in
// row*nx + col as the strip owner is, so compile_obs_set orders the observations exactly as for the season kernel.
// cells[o] = the cell of owner o.
std::vector<int> ocean_owners(const nesosim_ctx *ctx, int *list_end, std::vector<int> &cells) {
    std::vector<int> owner(ctx->mask_host.size(), -1);
    cells.clear();
    for (size_t i = 0; i < owner.size(); ++i) {
        const uint8_t m = ctx->mask_host[i];
        if (!(m > 10 || m < 1)) {
            owner[i] = (int)cells.size();
            cells.push_back((int)i);
        }
    }
    *list_end = (int)cells.size();
    return owner;
}

// The sampling entries of the general path: every sample slot of every set (sentinels excluded) as (cell, slot relative
// to the set's row), grouped by (set, day, day-kernel tile); begin[(s*T + day)*tiles + tile] starts a group.
void sample_lists(const nesosim_ctx *ctx, const ObsTables &t, const std::vector<int> &slot_base, const std::vector<int> &cells,
                  std::vector<int> &begin, std::vector<int2> &entry) {
    const int T = ctx->cfg.num_days, nx = ctx->cfg.nx, tgx = (nx + TX - 1) / TX;
    const long long tiles = (long long)tgx * ((ctx->cfg.ny + TY - 1) / TY), L = (long long)cells.size();
    const size_t S = slot_base.size();
    std::vector<long long> key;
    std::vector<int2> ent;
    for (size_t s = 0; s < S; ++s)
        for (long long o = 0; o < L; ++o) {
            const int cell = cells[o];
            const long long tile = (long long)(cell / nx / TY) * tgx + (cell % nx) / TX;
            for (int j = t.first[s * (L + 1) + o]; t.slot_day[j] != 0x7fffffff; ++j) {
                key.push_back(((long long)s * T + t.slot_day[j]) * tiles + tile);
                ent.push_back(make_int2(cell, j - slot_base[s]));
            }
        }
    begin.assign((size_t)(S * T * tiles) + 1, 0);
    for (long long k : key) ++begin[k + 1];
    for (size_t i = 1; i < begin.size(); ++i) begin[i] += begin[i - 1];
    entry.resize(ent.size());
    std::vector<int> fill(begin.begin(), begin.end() - 1);
    for (size_t i = 0; i < ent.size(); ++i) entry[fill[key[i]]++] = ent[i];
}

// appends one season's observations to `t`; returns the number of sample slots it added (sentinels included).
// Footprint points (kind -1, src = their index in the set's point table) take part in the slot assignment only:
// pt_slot[src] receives their slot, and they never enter the observation tables.
size_t compile_obs_set(std::vector<ObsPoint> &obs, int list_end, ObsTables &t, std::vector<int> &pt_slot) {
    std::stable_sort(obs.begin(), obs.end(), [](const ObsPoint &x, const ObsPoint &y) { return x.owner != y.owner ? x.owner < y.owner : x.day < y.day; });
    const size_t f0 = t.first.size(), s0 = t.slot_day.size();
    t.first.resize(f0 + (size_t)list_end + 1, -1);
    t.slot_day.reserve(s0 + obs.size() + list_end + 1);
    std::vector<int> slot(obs.size());
    size_t p = 0;
    for (int o = 0; o < list_end; ++o) {
        t.first[f0 + o] = (int)(t.slot_day.size() - s0);
        while (p < obs.size() && obs[p].owner == o) {
            if (t.slot_day.size() - s0 == (size_t)t.first[f0 + o] || t.slot_day.back() != obs[p].day) t.slot_day.push_back(obs[p].day);
            slot[p] = (int)(t.slot_day.size() - s0) - 1;
            if (obs[p].kind < 0) pt_slot[obs[p].src] = slot[p];
            ++p;
        }
        t.slot_day.push_back(0x7fffffff);                // sentinel
    }
    for (int k = 0; k < NESOSIM_OBS_KINDS; ++k) {
        t.kind_begin.push_back((int)t.o_slot.size());
        for (size_t q = 0; q < obs.size(); ++q) {
            if (obs[q].kind != k) continue;
            t.o_slot.push_back(slot[q]);
            t.o_day.push_back(obs[q].day);
            t.o_cell.push_back(obs[q].cell);
            t.o_src.push_back(obs[q].src);
            t.o_val.push_back(obs[q].val);
            t.o_sigma.push_back(obs[q].sigma);
        }
    }
    t.kind_begin.push_back((int)t.o_slot.size());
    return t.slot_day.size() - s0;
}

// replaces the context's observations by `t` (samples: `stride` slots per member)
int upload_obs(nesosim_ctx *ctx, const ObsTables &t, long long stride) {
    CU(cudaDeviceSynchronize());                         // nothing in flight still reads the previous set
    obs_release(ctx);
    auto &ob = ctx->obs;
    const int M = ctx->cfg.n_members;
    const size_t n = t.o_slot.size(), nb = std::max<size_t>(1, n);
    ob.stride = stride;
    CU(cudaMalloc(&ob.first, t.first.size() * sizeof(int)));
    CU(cudaMalloc(&ob.day, t.slot_day.size() * sizeof(int)));
    CU(cudaMalloc(&ob.samples, (size_t)M * ob.stride * sizeof(double2)));
    CU(cudaMalloc(&ob.val, nb * sizeof(double)));
    CU(cudaMalloc(&ob.sigma, nb * sizeof(double)));
    CU(cudaMalloc(&ob.o_slot, nb * sizeof(int)));
    CU(cudaMalloc(&ob.o_day, nb * sizeof(int)));
    CU(cudaMalloc(&ob.o_cell, nb * sizeof(int)));
    CU(cudaMalloc(&ob.src, nb * sizeof(int)));
    CU(cudaMalloc(&ob.kind_begin, t.kind_begin.size() * sizeof(int)));
    CU(cudaMemcpy(ob.first, t.first.data(), t.first.size() * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ob.day, t.slot_day.data(), t.slot_day.size() * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMemset(ob.samples, 0, (size_t)M * ob.stride * sizeof(double2)));
    CU(cudaMemcpy(ob.kind_begin, t.kind_begin.data(), t.kind_begin.size() * sizeof(int), cudaMemcpyHostToDevice));
    if (n) {
        CU(cudaMemcpy(ob.val, t.o_val.data(), n * sizeof(double), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ob.sigma, t.o_sigma.data(), n * sizeof(double), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ob.o_slot, t.o_slot.data(), n * sizeof(int), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ob.o_day, t.o_day.data(), n * sizeof(int), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ob.o_cell, t.o_cell.data(), n * sizeof(int), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ob.src, t.o_src.data(), n * sizeof(int), cudaMemcpyHostToDevice));
    }
    return NESOSIM_OK;
}

// Footprints of one set as the registration collects them: per footprint (input order within the set) its kind,
// value, sigma and range of kept points in the set's point arrays.
struct FpSet {
    std::vector<int> kind;
    std::vector<double> val, sigma;
    std::vector<long long> begin{0};                     // [footprints+1] into the point arrays
    std::vector<int> pt_slot, pt_day, pt_cell;
    std::vector<double> pt_w;
};
struct FpTables {
    std::vector<long long> begin;
    std::vector<int> kind, src, kind_begin, pt_slot, pt_day, pt_cell;
    std::vector<double> val, sigma, pt_w;
};

// appends one set's footprints to `t`, stable-partitioned by kind (each kind's footprints in input order)
void append_fp_set(const FpSet &f, FpTables &t) {
    for (int k = 0; k < NESOSIM_OBS_KINDS; ++k) {
        t.kind_begin.push_back((int)t.kind.size());
        for (size_t g = 0; g < f.kind.size(); ++g) {
            if (f.kind[g] != k) continue;
            t.begin.push_back((long long)t.pt_slot.size());
            t.kind.push_back(k);
            t.src.push_back((int)g);
            t.val.push_back(f.val[g]);
            t.sigma.push_back(f.sigma[g]);
            const long long b = f.begin[g], e = f.begin[g + 1];
            t.pt_slot.insert(t.pt_slot.end(), f.pt_slot.begin() + b, f.pt_slot.begin() + e);
            t.pt_day.insert(t.pt_day.end(), f.pt_day.begin() + b, f.pt_day.begin() + e);
            t.pt_cell.insert(t.pt_cell.end(), f.pt_cell.begin() + b, f.pt_cell.begin() + e);
            t.pt_w.insert(t.pt_w.end(), f.pt_w.begin() + b, f.pt_w.begin() + e);
        }
    }
    t.kind_begin.push_back((int)t.kind.size());
}

template <typename T>
int upload_vec(T **dst, const std::vector<T> &v) {
    CU(cudaMalloc(dst, std::max<size_t>(1, v.size()) * sizeof(T)));
    if (!v.empty()) CU(cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return NESOSIM_OK;
}

// adds the footprint tables `t` to the context's freshly uploaded observations
int upload_fp(nesosim_ctx *ctx, FpTables &t, long long row_len) {
    auto &ob = ctx->obs;
    t.begin.push_back((long long)t.pt_slot.size());
    ob.n_fp = (long long)t.kind.size();
    ob.fp_row_len = row_len;
    int rc;
    if ((rc = upload_vec(&ob.fp_begin, t.begin)) || (rc = upload_vec(&ob.fp_kind, t.kind)) ||
        (rc = upload_vec(&ob.fp_src, t.src)) || (rc = upload_vec(&ob.fp_val, t.val)) ||
        (rc = upload_vec(&ob.fp_sigma, t.sigma)) || (rc = upload_vec(&ob.fp_kind_begin, t.kind_begin)) ||
        (rc = upload_vec(&ob.pt_slot, t.pt_slot)) || (rc = upload_vec(&ob.pt_day, t.pt_day)) ||
        (rc = upload_vec(&ob.pt_cell, t.pt_cell)) || (rc = upload_vec(&ob.pt_w, t.pt_w)))
        return rc;
    CU(cudaMalloc(&ob.fp_mean, (size_t)ctx->cfg.n_members * std::max(1LL, row_len) * sizeof(double)));
    return NESOSIM_OK;
}

// The seed items of every sample slot of the general path, slot-major ([sets][stride] + 1 run starts), each slot's items
// in the order adjoint_seed_kernel sums them: the set's point observations in chi2's order (kinds in turn, table order),
// then its footprints in input order with their points in order.  `ft.begin` has its closing entry (upload_fp).
void adjoint_items(const ObsTables &t, const FpTables &ft, int S, long long stride, std::vector<int> &begin,
                   std::vector<int2> &item) {
    std::vector<long long> key;
    std::vector<int2> it;
    for (int s = 0; s < S; ++s) {
        const int *kb = t.kind_begin.data() + (size_t)s * (NESOSIM_OBS_KINDS + 1);
        for (int k = 0; k < NESOSIM_OBS_KINDS; ++k)
            for (int q = kb[k]; q < kb[k + 1]; ++q) {
                key.push_back((long long)s * stride + t.o_slot[q]);
                it.push_back(make_int2(q, -1 - k));
            }
        const int *fb = ft.kind_begin.data() + (size_t)s * (NESOSIM_OBS_KINDS + 1);
        std::vector<int> fq;
        for (int q = fb[0]; q < fb[NESOSIM_OBS_KINDS]; ++q) fq.push_back(q);
        std::stable_sort(fq.begin(), fq.end(), [&](int x, int y) { return ft.src[x] < ft.src[y]; });
        for (int q : fq)
            for (long long p = ft.begin[q]; p < ft.begin[q + 1]; ++p) {
                key.push_back((long long)s * stride + ft.pt_slot[p]);
                it.push_back(make_int2(q, (int)p));
            }
    }
    begin.assign((size_t)S * stride + 1, 0);
    for (long long k : key) ++begin[k + 1];
    for (size_t i = 1; i < begin.size(); ++i) begin[i] += begin[i - 1];
    item.resize(it.size());
    std::vector<int> fill(begin.begin(), begin.end() - 1);
    for (size_t i = 0; i < it.size(); ++i) item[fill[key[i]]++] = it[i];
}

// Validates every observation and footprint, then compiles them against the strip tables and replaces the context's
// observations.  sets: tagged with their forcing set (obs_set_host / fp_set_host); else one shared forcing.  Footprint
// points get sample slots with the point observations (one slot per distinct (cell, day)) but never enter the point
// tables, so the point results do not depend on the footprints.  Nothing is freed before the last check.
int register_observations(nesosim_ctx *ctx, bool sets, int64_t n_obs, const int32_t *obs_set_host, const int32_t *obs_day_host,
                          const int32_t *obs_row_host, const int32_t *obs_col_host, const int32_t *obs_kind_host,
                          const double *obs_value_host, const double *obs_sigma_host,
                          int64_t n_fp = 0, const int32_t *fp_set_host = nullptr, const int32_t *fp_kind_host = nullptr,
                          const double *fp_value_host = nullptr, const double *fp_sigma_host = nullptr,
                          const int64_t *fp_begin_host = nullptr, const int32_t *pt_day_host = nullptr,
                          const int32_t *pt_row_host = nullptr, const int32_t *pt_col_host = nullptr,
                          const double *pt_weight_host = nullptr) {
    if (!ctx || n_obs < 0 || n_fp < 0) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (n_obs > 0 && ((sets && !obs_set_host) || !obs_day_host || !obs_row_host || !obs_col_host || !obs_value_host))
        return fail(NESOSIM_ERR_ARG, "NULL observation array");
    if (n_fp > 0 && ((sets && !fp_set_host) || !fp_value_host || !fp_begin_host || !pt_day_host || !pt_row_host || !pt_col_host))
        return fail(NESOSIM_ERR_ARG, "NULL footprint array");
    if (sets && !ctx->member_set_dev) return fail(NESOSIM_ERR_STATE, "set observations need nesosim_set_forcing_sets first");
    CU(cudaSetDevice(ctx->cfg.device));
    const nesosim_config &c = ctx->cfg;
    const int T = c.num_days, ny = c.ny, nx = c.nx, S = sets ? ctx->n_sets : 1;
    nesosim_outputs none{};
    none.depth_member_stride = (int64_t)T * 2 * ctx->plane;
    none.plane_member_stride = (int64_t)T * ctx->plane;
    const char *why = "";
    const bool general = ctx->path == 1;
    if (general) {
        if (ctx->strip.on) return fail(NESOSIM_ERR_ARG, "the general scoring path does not take a strip of a decomposed grid");
        if (c.density_clim)
            return fail(NESOSIM_ERR_ARG, "the general scoring path does not take densityType='clim' (its density operator is densityCalc)");
    } else if (!ensemble_eligible(ctx, 0, T - 1, &none, &why)) {
        return fail(NESOSIM_ERR_ARG, std::string("misfit mode needs the season-resident kernel: ") + why);
    }
    int list_end = 0;
    std::vector<int> cells;
    const std::vector<int> owner = general ? ocean_owners(ctx, &list_end, cells) : obs_owners(ctx, &list_end);
    std::vector<std::vector<ObsPoint>> per_set((size_t)S);
    std::vector<int> n_in((size_t)S, 0);                 // input observations of every set so far (-> src)
    bool depth_only = true;
    for (int64_t i = 0; i < n_obs; ++i) {
        const int s = sets ? obs_set_host[i] : 0, d = obs_day_host[i], r = obs_row_host[i], col = obs_col_host[i];
        const int kind = obs_kind_host ? obs_kind_host[i] : NESOSIM_OBS_DEPTH;
        const double sigma = obs_sigma_host ? obs_sigma_host[i] : 1.0;
        if (s < 0 || s >= S) return fail(NESOSIM_ERR_ARG, "observation set index outside [0, n_sets)");
        if (d < 0 || d >= (sets ? ctx->set_days[s] : T)) return fail(NESOSIM_ERR_ARG, "observation day outside its season");
        if (r < 0 || r >= ny || col < 0 || col >= nx) return fail(NESOSIM_ERR_ARG, "observation outside the grid");
        if (kind < 0 || kind >= NESOSIM_OBS_KINDS) return fail(NESOSIM_ERR_ARG, "observation kind outside [0, NESOSIM_OBS_KINDS)");
        if (kind == NESOSIM_OBS_DENSITY && d == 0)
            return fail(NESOSIM_ERR_ARG, "density observation on day 0: the model has no density there (NESOSIM.py:350-376)");
        if (!(std::isfinite(sigma) && sigma > 0.0)) return fail(NESOSIM_ERR_ARG, "observation error sigma must be finite and > 0");
        depth_only = depth_only && kind == NESOSIM_OBS_DEPTH && sigma == 1.0;
        if (n_in[s] == INT_MAX) return fail(NESOSIM_ERR_ARG, "a set's observations do not fit the tables' int indices");
        const int src = n_in[s]++;
        const int o = owner[(size_t)r * nx + col];
        if (o < 0) continue;                             // land / lake: the model value is NaN, the observation is skipped
        per_set[s].push_back(ObsPoint{o, d, r * nx + col, kind, src, obs_value_host[i], sigma});
    }
    std::vector<FpSet> fps((size_t)S);
    if (n_fp > 0 && fp_begin_host[0] != 0) return fail(NESOSIM_ERR_ARG, "fp_begin[0] must be 0");
    for (int64_t g = 0; g < n_fp; ++g) {
        const int s = sets ? fp_set_host[g] : 0;
        const int kind = fp_kind_host ? fp_kind_host[g] : NESOSIM_OBS_DEPTH;
        const double sigma = fp_sigma_host ? fp_sigma_host[g] : 1.0;
        if (s < 0 || s >= S) return fail(NESOSIM_ERR_ARG, "footprint set index outside [0, n_sets)");
        if (kind < 0 || kind >= NESOSIM_OBS_KINDS) return fail(NESOSIM_ERR_ARG, "footprint kind outside [0, NESOSIM_OBS_KINDS)");
        if (!(std::isfinite(sigma) && sigma > 0.0)) return fail(NESOSIM_ERR_ARG, "footprint error sigma must be finite and > 0");
        if (fp_begin_host[g + 1] <= fp_begin_host[g]) return fail(NESOSIM_ERR_ARG, "fp_begin must increase: a footprint needs a point");
        FpSet &f = fps[s];
        if (f.kind.size() == (size_t)INT_MAX) return fail(NESOSIM_ERR_ARG, "a set's footprints do not fit the tables' int indices");
        const int days = sets ? ctx->set_days[s] : T;
        for (int64_t j = fp_begin_host[g]; j < fp_begin_host[g + 1]; ++j) {
            const int d = pt_day_host[j], r = pt_row_host[j], col = pt_col_host[j];
            const double w = pt_weight_host ? pt_weight_host[j] : 1.0;
            if (d < 0 || d >= days) return fail(NESOSIM_ERR_ARG, "footprint point day outside its season");
            if (r < 0 || r >= ny || col < 0 || col >= nx) return fail(NESOSIM_ERR_ARG, "footprint point outside the grid");
            if (kind == NESOSIM_OBS_DENSITY && d == 0)
                return fail(NESOSIM_ERR_ARG, "density footprint point on day 0: the model has no density there (NESOSIM.py:350-376)");
            if (!(std::isfinite(w) && w > 0.0)) return fail(NESOSIM_ERR_ARG, "footprint point weight must be finite and > 0");
            const int o = owner[(size_t)r * nx + col];
            if (o < 0) continue;                         // land / lake: dropped, as point observations are
            if (f.pt_day.size() + per_set[s].size() >= (size_t)INT_MAX)
                return fail(NESOSIM_ERR_ARG, "a set's points do not fit the tables' int indices");
            per_set[s].push_back(ObsPoint{o, d, r * nx + col, -1, (int)f.pt_day.size(), 0.0, 0.0});
            f.pt_day.push_back(d);
            f.pt_cell.push_back(r * nx + col);
            f.pt_w.push_back(w);
        }
        f.kind.push_back(kind);
        f.val.push_back(fp_value_host[g]);
        f.sigma.push_back(sigma);
        f.begin.push_back((long long)f.pt_day.size());
    }
    ObsTables t;
    FpTables ft;
    std::vector<int> slot_base(S);
    size_t stride = 0;                                   // a member samples one set only: the largest set, not the sum
    size_t fp_row_len = 0;
    for (int s = 0; s < S; ++s) {
        if (t.slot_day.size() + per_set[s].size() + list_end + 1 > (size_t)INT_MAX)
            return fail(NESOSIM_ERR_ARG, "the sample slots do not fit the tables' int indices");
        slot_base[s] = (int)t.slot_day.size();
        fps[s].pt_slot.assign(fps[s].pt_day.size(), 0);
        stride = std::max(stride, compile_obs_set(per_set[s], list_end, t, fps[s].pt_slot));
        for (int o = 0; o < list_end; ++o) t.first[(size_t)s * (list_end + 1) + o] += slot_base[s];   // -> index in `day`
        fp_row_len = std::max(fp_row_len, fps[s].kind.size());
    }
    if (t.o_slot.size() > (size_t)INT_MAX || (size_t)n_fp > (size_t)INT_MAX)
        return fail(NESOSIM_ERR_ARG, "the observations do not fit the tables' int indices");
    for (int s = 0; s < S; ++s) append_fp_set(fps[s], ft);
    std::vector<int> smp_begin;
    std::vector<int2> smp_entry;
    if (general) sample_lists(ctx, t, slot_base, cells, smp_begin, smp_entry);
    int rc = upload_obs(ctx, t, (long long)stride);
    if (rc) return rc;
    if ((rc = upload_fp(ctx, ft, (long long)fp_row_len))) return rc;
    auto &ob = ctx->obs;
    if (general) adjoint_items(t, ft, S, (long long)stride, ob.adj_begin_h, ob.adj_item_h);
    if (general) {
        if ((rc = upload_vec(&ob.smp_begin, smp_begin)) || (rc = upload_vec(&ob.smp_entry, smp_entry))) return rc;
        ob.smp_tiles = (int)(((nx + TX - 1) / TX) * ((ny + TY - 1) / TY));
        CU(cudaMalloc(&ob.ring, (size_t)4 * c.n_members * ctx->plane * sizeof(double)));
        ob.general = true;
    }
    ob.row_len = *std::max_element(n_in.begin(), n_in.end());
    ob.depth_only = depth_only;
    if (sets) {
        ob.first_stride = (long long)list_end + 1;
        CU(cudaMalloc(&ob.slot_base, S * sizeof(int)));
        CU(cudaMemcpy(ob.slot_base, slot_base.data(), S * sizeof(int), cudaMemcpyHostToDevice));
        ob.set_days = ctx->set_days;
    }
    ob.ready = true;
    return NESOSIM_OK;
}

// The sample producer of the general path: slot 0 of the depth ring (init_slot0_kernel), the T-1 scoring day kernels
// (day x samples day x, then advances the depths to slot x+1) and sample_last_day_kernel: T+1 launches, no pre-pass,
// nothing written outside the context, no synchronisation.
// grad: the gradient builds (day_step_grad_kernel, sample_last_day_grad_kernel), which also advance and sample the
// tangents; still T+1 launches.
// rec: the record builds (day_step_record_kernel, sample_last_day_traj_kernel) into the adjoint's trajectory; T+1 launches.
int run_score_days(nesosim_ctx *ctx, const double *ic_dev, int ic_per_member, cudaStream_t st, bool grad = false,
                   bool rec = false) {
    const auto &ob = ctx->obs;
    const nesosim_config &c = ctx->cfg;
    const int T = c.num_days, M = c.n_members;
    const long long plane = ctx->plane, layer = (long long)M * plane;
    auto ring = [&](int t, int l) {
        return rec ? ob.traj + ((long long)t * 2 + l) * layer : ob.ring + ((long long)(t & 1) * 2 + l) * layer;
    };
    InitArgs ia{};
    ia.plane = plane;
    ia.ic = ic_dev;
    ia.ic_stride = ic_per_member ? plane : 0;
    ia.conc0 = ctx->C;
    ia.member_set = ctx->member_set_dev;
    ia.set_stride = (long long)T * plane;
    ia.minConc = c.minConc;
    ia.slot0[V_H0] = ring(0, 0);
    ia.slot0[V_H1] = ring(0, 1);
    ia.stride[V_H0] = ia.stride[V_H1] = plane;
    init_slot0_kernel<<<dim3((unsigned)((plane + 255) / 256), M), 256, 0, st>>>(ia);
    ctx->launches++;
    CU(cudaGetLastError());
    SampleArgs sa;
    sa.begin = ob.smp_begin; sa.entry = ob.smp_entry; sa.samples = ob.samples; sa.stride = ob.stride;
    sa.T = T; sa.tiles = ob.smp_tiles;
    sa.ring = rec ? ob.traj : ob.ring; sa.plane = plane; sa.layer_stride = layer;
    sa.member_set = ctx->member_set_dev; sa.set_steps = ctx->set_steps_dev;
    const dim3 grid((c.nx + TX - 1) / TX, (c.ny + TY - 1) / TY, M);
    TangentArgs ta{};
    ta.layer_stride = layer;
    ta.dir_stride = 2 * layer;
    ta.samples = ob.tsamples;
    ta.ring = ob.tring;
    auto tring = [&](int t) { return ob.tring + (long long)(t & 1) * GRAD_DIRS * 2 * layer; };
    nesosim_outputs none{};
    for (int x = 0; x < T - 1; ++x) {
        DayArgs a;
        fill_day_args(ctx, x, ctx->P + x * plane, ctx->C + x * plane, ctx->W + x * plane, ctx->UV + (long long)x * 2 * plane,
                      ctx->UV + ((long long)x * 2 + 1) * plane, c.snowDensityFresh, &none, 0, x > 0, a);
        for (int v = 0; v < NVAR; ++v) a.prev[v] = a.next[v] = nullptr;
        for (int l = 0; l < 2; ++l) {
            a.prev[V_H0 + l] = ring(x, l);
            a.next[V_H0 + l] = ring(x + 1, l);
        }
        a.depth_mstride = a.plane_mstride = plane;
        const bool pdl = ctx->pdl && x > 0;       // behind this call's own previous day kernel only (see launch_day)
        if (rec) {
            const RecArgs ra{ob.rec_flags + (long long)x * layer};
            if (ctx->day_variant == 512) CU(launch_day_kernel(day_step_record_kernel_512, grid, 512, st, pdl, a, sa, ra));
            else CU(launch_day_kernel(day_step_record_kernel, grid, 256, st, pdl, a, sa, ra));
        } else if (grad) {
            ta.prev = tring(x);
            ta.next = tring(x + 1);
            if (ctx->day_variant == 512) CU(launch_day_kernel(day_step_grad_kernel_512, grid, 512, st, pdl, a, sa, ta));
            else CU(launch_day_kernel(day_step_grad_kernel, grid, 256, st, pdl, a, sa, ta));
        } else if (ctx->day_variant == 512) {
            CU(launch_day_kernel(day_step_score_kernel_512, grid, 512, st, pdl, a, sa));
        } else {
            CU(launch_day_kernel(day_step_score_kernel, grid, 256, st, pdl, a, sa));
        }
        ctx->launches++;
    }
    if (rec) sample_last_day_traj_kernel<<<M, 256, 0, st>>>(sa);
    else if (grad) sample_last_day_grad_kernel<<<M, 256, 0, st>>>(sa, ta);
    else sample_last_day_kernel<<<M, 256, 0, st>>>(sa);
    ctx->launches++;
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

// The season with fused sampling, then the scores epilogue: n_kinds = NESOSIM_OBS_KINDS (nesosim_run_season_scores) or
// 1 (nesosim_run_season_misfit: the depth sum only, which needs observations that are all depth with sigma 1).
// fp: nesosim_run_season_scores_fp -- the footprint means (footprint_mean_kernel) between the season and the epilogue,
// which then also scores them; without it, registered footprints are NESOSIM_ERR_STATE (their data would be dropped).
// g: nesosim_run_season_score_grads -- the gradient builds of the day kernel and of both epilogues (general path only).
struct GradOutputs {
    double *grad, *jac;
    int64_t jac_stride;
    double *fp_grad, *fp_jac;
    int64_t fp_jac_stride;
};
int run_season_scores(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev, int ic_per_member,
                      double *chi2_dev, int64_t *count_dev, int n_kinds, double *model_dev, int64_t model_stride,
                      void *stream, bool fp = false, double *fp_chi2_dev = nullptr, int64_t *fp_count_dev = nullptr,
                      double *fp_model_dev = nullptr, int64_t fp_model_stride = 0, const GradOutputs *g = nullptr) {
    if (g) {
        if (!ctx || !params_host || !chi2_dev || !g->grad) return fail(NESOSIM_ERR_ARG, "bad argument");
        if (!ctx->obs.ready || !ctx->obs.general)
            return fail(NESOSIM_ERR_STATE, "gradients need observations registered on the general path (nesosim_set_path(ctx, 1) first)");
        if (ctx->obs.n_fp && (!fp_chi2_dev || !g->fp_grad))
            return fail(NESOSIM_ERR_STATE, "footprints are registered: fp_chi2_dev and fp_grad_dev are required");
        if (g->jac && g->jac_stride < ctx->obs.row_len) return fail(NESOSIM_ERR_ARG, "jac_stride is shorter than the observation row");
        if (ctx->obs.n_fp && g->fp_jac && g->fp_jac_stride < ctx->obs.fp_row_len)
            return fail(NESOSIM_ERR_ARG, "fp_jac_stride is shorter than the footprint row");
        if (ctx->cfg.n_members > 65535 || (ctx->cfg.ny + TY - 1) / TY > 65535)
            return fail(NESOSIM_ERR_ARG, "members or tile rows exceed the day kernel's grid dimensions");
        fp = ctx->obs.n_fp > 0;
    }
    if (!ctx || !params_host || !chi2_dev || (fp && !fp_chi2_dev)) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (!ctx->P) return fail(NESOSIM_ERR_STATE, "nesosim_set_forcing has not been called");
    if (!ctx->obs.ready) return fail(NESOSIM_ERR_STATE, "nesosim_set_observations has not been called");
    if (!fp && ctx->obs.n_fp)
        return fail(NESOSIM_ERR_STATE, "footprints are registered; use nesosim_run_season_scores_fp");
    if (n_kinds == 1 && !ctx->obs.depth_only)
        return fail(NESOSIM_ERR_STATE, "the registered observations are not all depth with sigma 1; use nesosim_run_season_scores");
    if (model_dev && model_stride < ctx->obs.row_len) return fail(NESOSIM_ERR_ARG, "model_stride is shorter than the observation row");
    if (fp_model_dev && fp_model_stride < ctx->obs.fp_row_len)
        return fail(NESOSIM_ERR_ARG, "fp_model_stride is shorter than the footprint row");
    const bool sets = !ctx->obs.set_days.empty();
    if (!sets && ctx->member_set_dev) return fail(NESOSIM_ERR_ARG, "misfit mode runs on one shared forcing");
    if (sets && ctx->obs.set_days != ctx->set_days)
        return fail(NESOSIM_ERR_STATE, "the forcing sets changed since nesosim_set_observations_sets; register the observations again");
    const bool general = ctx->obs.general;
    if (general != (ctx->path == 1))
        return fail(NESOSIM_ERR_STATE, "the kernel path changed since the observations were registered; register them again");
    CU(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const nesosim_config &c = ctx->cfg;
    const int T = c.num_days, M = c.n_members;
    int rc;
    auto &ob = ctx->obs;
    if (g) {
        const size_t tr = (size_t)2 * GRAD_DIRS * 2 * M * ctx->plane, ts = (size_t)M * GRAD_DIRS * ob.stride;
        if (!ob.tring) CU(cudaMalloc(&ob.tring, tr * sizeof(double)));
        if (!ob.tsamples) {
            CU(cudaMalloc(&ob.tsamples, ts * sizeof(double2)));
            CU(cudaMemset(ob.tsamples, 0, ts * sizeof(double2)));
        }
        if (!ob.fp_dmean) CU(cudaMalloc(&ob.fp_dmean, (size_t)M * GRAD_DIRS * std::max(1LL, ob.fp_row_len) * sizeof(double)));
    }
    if (general) {
        if ((rc = upload_coef(ctx, params_host, st))) return rc;
        ctx->last_path = 1;
        if ((rc = run_score_days(ctx, ic_dev, ic_per_member, st, g != nullptr))) return rc;
    } else {
        nesosim_outputs none{};
        none.depth_member_stride = (int64_t)T * 2 * ctx->plane;
        none.plane_member_stride = (int64_t)T * ctx->plane;
        const char *why = "";
        if (!ensemble_eligible(ctx, 0, T - 1, &none, &why))
            return fail(NESOSIM_ERR_ARG, std::string("misfit mode needs the season-resident kernel: ") + why);
        if ((rc = upload_coef(ctx, params_host, st))) return rc;
        ObsDevice od;
        od.first = ctx->obs.first; od.day = ctx->obs.day; od.sample_hh = ctx->obs.samples; od.sample_stride = ctx->obs.stride;
        od.first_stride = ctx->obs.first_stride; od.slot_base = ctx->obs.slot_base;
        ctx->last_path = 2;
        rc = run_ensemble(ctx, ic_dev, ic_per_member, &none, 0, M, st, &od);     // synchronises the stream (operand-range flag)
        if (rc) return rc;
    }
    // observations dropped at registration (land, lake) have no model value: their entries stay NaN (all bits set)
    if (model_dev && ctx->obs.row_len)
        CU(cudaMemset2DAsync(model_dev, (size_t)model_stride * sizeof(double), 0xff, (size_t)ctx->obs.row_len * sizeof(double), M, st));
    if (g && g->jac && ob.row_len)
        CU(cudaMemset2DAsync(g->jac, (size_t)g->jac_stride * sizeof(double), 0xff, (size_t)ob.row_len * sizeof(double),
                             (size_t)M * GRAD_DIRS, st));
    MisfitGrad mg{};
    if (g) {
        mg.tsamples = ob.tsamples; mg.grad = g->grad; mg.jac = g->jac; mg.jac_stride = g->jac_stride;
        mg.fp_dmean = ob.fp_dmean; mg.fp_grad = g->fp_grad;
    }
    MisfitArgs ma;
    ma.samples = ctx->obs.samples; ma.stride = ctx->obs.stride;
    ma.obs_slot = ctx->obs.o_slot; ma.obs_day = ctx->obs.o_day; ma.obs_cell = ctx->obs.o_cell; ma.src = ctx->obs.src;
    ma.obs_val = ctx->obs.val; ma.sigma = ctx->obs.sigma; ma.kind_begin = ctx->obs.kind_begin;
    ma.conc = ctx->C; ma.plane = ctx->plane; ma.k = ctx->k;
    ma.chi2 = chi2_dev; ma.count = (long long *)count_dev; ma.n_kinds = n_kinds;
    ma.model = model_dev; ma.model_stride = model_stride;
    ma.member_set = ctx->member_set_dev; ma.conc_set_stride = (long long)T * ctx->plane;
    ma.fp_chi2 = nullptr; ma.fp_count = nullptr;
    if (fp) {
        if (ob.fp_row_len) {
            FootprintArgs fa;
            fa.samples = ob.samples; fa.stride = ob.stride;
            fa.begin = ob.fp_begin; fa.kind = ob.fp_kind; fa.src = ob.fp_src;
            fa.pt_slot = ob.pt_slot; fa.pt_day = ob.pt_day; fa.pt_cell = ob.pt_cell; fa.pt_w = ob.pt_w;
            fa.kind_begin = ob.fp_kind_begin; fa.conc = ctx->C; fa.plane = ctx->plane; fa.k = ctx->k;
            fa.n_members = M; fa.row_len = ob.fp_row_len; fa.mean = ob.fp_mean; fa.mean_stride = ob.fp_row_len;
            fa.model = fp_model_dev; fa.model_stride = fp_model_stride;
            fa.member_set = ctx->member_set_dev; fa.conc_set_stride = (long long)T * ctx->plane;
            const long long blocks = ob.fp_row_len * M;
            if (blocks > INT_MAX) return fail(NESOSIM_ERR_ARG, "too many footprints x members for one launch");
            FootprintGrad fg{ob.tsamples, ob.fp_dmean, g ? g->fp_jac : nullptr, g ? g->fp_jac_stride : 0};
            if (g && sets) footprint_mean_grad_kernel<true><<<(unsigned)blocks, 32, 0, st>>>(fa, fg);
            else if (g) footprint_mean_grad_kernel<false><<<(unsigned)blocks, 32, 0, st>>>(fa, fg);
            else if (sets) footprint_mean_kernel<true><<<(unsigned)blocks, 32, 0, st>>>(fa);
            else footprint_mean_kernel<false><<<(unsigned)blocks, 32, 0, st>>>(fa);
            ctx->launches++;
            CU(cudaGetLastError());
        }
        ma.fp_mean = ob.fp_mean; ma.fp_stride = std::max(1LL, ob.fp_row_len);
        ma.fp_val = ob.fp_val; ma.fp_sigma = ob.fp_sigma; ma.fp_kind_begin = ob.fp_kind_begin;
        ma.fp_chi2 = fp_chi2_dev; ma.fp_count = (long long *)fp_count_dev;
    }
    if (g && sets) misfit_finish_grad_kernel<true><<<M, 256, 0, st>>>(ma, mg);
    else if (g) misfit_finish_grad_kernel<false><<<M, 256, 0, st>>>(ma, mg);
    else if (sets) misfit_finish_kernel<true><<<M, 256, 0, st>>>(ma);
    else misfit_finish_kernel<false><<<M, 256, 0, st>>>(ma);
    ctx->launches++;
    CU(cudaGetLastError());
    if (!general && ctx->ens_status) return fail(NESOSIM_ERR_ARG, "an operand left the range of the season-resident kernel's fast divisions; misfit mode has no general-path fallback");
    return NESOSIM_OK;
}

// nesosim_run_season_score_adjoint: the record build of the season (T+1 launches), the footprint means with their seed
// coefficients (one launch, with footprints), the scores epilogue (one), the seeds (one), lambda at the last slots (one),
// the T-1 backward day kernels and the finish (one): 2T+4 launches, 2T+5 with footprints (the seeds are skipped on a
// grid without ocean), and one memset (two with model rows).  With `forcing` (nesosim_run_season_score_adjoint_forcing)
// the seed, init, backward and finish kernels are their forcing builds, and one more memset clears the accumulators.
// With `drift` (nesosim_run_season_score_adjoint_drift) the backward and finish kernels are their drift builds (with the
// forcing terms too when `forcing` is also given), and one more memset clears the drift accumulators.
struct AdjOutputs {
    const double *w, *fw;           // host [NESOSIM_OBS_KINDS]
    double *theta_grad, *ic_grad;
};
static_assert(FORCING_DIRS == NESOSIM_FORCING_DIRS, "forcing directions");
struct ForcingOutputs {
    double *scale_grad, *scale_total;   // [M][FORCING_DIRS][plane], [M][FORCING_DIRS]
    double *day[FORCING_DIRS];          // [M][T][plane] or NULL
};
static_assert(DRIFT_DIRS == NESOSIM_DRIFT_DIRS, "drift directions");
struct DriftOutputs {
    double *scale_grad, *scale_total;   // [M][DRIFT_DIRS][plane], [M][DRIFT_DIRS]
    double *day;                        // [M][T][DRIFT_DIRS][plane] or NULL
};
// the drift builds of the backward day kernel take their shared memory dynamically (AdjDriftSmem in day_kernels.cuh)
template <typename... KArgs>
cudaError_t allow_drift_smem(void (*kern)(KArgs...), size_t bytes) {
    return cudaFuncSetAttribute((const void *)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}
// frees the per-call adjoint state (the seed item tables stay: they belong to the registration)
template <typename Obs>
void adj_release(Obs &ob) {
    cudaFree(ob.traj); cudaFree(ob.rec_flags); cudaFree(ob.lam); cudaFree(ob.theta_acc); cudaFree(ob.seeds);
    cudaFree(ob.fp_coef); cudaFree(ob.cseed); cudaFree(ob.forcing_acc); cudaFree(ob.drift_acc);
    ob.traj = ob.lam = ob.theta_acc = ob.fp_coef = ob.cseed = ob.forcing_acc = ob.drift_acc = nullptr;
    ob.rec_flags = nullptr;
    ob.seeds = nullptr;
}
template <typename T>
int adj_alloc(T **p, size_t n) {
    if (*p) return NESOSIM_OK;
    if (cudaMalloc(p, std::max<size_t>(1, n) * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();
        *p = nullptr;
        return fail(NESOSIM_ERR_NOMEM, "the adjoint state does not fit the device");
    }
    return NESOSIM_OK;
}
int run_season_score_adjoint(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                             int ic_per_member, double *chi2_dev, int64_t *count_dev, double *model_dev,
                             int64_t model_stride, double *fp_chi2_dev, int64_t *fp_count_dev, double *fp_model_dev,
                             int64_t fp_model_stride, const AdjOutputs &ad, void *stream,
                             const ForcingOutputs *fo = nullptr, const DriftOutputs *dro = nullptr) {
    if (!ctx || !params_host || !chi2_dev || !ad.theta_grad || !ad.ic_grad || !ad.w || !ad.fw)
        return fail(NESOSIM_ERR_ARG, "bad argument");
    if (fo && (!fo->scale_grad || !fo->scale_total)) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (dro && (!dro->scale_grad || !dro->scale_total)) return fail(NESOSIM_ERR_ARG, "bad argument");
    for (int k = 0; k < NESOSIM_OBS_KINDS; ++k)
        if (!(std::isfinite(ad.w[k]) && ad.w[k] >= 0.0 && std::isfinite(ad.fw[k]) && ad.fw[k] >= 0.0))
            return fail(NESOSIM_ERR_ARG, "the objective's weights must be finite and >= 0");
    if (!ctx->obs.ready || !ctx->obs.general)
        return fail(NESOSIM_ERR_STATE, "the adjoint needs observations registered on the general path (nesosim_set_path(ctx, 1) first)");
    auto &ob = ctx->obs;
    if (ob.n_fp && !fp_chi2_dev) return fail(NESOSIM_ERR_STATE, "footprints are registered: fp_chi2_dev is required");
    if (model_dev && model_stride < ob.row_len) return fail(NESOSIM_ERR_ARG, "model_stride is shorter than the observation row");
    if (ob.n_fp && fp_model_dev && fp_model_stride < ob.fp_row_len)
        return fail(NESOSIM_ERR_ARG, "fp_model_stride is shorter than the footprint row");
    if (ctx->cfg.n_members > 65535 || (ctx->cfg.ny + TY - 1) / TY > 65535)
        return fail(NESOSIM_ERR_ARG, "members or tile rows exceed the day kernel's grid dimensions");
    if (!ctx->P) return fail(NESOSIM_ERR_STATE, "nesosim_set_forcing has not been called");
    const bool sets = !ob.set_days.empty();
    if (!sets && ctx->member_set_dev) return fail(NESOSIM_ERR_ARG, "misfit mode runs on one shared forcing");
    if (sets && ob.set_days != ctx->set_days)
        return fail(NESOSIM_ERR_STATE, "the forcing sets changed since nesosim_set_observations_sets; register the observations again");
    if (ctx->path != 1)
        return fail(NESOSIM_ERR_STATE, "the kernel path changed since the observations were registered; register them again");
    CU(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const nesosim_config &c = ctx->cfg;
    const int T = c.num_days, M = c.n_members;
    const long long plane = ctx->plane, layer = (long long)M * plane;
    int rc;
    if (!ob.adj_begin) {          // both tables or neither: a failed upload leaves nothing behind
        int *b = nullptr;
        int2 *it = nullptr;
        if ((rc = upload_vec(&b, ob.adj_begin_h)) || (rc = upload_vec(&it, ob.adj_item_h))) {
            cudaFree(b);
            cudaFree(it);
            cudaGetLastError();
            return rc;
        }
        ob.adj_begin = b;
        ob.adj_item = it;
    }
    if ((rc = adj_alloc(&ob.traj, (size_t)T * 2 * layer)) || (rc = adj_alloc(&ob.rec_flags, (size_t)std::max(1, T - 1) * layer)) ||
        (rc = adj_alloc(&ob.lam, (size_t)4 * layer)) || (rc = adj_alloc(&ob.theta_acc, (size_t)GRAD_DIRS * layer)) ||
        (rc = adj_alloc(&ob.seeds, (size_t)M * ob.stride)) ||
        (rc = adj_alloc(&ob.fp_coef, (size_t)M * std::max(1LL, ob.fp_row_len))) ||
        (fo && ((rc = adj_alloc(&ob.cseed, (size_t)M * ob.stride)) ||
                (rc = adj_alloc(&ob.forcing_acc, (size_t)FORCING_DIRS * layer)))) ||
        (dro && (rc = adj_alloc(&ob.drift_acc, (size_t)DRIFT_DIRS * layer)))) {
        adj_release(ob);          // what did fit is not kept for a call that cannot run
        return rc;
    }
    if ((rc = upload_coef(ctx, params_host, st))) return rc;
    ctx->last_path = 1;
    CU(cudaMemsetAsync(ob.theta_acc, 0, (size_t)GRAD_DIRS * layer * sizeof(double), st));
    if (fo) CU(cudaMemsetAsync(ob.forcing_acc, 0, (size_t)FORCING_DIRS * layer * sizeof(double), st));
    if (dro) CU(cudaMemsetAsync(ob.drift_acc, 0, (size_t)DRIFT_DIRS * layer * sizeof(double), st));
    if ((rc = run_score_days(ctx, ic_dev, ic_per_member, st, false, true))) return rc;
    if (model_dev && ob.row_len)
        CU(cudaMemset2DAsync(model_dev, (size_t)model_stride * sizeof(double), 0xff, (size_t)ob.row_len * sizeof(double), M, st));
    MisfitArgs ma;
    ma.samples = ob.samples; ma.stride = ob.stride;
    ma.obs_slot = ob.o_slot; ma.obs_day = ob.o_day; ma.obs_cell = ob.o_cell; ma.src = ob.src;
    ma.obs_val = ob.val; ma.sigma = ob.sigma; ma.kind_begin = ob.kind_begin;
    ma.conc = ctx->C; ma.plane = plane; ma.k = ctx->k;
    ma.chi2 = chi2_dev; ma.count = (long long *)count_dev; ma.n_kinds = NESOSIM_OBS_KINDS;
    ma.model = model_dev; ma.model_stride = model_stride;
    ma.member_set = ctx->member_set_dev; ma.conc_set_stride = (long long)T * plane;
    ma.fp_chi2 = nullptr; ma.fp_count = nullptr;
    if (ob.n_fp) {
        if (ob.fp_row_len) {
            FootprintArgs fa;
            fa.samples = ob.samples; fa.stride = ob.stride;
            fa.begin = ob.fp_begin; fa.kind = ob.fp_kind; fa.src = ob.fp_src;
            fa.pt_slot = ob.pt_slot; fa.pt_day = ob.pt_day; fa.pt_cell = ob.pt_cell; fa.pt_w = ob.pt_w;
            fa.kind_begin = ob.fp_kind_begin; fa.conc = ctx->C; fa.plane = plane; fa.k = ctx->k;
            fa.n_members = M; fa.row_len = ob.fp_row_len; fa.mean = ob.fp_mean; fa.mean_stride = ob.fp_row_len;
            fa.model = fp_model_dev; fa.model_stride = fp_model_stride;
            fa.member_set = ctx->member_set_dev; fa.conc_set_stride = (long long)T * plane;
            const long long blocks = ob.fp_row_len * M;
            if (blocks > INT_MAX) return fail(NESOSIM_ERR_ARG, "too many footprints x members for one launch");
            FootprintAdj fj;
            fj.coef = ob.fp_coef; fj.val = ob.fp_val; fj.sigma = ob.fp_sigma;
            for (int k = 0; k < NESOSIM_OBS_KINDS; ++k) fj.fw[k] = ad.fw[k];
            if (sets) footprint_mean_adj_kernel<true><<<(unsigned)blocks, 32, 0, st>>>(fa, fj);
            else footprint_mean_adj_kernel<false><<<(unsigned)blocks, 32, 0, st>>>(fa, fj);
            ctx->launches++;
            CU(cudaGetLastError());
        }
        ma.fp_mean = ob.fp_mean; ma.fp_stride = std::max(1LL, ob.fp_row_len);
        ma.fp_val = ob.fp_val; ma.fp_sigma = ob.fp_sigma; ma.fp_kind_begin = ob.fp_kind_begin;
        ma.fp_chi2 = fp_chi2_dev; ma.fp_count = (long long *)fp_count_dev;
    }
    if (sets) misfit_finish_kernel<true><<<M, 256, 0, st>>>(ma);
    else misfit_finish_kernel<false><<<M, 256, 0, st>>>(ma);
    ctx->launches++;
    CU(cudaGetLastError());

    SeedArgs sd;
    sd.samples = ob.samples; sd.seeds = ob.seeds; sd.stride = ob.stride;
    sd.begin = ob.adj_begin; sd.item = ob.adj_item;
    sd.obs_day = ob.o_day; sd.obs_cell = ob.o_cell; sd.obs_val = ob.val; sd.sigma = ob.sigma;
    sd.fp_coef = ob.fp_coef; sd.fp_stride = std::max(1LL, ob.fp_row_len);
    sd.fp_kind = ob.fp_kind; sd.fp_kind_begin = ob.fp_kind_begin; sd.pt_day = ob.pt_day; sd.pt_cell = ob.pt_cell;
    sd.pt_w = ob.pt_w; sd.conc = ctx->C; sd.plane = plane; sd.conc_set_stride = (long long)T * plane;
    sd.member_set = ctx->member_set_dev; sd.k = ctx->k;
    for (int k = 0; k < NESOSIM_OBS_KINDS; ++k) sd.w[k] = ad.w[k];
    if (ob.stride) {              // a grid without an ocean cell has no sample slot and nothing to seed
        const dim3 sg((unsigned)((ob.stride + 255) / 256), M);
        if (fo) adjoint_seed_forcing_kernel<<<sg, 256, 0, st>>>(sd, ob.cseed);
        else adjoint_seed_kernel<<<sg, 256, 0, st>>>(sd);
        ctx->launches++;
        CU(cudaGetLastError());
    }

    AdjInitArgs ai;
    ai.lam = ob.lam; ai.plane = plane; ai.layer_stride = layer; ai.seeds = ob.seeds; ai.stride = ob.stride;
    ai.begin = ob.smp_begin; ai.entry = ob.smp_entry; ai.T = T; ai.tiles = ob.smp_tiles;
    ai.member_set = ctx->member_set_dev; ai.set_steps = ctx->set_steps_dev;
    ForcingInitArgs fi{};
    ForcingAdjArgs fj{};
    if (fo) {
        fi.cseed = fj.cseed = ob.cseed;
        fi.acc = fj.acc = ob.forcing_acc;
        fi.conc = ctx->C;
        for (int f = 0; f < FORCING_DIRS; ++f) fi.day[f] = fo->day[f];
        fj.day_mstride = (long long)T * plane;
        adjoint_init_forcing_kernel<<<M, 256, 0, st>>>(ai, fi);
    } else {
        adjoint_init_kernel<<<M, 256, 0, st>>>(ai);
    }
    ctx->launches++;
    CU(cudaGetLastError());

    auto lam = [&](int t) { return ob.lam + (long long)(t & 1) * 2 * layer; };
    AdjArgs aj;
    aj.layer_stride = layer; aj.theta = ob.theta_acc; aj.seeds = ob.seeds;
    aj.begin = ob.smp_begin; aj.entry = ob.smp_entry; aj.stride = ob.stride; aj.T = T; aj.tiles = ob.smp_tiles;
    const dim3 grid((c.nx + TX - 1) / TX, (c.ny + TY - 1) / TY, M);
    DriftAdjArgs dj{};
    size_t drift_smem = 0;
    void (*drift_kernel)(const DayArgs, const AdjArgs, const DriftAdjArgs) = nullptr;
    void (*forcing_drift_kernel)(const DayArgs, const AdjArgs, const ForcingAdjArgs, const DriftAdjArgs) = nullptr;
    if (dro) {
        dj.acc = ob.drift_acc;
        dj.day_mstride = (long long)T * DRIFT_DIRS * plane;
        if (fo) {
            forcing_drift_kernel = ctx->day_variant == 512 ? day_step_adjoint_forcing_drift_kernel_512
                                                           : day_step_adjoint_forcing_drift_kernel;
            drift_smem = sizeof(AdjDriftSmem<true>);
            CU(allow_drift_smem(forcing_drift_kernel, drift_smem));
        } else {
            drift_kernel = ctx->day_variant == 512 ? day_step_adjoint_drift_kernel_512 : day_step_adjoint_drift_kernel;
            drift_smem = sizeof(AdjDriftSmem<false>);
            CU(allow_drift_smem(drift_kernel, drift_smem));
        }
    }
    nesosim_outputs none{};
    for (int x = T - 2; x >= 0; --x) {
        DayArgs a;
        fill_day_args(ctx, x, ctx->P + x * plane, ctx->C + x * plane, ctx->W + x * plane, ctx->UV + (long long)x * 2 * plane,
                      ctx->UV + ((long long)x * 2 + 1) * plane, c.snowDensityFresh, &none, 0, x > 0, a);
        for (int v = 0; v < NVAR; ++v) a.prev[v] = a.next[v] = nullptr;
        a.depth_mstride = a.plane_mstride = plane;
        aj.lam_in = lam(x + 1);
        aj.lam_out = lam(x);
        aj.h0 = ob.traj + (long long)x * 2 * layer;
        aj.flags = ob.rec_flags + (long long)x * layer;
        const bool pdl = ctx->pdl && x < T - 2;   // behind this call's own previous backward kernel only
        if (fo) for (int f = 0; f < FORCING_DIRS; ++f) fj.day[f] = fo->day[f] ? fo->day[f] + (long long)x * plane : nullptr;
        if (dro) {
            dj.day = dro->day ? dro->day + (long long)x * DRIFT_DIRS * plane : nullptr;
            if (fo) CU(launch_day_kernel_smem(forcing_drift_kernel, grid, ctx->day_variant, drift_smem, st, pdl, a, aj, fj, dj));
            else CU(launch_day_kernel_smem(drift_kernel, grid, ctx->day_variant, drift_smem, st, pdl, a, aj, dj));
        } else if (fo) {
            if (ctx->day_variant == 512) CU(launch_day_kernel(day_step_adjoint_forcing_kernel_512, grid, 512, st, pdl, a, aj, fj));
            else CU(launch_day_kernel(day_step_adjoint_forcing_kernel, grid, 256, st, pdl, a, aj, fj));
        } else if (ctx->day_variant == 512) {
            CU(launch_day_kernel(day_step_adjoint_kernel_512, grid, 512, st, pdl, a, aj));
        } else {
            CU(launch_day_kernel(day_step_adjoint_kernel, grid, 256, st, pdl, a, aj));
        }
        ctx->launches++;
    }
    AdjFinishArgs af;
    af.theta_acc = ob.theta_acc; af.lam0 = ob.lam; af.plane = plane; af.layer_stride = layer;
    af.conc0 = ctx->C; af.set_stride = (long long)T * plane; af.member_set = ctx->member_set_dev; af.minConc = c.minConc;
    af.theta_grad = ad.theta_grad; af.ic_grad = ad.ic_grad;
    const ForcingFinishArgs ff{ob.forcing_acc, fo ? fo->scale_grad : nullptr, fo ? fo->scale_total : nullptr};
    const DriftFinishArgs df{ob.drift_acc, dro ? dro->scale_grad : nullptr, dro ? dro->scale_total : nullptr,
                             dro ? dro->day : nullptr, ctx->set_steps_dev, T};
    if (fo && dro) adjoint_finish_forcing_drift_kernel<<<M, 256, 0, st>>>(af, ff, df);
    else if (dro) adjoint_finish_drift_kernel<<<M, 256, 0, st>>>(af, df);
    else if (fo) adjoint_finish_forcing_kernel<<<M, 256, 0, st>>>(af, ff);
    else adjoint_finish_kernel<<<M, 256, 0, st>>>(af);
    ctx->launches++;
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

extern "C" {

// Observations of the calibration driver, compiled against the strip tables and kept on the device until they are
// replaced: -> (strip, index in the strip's ocean list), sorted by owner and day, one sentinel per ocean cell.
int nesosim_set_observations(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_day_host, const int32_t *obs_row_host,
                             const int32_t *obs_col_host, const double *obs_depth_host) {
    return register_observations(ctx, false, n_obs, nullptr, obs_day_host, obs_row_host, obs_col_host, nullptr,
                                 obs_depth_host, nullptr);
}

int nesosim_set_observations_sets(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_set_host, const int32_t *obs_day_host,
                                  const int32_t *obs_row_host, const int32_t *obs_col_host, const double *obs_depth_host) {
    return register_observations(ctx, true, n_obs, obs_set_host, obs_day_host, obs_row_host, obs_col_host, nullptr,
                                 obs_depth_host, nullptr);
}

int nesosim_set_observations_ex(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_set_host, const int32_t *obs_day_host,
                                const int32_t *obs_row_host, const int32_t *obs_col_host, const int32_t *obs_kind_host,
                                const double *obs_value_host, const double *obs_sigma_host) {
    return register_observations(ctx, obs_set_host != nullptr, n_obs, obs_set_host, obs_day_host, obs_row_host,
                                 obs_col_host, obs_kind_host, obs_value_host, obs_sigma_host);
}

int nesosim_observation_row_length(const nesosim_ctx *ctx, int64_t *row_len) {
    if (!ctx || !row_len) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (!ctx->obs.ready) return fail(NESOSIM_ERR_STATE, "no observations are registered");
    *row_len = ctx->obs.row_len;
    return NESOSIM_OK;
}

int nesosim_run_season_misfit(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                              int ic_per_member, double *misfit_dev, int64_t *count_dev, void *stream) {
    return run_season_scores(ctx, params_host, ic_dev, ic_per_member, misfit_dev, count_dev, 1, nullptr, 0, stream);
}

int nesosim_run_season_scores(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                              int ic_per_member, double *chi2_dev, int64_t *count_dev, double *model_dev,
                              int64_t model_stride, void *stream) {
    return run_season_scores(ctx, params_host, ic_dev, ic_per_member, chi2_dev, count_dev, NESOSIM_OBS_KINDS, model_dev,
                             model_stride, stream);
}

int nesosim_set_observations_fp(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_set_host, const int32_t *obs_day_host,
                                const int32_t *obs_row_host, const int32_t *obs_col_host, const int32_t *obs_kind_host,
                                const double *obs_value_host, const double *obs_sigma_host, int64_t n_fp,
                                const int32_t *fp_set_host, const int32_t *fp_kind_host, const double *fp_value_host,
                                const double *fp_sigma_host, const int64_t *fp_begin_host, const int32_t *pt_day_host,
                                const int32_t *pt_row_host, const int32_t *pt_col_host, const double *pt_weight_host) {
    return register_observations(ctx, obs_set_host != nullptr || fp_set_host != nullptr, n_obs, obs_set_host,
                                 obs_day_host, obs_row_host, obs_col_host, obs_kind_host, obs_value_host, obs_sigma_host,
                                 n_fp, fp_set_host, fp_kind_host, fp_value_host, fp_sigma_host, fp_begin_host,
                                 pt_day_host, pt_row_host, pt_col_host, pt_weight_host);
}

int nesosim_footprint_row_length(const nesosim_ctx *ctx, int64_t *row_len) {
    if (!ctx || !row_len) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (!ctx->obs.ready) return fail(NESOSIM_ERR_STATE, "no observations are registered");
    *row_len = ctx->obs.fp_row_len;
    return NESOSIM_OK;
}

int nesosim_run_season_scores_fp(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                                 int ic_per_member, double *chi2_dev, int64_t *count_dev, double *model_dev,
                                 int64_t model_stride, double *fp_chi2_dev, int64_t *fp_count_dev, double *fp_model_dev,
                                 int64_t fp_model_stride, void *stream) {
    return run_season_scores(ctx, params_host, ic_dev, ic_per_member, chi2_dev, count_dev, NESOSIM_OBS_KINDS, model_dev,
                             model_stride, stream, true, fp_chi2_dev, fp_count_dev, fp_model_dev, fp_model_stride);
}

int nesosim_run_season_score_grads(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                                   int ic_per_member, double *chi2_dev, int64_t *count_dev, double *model_dev,
                                   int64_t model_stride, double *grad_dev, double *jac_dev, int64_t jac_stride,
                                   double *fp_chi2_dev, int64_t *fp_count_dev, double *fp_model_dev,
                                   int64_t fp_model_stride, double *fp_grad_dev, double *fp_jac_dev, int64_t fp_jac_stride,
                                   void *stream) {
    const GradOutputs g{grad_dev, jac_dev, jac_stride, fp_grad_dev, fp_jac_dev, fp_jac_stride};
    return run_season_scores(ctx, params_host, ic_dev, ic_per_member, chi2_dev, count_dev, NESOSIM_OBS_KINDS, model_dev,
                             model_stride, stream, false, fp_chi2_dev, fp_count_dev, fp_model_dev, fp_model_stride, &g);
}

int nesosim_run_season_score_adjoint(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                                     int ic_per_member, const double *weights_host, const double *fp_weights_host,
                                     double *chi2_dev, int64_t *count_dev, double *model_dev, int64_t model_stride,
                                     double *fp_chi2_dev, int64_t *fp_count_dev, double *fp_model_dev,
                                     int64_t fp_model_stride, double *theta_grad_dev, double *ic_grad_dev, void *stream) {
    const AdjOutputs ad{weights_host, fp_weights_host, theta_grad_dev, ic_grad_dev};
    return run_season_score_adjoint(ctx, params_host, ic_dev, ic_per_member, chi2_dev, count_dev, model_dev, model_stride,
                                    fp_chi2_dev, fp_count_dev, fp_model_dev, fp_model_stride, ad, stream);
}

int nesosim_run_season_score_adjoint_forcing(nesosim_ctx *ctx, const nesosim_member_params *params_host,
                                             const double *ic_dev, int ic_per_member, const double *weights_host,
                                             const double *fp_weights_host, double *chi2_dev, int64_t *count_dev,
                                             double *model_dev, int64_t model_stride, double *fp_chi2_dev,
                                             int64_t *fp_count_dev, double *fp_model_dev, int64_t fp_model_stride,
                                             double *theta_grad_dev, double *ic_grad_dev,
                                             double *forcing_scale_grad_dev, double *forcing_scale_total_dev,
                                             double *precip_day_dev, double *wind_day_dev, double *conc_day_dev,
                                             void *stream) {
    const AdjOutputs ad{weights_host, fp_weights_host, theta_grad_dev, ic_grad_dev};
    const ForcingOutputs fo{forcing_scale_grad_dev, forcing_scale_total_dev, {precip_day_dev, wind_day_dev, conc_day_dev}};
    return run_season_score_adjoint(ctx, params_host, ic_dev, ic_per_member, chi2_dev, count_dev, model_dev, model_stride,
                                    fp_chi2_dev, fp_count_dev, fp_model_dev, fp_model_stride, ad, stream, &fo);
}

int nesosim_run_season_score_adjoint_drift(nesosim_ctx *ctx, const nesosim_member_params *params_host,
                                           const double *ic_dev, int ic_per_member, const double *weights_host,
                                           const double *fp_weights_host, double *chi2_dev, int64_t *count_dev,
                                           double *model_dev, int64_t model_stride, double *fp_chi2_dev,
                                           int64_t *fp_count_dev, double *fp_model_dev, int64_t fp_model_stride,
                                           double *theta_grad_dev, double *ic_grad_dev,
                                           double *forcing_scale_grad_dev, double *forcing_scale_total_dev,
                                           double *precip_day_dev, double *wind_day_dev, double *conc_day_dev,
                                           double *drift_scale_grad_dev, double *drift_scale_total_dev,
                                           double *drift_day_dev, void *stream) {
    const bool forcing = forcing_scale_grad_dev || forcing_scale_total_dev;
    if (forcing && !(forcing_scale_grad_dev && forcing_scale_total_dev))
        return fail(NESOSIM_ERR_ARG, "forcing_scale_grad_dev and forcing_scale_total_dev are given together or not at all");
    if (!forcing && (precip_day_dev || wind_day_dev || conc_day_dev))
        return fail(NESOSIM_ERR_ARG, "per-day forcing gradients need forcing_scale_grad_dev and forcing_scale_total_dev");
    const AdjOutputs ad{weights_host, fp_weights_host, theta_grad_dev, ic_grad_dev};
    const ForcingOutputs fo{forcing_scale_grad_dev, forcing_scale_total_dev, {precip_day_dev, wind_day_dev, conc_day_dev}};
    const DriftOutputs dro{drift_scale_grad_dev, drift_scale_total_dev, drift_day_dev};
    return run_season_score_adjoint(ctx, params_host, ic_dev, ic_per_member, chi2_dev, count_dev, model_dev, model_stride,
                                    fp_chi2_dev, fp_count_dev, fp_model_dev, fp_model_stride, ad, stream,
                                    forcing ? &fo : nullptr, &dro);
}

int nesosim_set_async(nesosim_ctx *ctx, int on) {
    if (!ctx) return fail(NESOSIM_ERR_ARG, "NULL context");
    CU(cudaSetDevice(ctx->cfg.device));
    if (!on) {
        int rc = resolve_pending(ctx, true, nullptr);
        if (rc) return rc;
    }
    if (on && !ctx->flag_pool) CU(cudaMallocHost(&ctx->flag_pool, 256 * sizeof(int)));
    ctx->async_mode = on != 0;
    return NESOSIM_OK;
}

int nesosim_sync(nesosim_ctx *ctx, int *seasons_redone) {
    if (!ctx) return fail(NESOSIM_ERR_ARG, "NULL context");
    CU(cudaSetDevice(ctx->cfg.device));
    if (seasons_redone) *seasons_redone = 0;
    return resolve_pending(ctx, true, seasons_redone);
}

int nesosim_step_day(nesosim_ctx *ctx, int x, const double *conc_dev, const double *precip_dev,
                     const double *drift_dev, const double *wind_dev, double rho_new,
                     const nesosim_member_params *params_host, const nesosim_outputs *out, void *stream) {
    if (!ctx || !conc_dev || !precip_dev || !drift_dev || !wind_dev || !params_host)
        return fail(NESOSIM_ERR_ARG, "NULL argument");
    if (x < 0 || x + 1 >= ctx->cfg.num_days) return fail(NESOSIM_ERR_ARG, "x outside [0, num_days-2]");
    int rc = check_outputs(ctx, out);
    if (rc) return rc;
    if (any_missing(out)) return fail(NESOSIM_ERR_ARG, "nesosim_step_day needs every accumulator and snowDepths (density optional)");
    CU(cudaSetDevice(ctx->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = upload_coef(ctx, params_host, st))) return rc;
    return launch_day(ctx, x, precip_dev, conc_dev, wind_dev, drift_dev, drift_dev + ctx->plane, rho_new, out, 0,
                      ctx->cfg.n_members, st);
}

int nesosim_smooth(const double *in_dev, double *out_dev, int ny, int nx, const double weights_host[9],
                   double divisor, void *stream) {
    if (!in_dev || !out_dev || !weights_host || ny < 1 || nx < 1 || in_dev == out_dev)
        return fail(NESOSIM_ERR_ARG, "bad argument to nesosim_smooth");
    cudaStream_t st = (cudaStream_t)stream;
    int *flags;
    CU(cudaMallocAsync(&flags, sizeof(int), st));
    CU(cudaMemsetAsync(flags, 0, sizeof(int), st));
    const long long n = (long long)ny * nx;
    scan_nonfinite_kernel<<<(unsigned)std::min<long long>((n + 255) / 256, 1184), 256, 0, st>>>(in_dev, n, flags);
    SmoothArgs a;
    a.in = in_dev; a.out = out_dev; a.ny = ny; a.nx = nx;
    std::memcpy(a.w, weights_host, sizeof(a.w));
    a.div = const_div_host(divisor);
    a.flags = flags;
    dim3 blk(32, 8), grid((nx + 31) / 32, (ny + 7) / 8);
    smooth_kernel<<<grid, blk, 0, st>>>(a);
    CU(cudaGetLastError());
    CU(cudaFreeAsync(flags, st));
    return NESOSIM_OK;
}

int nesosim_op_dynamics(const double *drift_dev, const double *depths_dev, double dx, double deltaT, int ny,
                        int nx, double *adv_dev, double *div_dev, void *stream) {
    if (!drift_dev || !depths_dev || !adv_dev || !div_dev || ny < 2 || nx < 2) return fail(NESOSIM_ERR_ARG, "bad argument");
    GradConsts g;
    g.dx = const_div_host(dx);
    g.two_dx = const_div_host(2. * dx);
    dim3 blk(32, 8), grid((nx + 31) / 32, (ny + 7) / 8);
    op_dynamics_kernel<<<grid, blk, 0, (cudaStream_t)stream>>>(drift_dev, depths_dev, ny, nx, deltaT, g, adv_dev, div_dev);
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

int nesosim_op_wind_terms(const double *h0_dev, const double *wind_dev, const double *conc_dev, int64_t n,
                          const nesosim_member_params *p, double deltaT, double rhoFresh, double rhoOld,
                          double *lead_dev, double *atm_dev, double *wp_loss_dev, double *wp_gain_dev,
                          double *wp_net_dev, void *stream) {
    if (!h0_dev || !wind_dev || !conc_dev || !p || n < 0) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (n == 0) return NESOSIM_OK;
    MemberCoef mc{p->leadLossFactor, p->atmLossFactor, p->windPackThresh, (-p->windPackFactor) * deltaT,
                  p->windPackFactor * deltaT};
    ModelConsts k{deltaT, rhoFresh, rhoOld, rhoFresh / rhoOld, 0.0, 0.0};
    op_wind_terms_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        h0_dev, wind_dev, conc_dev, n, mc, k, lead_dev, atm_dev, wp_loss_dev, wp_gain_dev, wp_net_dev);
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

int nesosim_op_fill_zero(double *arr_dev, int64_t n, void *stream) {
    if (!arr_dev || n < 0) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (n == 0) return NESOSIM_OK;
    op_fill_zero_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(arr_dev, n);
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

int nesosim_op_fill_nan_no_negative(double *arr_dev, const uint8_t *mask_dev, int64_t n, int negative_to_zero,
                                    void *stream) {
    if (!arr_dev || !mask_dev || n < 0) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (n == 0) return NESOSIM_OK;
    op_fill_nan_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(arr_dev, mask_dev, n, negative_to_zero);
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

int nesosim_op_density(const double *depths_dev, const uint8_t *mask_dev, int64_t n, double rhoFresh,
                       double rhoOld, double minSnowD, double *density_dev, void *stream) {
    if (!depths_dev || !mask_dev || !density_dev || n < 0) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (n == 0) return NESOSIM_OK;
    ModelConsts k{0.0, rhoFresh, rhoOld, rhoFresh / rhoOld, minSnowD, 0.0};
    op_density_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(depths_dev, mask_dev, n, k, density_dev);
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

int nesosim_final_products(const double *depths_dev, const double *density_dev, const double *conc_dev,
                           const double *precip_dev, const double *wind_dev, int num_days, int forcing_days, int64_t plane,
                           double ice_conc_mask, float *snow_depth_dev, float *snow_volume_dev,
                           float *snow_density_dev, float *ice_conc_dev, float *precip_out_dev, float *wind_out_dev,
                           void *stream) {
    if (!depths_dev || !conc_dev || num_days < 1 || plane < 1 || forcing_days < 0) return fail(NESOSIM_ERR_ARG, "bad argument");
    if (forcing_days == 0) forcing_days = num_days;
    if (num_days % forcing_days) return fail(NESOSIM_ERR_ARG, "num_days must be a multiple of forcing_days");
    if (snow_density_dev && !density_dev) return fail(NESOSIM_ERR_ARG, "snow_density wanted but density is NULL");
    if ((precip_out_dev && !precip_dev) || (wind_out_dev && !wind_dev)) return fail(NESOSIM_ERR_ARG, "forcing output wanted but its input is NULL");
    FinalArgs a;
    a.depths = depths_dev; a.density = density_dev; a.conc = conc_dev; a.precip = precip_dev; a.wind = wind_dev;
    a.plane = plane; a.n = (long long)num_days * plane; a.forcing_days = forcing_days; a.ice_conc_mask = ice_conc_mask;
    a.snow_depth = snow_depth_dev; a.snow_volume = snow_volume_dev; a.snow_density = snow_density_dev;
    a.ice_conc = ice_conc_dev; a.precip_out = precip_out_dev; a.wind_out = wind_out_dev;
    const unsigned blocks = (unsigned)std::min<long long>((a.n + 255) / 256, 148 * 16);
    final_products_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(a);
    CU(cudaGetLastError());
    return NESOSIM_OK;
}

int64_t nesosim_launch_count(const nesosim_ctx *ctx) { return ctx ? ctx->launches : 0; }
int64_t nesosim_rerun_count(const nesosim_ctx *ctx) { return ctx ? ctx->ens_reruns : 0; }

int nesosim_host_drain_info(const nesosim_ctx *ctx, int *compacted, int64_t *full_chunks) {
    if (!ctx) return fail(NESOSIM_ERR_ARG, "NULL context");
    if (compacted) *compacted = ctx->hp_last_compact;
    if (full_chunks) *full_chunks = ctx->hp_full_chunks;
    return NESOSIM_OK;
}

int nesosim_host_drain_blocks(const nesosim_ctx *ctx, int64_t *packed, int64_t *plain) {
    if (!ctx) return fail(NESOSIM_ERR_ARG, "NULL context");
    if (packed) *packed = ctx->hp_last_compact ? ctx->hp_blocks_packed : 0;
    if (plain) *plain = ctx->hp_last_compact ? ctx->hp_blocks_plain : 0;
    return NESOSIM_OK;
}
int nesosim_season_kernel_time(const nesosim_ctx *ctx, double *total_ms, int64_t *launches) {
    if (!ctx || !total_ms || !launches) return fail(NESOSIM_ERR_ARG, "NULL argument");
    *total_ms = ctx->ens_kernel_ms;           // (asynchronous launches count once nesosim_sync / a later call has seen them)
    *launches = ctx->ens_kernel_launches;
    return NESOSIM_OK;
}

// ---- row-strip domain decomposition over peer memory

int nesosim_strip_setup(nesosim_ctx *ctx, int has_up, int has_dn) {
    if (!ctx) return fail(NESOSIM_ERR_ARG, "NULL context");
    if (ctx->cfg.n_members != 1 || ctx->n_sets != 1)
        return fail(NESOSIM_ERR_ARG, "strips are for a single member on a single forcing set");
    const int ghosts = (has_up ? STRIP_GHOST : 0) + (has_dn ? STRIP_GHOST : 0);
    if (ctx->cfg.ny < ghosts + STRIP_GHOST)
        return fail(NESOSIM_ERR_ARG, "a strip must own at least two rows besides its ghost rows");
    CU(cudaSetDevice(ctx->cfg.device));
    strip_release(ctx);
    const size_t bytes = strip_block_bytes(ctx->cfg.nx);
    CU(cudaMalloc(&ctx->strip.block, bytes));
    CU(cudaMemset(ctx->strip.block, 0, bytes));
    CU(cudaDeviceSynchronize());
    ctx->strip.has_up = has_up != 0;
    ctx->strip.has_dn = has_dn != 0;
    ctx->strip.epoch = 0;
    ctx->strip.on = true;
    return NESOSIM_OK;
}

int nesosim_strip_block(nesosim_ctx *ctx, void **block_dev, int64_t *bytes) {
    if (!ctx || !ctx->strip.on) return fail(NESOSIM_ERR_STATE, "nesosim_strip_setup has not been called");
    if (block_dev) *block_dev = ctx->strip.block;
    if (bytes) *bytes = (int64_t)strip_block_bytes(ctx->cfg.nx);
    return NESOSIM_OK;
}

int nesosim_strip_export(nesosim_ctx *ctx, void *handle64) {
    if (!ctx || !handle64) return fail(NESOSIM_ERR_ARG, "NULL argument");
    if (!ctx->strip.on) return fail(NESOSIM_ERR_STATE, "nesosim_strip_setup has not been called");
    static_assert(sizeof(cudaIpcMemHandle_t) == NESOSIM_IPC_HANDLE_BYTES, "IPC handle size");
    CU(cudaSetDevice(ctx->cfg.device));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, ctx->strip.block));
    std::memcpy(handle64, &h, sizeof(h));
    return NESOSIM_OK;
}

int nesosim_strip_connect_local(nesosim_ctx *ctx, void *up_block_dev, void *dn_block_dev) {
    if (!ctx || !ctx->strip.on) return fail(NESOSIM_ERR_STATE, "nesosim_strip_setup has not been called");
    if ((ctx->strip.has_up && !up_block_dev) || (ctx->strip.has_dn && !dn_block_dev))
        return fail(NESOSIM_ERR_ARG, "a neighbour declared in nesosim_strip_setup is missing");
    if (ctx->strip.ipc_up && ctx->strip.peer_up) cudaIpcCloseMemHandle(ctx->strip.peer_up);      // reconnecting
    if (ctx->strip.ipc_dn && ctx->strip.peer_dn) cudaIpcCloseMemHandle(ctx->strip.peer_dn);
    ctx->strip.peer_up = ctx->strip.has_up ? (char *)up_block_dev : nullptr;
    ctx->strip.peer_dn = ctx->strip.has_dn ? (char *)dn_block_dev : nullptr;
    ctx->strip.ipc_up = ctx->strip.ipc_dn = false;
    return NESOSIM_OK;
}

int nesosim_strip_connect(nesosim_ctx *ctx, const void *up_handle64, const void *dn_handle64) {
    if (!ctx || !ctx->strip.on) return fail(NESOSIM_ERR_STATE, "nesosim_strip_setup has not been called");
    if ((ctx->strip.has_up && !up_handle64) || (ctx->strip.has_dn && !dn_handle64))
        return fail(NESOSIM_ERR_ARG, "a neighbour declared in nesosim_strip_setup is missing");
    CU(cudaSetDevice(ctx->cfg.device));
    if (ctx->strip.ipc_up && ctx->strip.peer_up) cudaIpcCloseMemHandle(ctx->strip.peer_up);      // reconnecting
    if (ctx->strip.ipc_dn && ctx->strip.peer_dn) cudaIpcCloseMemHandle(ctx->strip.peer_dn);
    ctx->strip.peer_up = ctx->strip.peer_dn = nullptr;
    ctx->strip.ipc_up = ctx->strip.ipc_dn = false;
    auto open = [&](const void *h64, char **out) -> int {
        cudaIpcMemHandle_t h;
        std::memcpy(&h, h64, sizeof(h));
        void *p = nullptr;
        CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        *out = (char *)p;
        return NESOSIM_OK;
    };
    int rc;
    if (ctx->strip.has_up) {
        if ((rc = open(up_handle64, &ctx->strip.peer_up))) return rc;
        ctx->strip.ipc_up = true;
    }
    if (ctx->strip.has_dn) {
        if ((rc = open(dn_handle64, &ctx->strip.peer_dn))) return rc;
        ctx->strip.ipc_dn = true;
    }
    return NESOSIM_OK;
}

int nesosim_strip_status(nesosim_ctx *ctx, int *timed_out) {
    if (!ctx || !timed_out) return fail(NESOSIM_ERR_ARG, "NULL argument");
    if (!ctx->strip.on) return fail(NESOSIM_ERR_STATE, "nesosim_strip_setup has not been called");
    CU(cudaSetDevice(ctx->cfg.device));
    const size_t off = 2 * strip_mail_bytes(ctx->cfg.nx) + 2 * sizeof(unsigned long long) + 2 * sizeof(unsigned int);
    CU(cudaMemcpy(timed_out, ctx->strip.block + off, sizeof(int), cudaMemcpyDeviceToHost));
    return NESOSIM_OK;
}

int nesosim_strip_set_timeout(nesosim_ctx *ctx, double seconds) {
    if (!ctx || !(seconds > 0)) return fail(NESOSIM_ERR_ARG, "bad argument");
    ctx->strip.timeout_s = seconds;
    return NESOSIM_OK;
}

int nesosim_set_path(nesosim_ctx *ctx, int path) {
    if (!ctx || path < 0 || path > 2) return fail(NESOSIM_ERR_ARG, "path must be 0 (auto), 1 (per-day kernel) or 2 (season-resident)");
    ctx->path = path;
    return NESOSIM_OK;
}

int nesosim_last_path(const nesosim_ctx *ctx) { return ctx ? ctx->last_path : 0; }

int nesosim_const_div_is_fast(double c) { return const_div_host(c).fast; }

double nesosim_const_div_eval_host(double x, double c) {
    const ConstDiv d = const_div_host(c);
    unsigned long long bits;
    std::memcpy(&bits, &x, 8);
    const unsigned e = (unsigned)(bits >> 52) & 0x7ffu;
    const double q0 = x * d.rc;
    if (d.fast && (e - 400u) <= 1246u) return std::fma(std::fma(-d.c, q0, x), d.rc, q0);
    if (e == 0x7ffu || x == 0.0) return q0;
    return x / d.c;
}

}  // extern "C"

#include "host_path.inl"
