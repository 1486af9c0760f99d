/* nesosim_b200.h -- C ABI of the B200-native NESOSIM daily snow-budget path.
 *
 * Drop-in boundary for ONE hot path of ac137/NESOSIM: `calcBudget` and its callees
 * (reference: source/NESOSIM.py:51-347,458-473) plus the day loop of `main` that drives it
 * (source/NESOSIM.py:586-649).  The reference is pure Python, so there is no existing FFI; these are the
 * entry points a ctypes binding for that path binds (see INTEGRATION.md for the reference-side stub).
 *
 * Conventions
 *   - plain C, no torch/CUDA types in signatures; `stream` is a cudaStream_t passed as void* (NULL = default).
 *   - every `*_dev` / "device pointer" argument is a CUDA device address (e.g. torch.Tensor.data_ptr());
 *     arguments documented "host" are ordinary host memory.
 *   - all fields are float64 unless stated; planes are dense row-major (ny rows, nx columns), time-major
 *     stacks are [T][ny][nx] exactly like the reference's numpy arrays (genEmptyArrays, NESOSIM.py:350-376).
 *   - functions return 0 (NESOSIM_OK) or a negative error code; nesosim_last_error() gives the message for
 *     the calling thread.  NaN/inf in the data are data, not errors (NESOSIM.py relies on NaN algebra).
 *   - the caller owns every buffer; the library allocates only an opaque context (and optional scratch).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns NESOSIM_ERR_CUDA.
 */
#ifndef NESOSIM_B200_H
#define NESOSIM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NESOSIM_ABI_VERSION 1

#define NESOSIM_OK            0
#define NESOSIM_ERR_ARG      -1   /* bad argument (NULL, non-positive size, ny or nx < 2, ...) */
#define NESOSIM_ERR_CUDA     -2   /* CUDA runtime error or no device */
#define NESOSIM_ERR_STATE    -3   /* call order (e.g. run_season before set_forcing) */
#define NESOSIM_ERR_NOMEM    -4

typedef struct nesosim_ctx nesosim_ctx;

/* Model constants `main` assigns to module globals (NESOSIM.py:527-541) + grid + switches of calcBudget
 * (NESOSIM.py:227).  conv_weights is `Gaussian2DKernel(x_stddev=1,x_size=3,y_size=3).array` (row-major 3x3)
 * and conv_divisor its `.sum()`, both computed by the HOST with numpy so the device uses bit-identical
 * constants (smooth_snow, NESOSIM.py:170-187); pass weights/sum and divisor 1.0 for a pre-normalised kernel. */
typedef struct nesosim_config {
    int32_t ny, nx;              /* grid rows / columns (>= 2 each: np.gradient needs two points)        */
    int32_t num_days;            /* T = numDays: number of time slots; the season has T-1 steps          */
    int32_t n_members;           /* M parameter sets sharing one forcing (1 for a plain `main` run)      */
    double  dx;                  /* grid spacing [m]: the `dx` argument of main / calcDynamics           */
    double  deltaT;              /* 86400.                                                               */
    double  snowDensityFresh;    /* 200.                                                                 */
    double  snowDensityOld;      /* 350.                                                                 */
    double  minSnowD;            /* 0.02                                                                 */
    double  minConc;             /* 0.15                                                                 */
    double  conv_weights[9];
    double  conv_divisor;
    int32_t dynamicsInc, leadlossInc, windpackInc, atmlossInc;
    int32_t density_clim;        /* 0: densityType='variable', 1: 'clim' (needs rho_clim)                */
    int32_t device;              /* CUDA device ordinal                                                  */
} nesosim_config;

/* Per-member coefficients: windPackFactorT, windPackThreshT, leadLossFactorT, atmLossFactorT of main. */
typedef struct nesosim_member_params {
    double windPackFactor, windPackThresh, leadLossFactor, atmLossFactor;
} nesosim_member_params;

/* The twelve arrays calcBudget advances (NESOSIM.py:264-347).  Device pointers; member m of variable v
 * starts at v + m*member_stride elements; within a member the layout is the reference's:
 * snowDepths [T][2][ny][nx], everything else [T][ny][nx].  NULL = not wanted (kept in internal scratch). */
typedef struct nesosim_outputs {
    double *snowDepths;
    double *density;
    double *snowAcc, *snowOcean, *snowAdv, *snowDiv, *snowLead, *snowAtm;
    double *snowWindPackLoss, *snowWindPackGain, *snowWindPack;
    int64_t depth_member_stride;   /* elements between members in snowDepths (>= T*2*ny*nx)             */
    int64_t plane_member_stride;   /* elements between members in every other array (>= T*ny*nx)         */
} nesosim_outputs;

int         nesosim_abi_version(void);
const char *nesosim_last_error(void);
/* Number of CUDA devices visible (0 on a CPU-only host; never fails). */
int         nesosim_device_count(void);

/* Context = grid, constants, region mask.  `region_mask_host` is ny*nx uint8 region codes (host memory);
 * only `>10` (land/coast) and `<1` (lakes) are ever tested (fill_nan_no_negative, NESOSIM.py:158-162). */
int nesosim_create(const nesosim_config *cfg, const uint8_t *region_mask_host, nesosim_ctx **out);
int nesosim_destroy(nesosim_ctx *ctx);

/* Register a season of forcing already resident in HBM (what loadData returns per day, NESOSIM.py:379-456,
 * stacked over T days): precip/conc/wind [T][ny][nx], drift [T][2][ny][nx], rho_clim [T] (fresh-snow density
 * per step for density_clim=1, else NULL).  Pointers are borrowed, not copied. */
int nesosim_set_forcing(nesosim_ctx *ctx, const double *precip_dev, const double *conc_dev,
                        const double *wind_dev, const double *drift_dev, const double *rho_clim_dev);

/* A batch of seasons in one context (the loop of run_multiseason.py:39-50 as one native call): `n_sets` independent
 * forcing stacks laid out [n_sets][T][ny][nx] (drift [n_sets][T][2][ny][nx]); member m runs on stack
 * member_set_host[m] for set_days_host[set] days (2 <= days <= T: seasons of different length, e.g. leap years).  Every
 * later nesosim_run_season advances each member through ITS season; output slots beyond a member's last day are left
 * untouched.  densityType='variable' only.  nesosim_set_forcing returns the context to a single shared season. */
int nesosim_set_forcing_sets(nesosim_ctx *ctx, int n_sets, const double *precip_dev, const double *conc_dev,
                             const double *wind_dev, const double *drift_dev, const int32_t *member_set_host,
                             const int32_t *set_days_host);

/* The season: IC handling of main (NESOSIM.py:604-609; ic_dev = [ny][nx] total depth shared by all members,
 * or [M][ny][nx] when ic_per_member != 0, or NULL for zero depth) when first_step == 0, then steps
 * x = first_step .. first_step+num_steps-1 of `for x in range(numDays-1): calcBudget(...)`
 * (NESOSIM.py:614-639) for every member.  Slot 0 of every non-NULL output is (re)written when
 * first_step == 0 (zeros; IC halves for snowDepths) so callers need not zero-fill.  num_steps < 0 means
 * "to the end" (T-1-first_step).  Asynchronous on `stream`, except that the season-resident path (see
 * nesosim_set_path) synchronises the stream once at the end to read its operand-range flag: that kernel only
 * carries the proven-exact fast divisions, and a season in which some operand left their range (denormal or
 * > 2^624 magnitudes; never on physical data) is transparently redone by the general per-day kernels. */
int nesosim_run_season(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                       int ic_per_member, const nesosim_outputs *out, int first_step, int num_steps,
                       void *stream);

/* One calcBudget call (NESOSIM.py:224-347) with that day's forcing planes given explicitly: advances slot x
 * to slot x+1 of `out` in place for every member.  rho_new is used only when density_clim=1. */
int nesosim_step_day(nesosim_ctx *ctx, int x, const double *conc_dev, const double *precip_dev,
                     const double *drift_dev, const double *wind_dev, double rho_new,
                     const nesosim_member_params *params_host, const nesosim_outputs *out, void *stream);

/* Same as nesosim_run_season but every data pointer is HOST memory (pinned or pageable): copies the forcing
 * to the device, runs the season, copies every non-NULL output back, synchronises.  This is the call
 * bench.py times for the end-to-end figure.  `out_host` strides are in elements like nesosim_outputs.
 * Members are processed in batches so that device and pinned staging memory stay bounded; bytes moved are
 * reported through h2d_bytes / d2h_bytes when non-NULL.  snowAcc and snowOcean do not depend on the member (forcing
 * only, NESOSIM.py:263-270): with one shared forcing a single copy crosses the link and host threads replicate it into
 * every member's slot of the caller's arrays.  When the process has at least 6 host threads to itself
 * (NESOSIM_HOST_THREADS; default: cores / visible GPUs) and at most 60 % of the grid is ocean, the other nine arrays are
 * drained in packed form -- ocean cells, plus the land cells of the first three time slots -- and scattered into the
 * caller's arrays by those threads (NESOSIM_HOST_COMPACT=0/1 overrides); the arrays are the same either way
 * (nesosim_host_drain_info). */
int nesosim_run_season_host(nesosim_ctx *ctx, const double *precip, const double *conc, const double *wind,
                            const double *drift, const double *rho_clim,
                            const nesosim_member_params *params, const double *ic, int ic_per_member,
                            const nesosim_outputs *out_host, int64_t *h2d_bytes, int64_t *d2h_bytes);

/* smooth_snow (NESOSIM.py:170-187) = astropy convolve(arr, 3x3 kernel) with defaults, both branches
 * (plain, and NaN-interpolating when the input sum is NaN).  in/out are distinct [ny][nx] device planes. */
int nesosim_smooth(const double *in_dev, double *out_dev, int ny, int nx, const double weights_host[9],
                   double divisor, void *stream);

/* Per-function entry points (device planes), one per reference function, for known-answer tests. */
/* calcDynamics (NESOSIM.py:189-222): drift [2][ny][nx], depths [2][ny][nx] -> adv [2][ny][nx], div [2][ny][nx] */
int nesosim_op_dynamics(const double *drift_dev, const double *depths_dev, double dx, double deltaT,
                        int ny, int nx, double *adv_dev, double *div_dev, void *stream);
/* calcLeadLoss / calcAtmLoss / calcWindPacking (NESOSIM.py:51-125): five output planes, any may be NULL */
int nesosim_op_wind_terms(const double *h0_dev, const double *wind_dev, const double *conc_dev, int64_t n,
                          const nesosim_member_params *p_host, double deltaT, double rhoFresh, double rhoOld,
                          double *lead_dev, double *atm_dev, double *wp_loss_dev, double *wp_gain_dev,
                          double *wp_net_dev, void *stream);
/* fillMaskAndNaNWithZero (NESOSIM.py:127-139), in place */
int nesosim_op_fill_zero(double *arr_dev, int64_t n, void *stream);
/* fill_nan_no_negative (NESOSIM.py:141-166), in place; mask_dev is uint8 [n] on the device */
int nesosim_op_fill_nan_no_negative(double *arr_dev, const uint8_t *mask_dev, int64_t n,
                                    int negative_to_zero, void *stream);
/* densityCalc (NESOSIM.py:458-473): depths [2][n] -> density [n] */
int nesosim_op_density(const double *depths_dev, const uint8_t *mask_dev, int64_t n, double rhoFresh,
                       double rhoOld, double minSnowD, double *density_dev, void *stream);

/* Final-product diagnostics: the array preparation of OutputSnowModelFinal (utils.py:161-179) on what main hands it
 * (NESOSIM.py:654: snowVol = h0+h1, snowDepth = snowVol/iceConc), fused into one pass and written as the float32
 * fields the NetCDF file stores: every field np.around(x, 4) (= rint(x*1e4)/1e4 in fp64) then cast to float32;
 * snow_volume, snow_depth and snow_density are NaN where iceConc < ice_conc_mask (skipped when ice_conc_mask <= 0),
 * ice_concentration is then NaN where iceConc < 0.15.  Inputs are device arrays of one member: depths [T][2][plane],
 * everything else [T][plane]; any output may be NULL.  96 B -> 24 B per cell-day on the way to the host.
 * For an ensemble pass the members' stacked arrays as num_days = M*T and forcing_days = T: depths/density (and the
 * outputs) then hold M*T days while conc/precip/wind hold T days that every member shares (0 = same as num_days). */
int nesosim_final_products(const double *depths_dev, const double *density_dev, const double *conc_dev,
                           const double *precip_dev, const double *wind_dev, int num_days, int forcing_days, int64_t plane,
                           double ice_conc_mask, float *snow_depth_dev, float *snow_volume_dev,
                           float *snow_density_dev, float *ice_conc_dev, float *precip_out_dev, float *wind_out_dev,
                           void *stream);

/* Calibration driver (SURVEY.md 8f N3; the reference has no counterpart): the season of nesosim_run_season with the
 * observation sampling FUSED into the season-resident kernel -- no output array is written at all.
 * nesosim_set_observations registers point observations (day slot 0..T-1, row, col, observed snow depth over ice [m];
 * host arrays, copied): they are compiled against the kernel's cell ownership once (distinct (cell, day) pairs =
 * "sample slots", sorted per owning thread) and stay on the device until replaced.  During nesosim_run_season_misfit the
 * thread that owns an observed cell stores the two layers h0, h1 of the observed days -- 16 bytes per observed cell-day
 * instead of 96 per cell-day, nothing on the day's critical path waits for it -- and a one-CTA-per-member epilogue forms
 * model = (h0+h1)/iceConc at that slot and cell (what main writes as snow depth, NESOSIM.py:654) and
 * misfit_dev[m] = sum over the observations of (model - observed)^2, skipping non-finite differences (land, NaN forcing,
 * zero concentration); count_dev[m] (may be NULL) = the number of observations used.  Sums are formed in a fixed order
 * (bit-reproducible).  Needs the season-resident path (grid up to 96 columns, variable density, one shared forcing --
 * or forcing sets with observations from nesosim_set_observations_sets, below); NESOSIM_ERR_ARG otherwise -- unless
 * the observations are registered after nesosim_set_path(ctx, 1): then the general day kernel produces the same
 * samples on any grid (see nesosim_set_path). */
int nesosim_set_observations(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_day_host, const int32_t *obs_row_host,
                             const int32_t *obs_col_host, const double *obs_depth_host);
int nesosim_run_season_misfit(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                              int ic_per_member, double *misfit_dev, int64_t *count_dev, void *stream);

/* Multi-season calibration: observations tagged with the forcing set (season) they belong to; needs
 * nesosim_set_forcing_sets first (NESOSIM_ERR_STATE otherwise).  obs_day must be < set_days[obs_set]; land/lake
 * observations are skipped as in nesosim_set_observations; a set index outside [0, n_sets), a day outside its set's
 * season or a cell outside the grid is NESOSIM_ERR_ARG.  Each set is compiled exactly as nesosim_set_observations
 * compiles its season, and the next nesosim_run_season_misfit runs every member through its season in one batch and scores
 * member m against the observations of set member_set[m] only: misfit_dev[m] and count_dev[m] equal, bit for bit, what
 * that member's season gives on a single-forcing context with the same strips (NESOSIM_ENS_CLUSTER).  The observations
 * remember the (n_sets, set_days) they were compiled against: once the forcing is registered again with another layout,
 * or with nesosim_set_forcing, nesosim_run_season_misfit returns NESOSIM_ERR_STATE until observations are registered
 * again.  Plain observations on a context with forcing sets stay NESOSIM_ERR_ARG at run time. */
int nesosim_set_observations_sets(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_set_host,
                                  const int32_t *obs_day_host, const int32_t *obs_row_host,
                                  const int32_t *obs_col_host, const double *obs_depth_host);

/* Calibration scores: observation errors, several observed quantities and the model value at every observation.
 * nesosim_set_observations_ex registers observations of any kind with an error sigma each (obs_set NULL: one shared
 * forcing, as nesosim_set_observations; else tagged with their forcing set, as nesosim_set_observations_sets; obs_kind
 * NULL: all depth; obs_sigma NULL: all 1) and replaces the registered ones.  Every kind is a function of the two snow
 * layers (h0, h1) of the observed day, which the season kernel stores per observed (cell, day): observations of several
 * kinds at one cell and day share that sample.  nesosim_run_season_scores runs the season as nesosim_run_season_misfit and
 * writes, per member m and kind k, chi2_dev[m][k] = sum over the member's observations of that kind of
 * ((model - observed)/sigma)^2 and count_dev[m][k] (may be NULL) = the number of terms; a term is used only if it is
 * finite (land, NaN forcing, zero concentration, density below minSnowD and NaN observed values are skipped).  Each kind
 * is summed in a fixed order, exactly as if it had been registered alone: with sigma 1, chi2_dev[m][NESOSIM_OBS_DEPTH]
 * of depth observations is bit-identical to nesosim_run_season_misfit's misfit.  model_dev (may be NULL) receives the
 * fp64 model value of every observation at its index among its set's input observations (its input index with one
 * forcing): model_dev[m*model_stride + i]; observations on land or lake hold NaN.  A density observation on day 0 has no
 * model counterpart (the reference never computes density[0], NESOSIM.py:350-376) and is rejected.
 * NESOSIM_ERR_ARG: a kind outside [0, NESOSIM_OBS_KINDS), a density observation on day 0, a sigma that is not finite and
 * > 0, model_stride < the row length, and whatever nesosim_set_observations / _sets reject; a rejected registration
 * leaves the previous observations in force.  NESOSIM_ERR_STATE as for nesosim_run_season_misfit; and
 * nesosim_run_season_misfit itself returns it when the registered observations hold a kind other than depth or a
 * sigma other than 1, which its one number per member cannot report. */
#define NESOSIM_OBS_DEPTH   0   /* snow depth over ice (h0+h1)/iceConc [m] (NESOSIM.py:654)        */
#define NESOSIM_OBS_VOLUME  1   /* snow volume per grid-cell area h0+h1 [m]                         */
#define NESOSIM_OBS_DENSITY 2   /* bulk snow density, densityCalc (NESOSIM.py:458-473) [kg m^-3]    */
#define NESOSIM_OBS_KINDS   3

int nesosim_set_observations_ex(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_set_host,
                                const int32_t *obs_day_host, const int32_t *obs_row_host, const int32_t *obs_col_host,
                                const int32_t *obs_kind_host, const double *obs_value_host, const double *obs_sigma_host);
/* length of a member's model row: the largest number of input observations of one set (n_obs with one forcing) */
int nesosim_observation_row_length(const nesosim_ctx *ctx, int64_t *row_len);
/* chi2_dev [M][NESOSIM_OBS_KINDS]; count_dev same shape or NULL; model_dev [M][model_stride] or NULL */
int nesosim_run_season_scores(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                              int ic_per_member, double *chi2_dev, int64_t *count_dev,
                              double *model_dev, int64_t model_stride, void *stream);

/* Footprint observations: means over many cells and/or days (drifting-station climatologies, monthly gridded products,
 * basin means).  A footprint belongs to one forcing set (fp_set NULL: one shared forcing), has a kind (fp_kind NULL: all
 * depth), an observed value, a sigma (fp_sigma NULL: all 1) and the points [fp_begin[g], fp_begin[g+1]) of the
 * pt_* arrays, each (day, row, col, weight) (pt_weight NULL: all 1).  nesosim_set_observations_fp registers point
 * observations (exactly as nesosim_set_observations_ex) and footprints together and replaces what was registered.
 * Footprint points on land or lake cells are dropped, as point observations are.  The points share the sample slots of
 * the observed (cell, day) pairs with the point observations but never enter the point tables: the point results are
 * bit-identical with and without footprints.
 * nesosim_run_season_scores_fp writes the point outputs of nesosim_run_season_scores, and per member m: the model value
 * of footprint g, fp_model_dev[m*fp_model_stride + g] (g = its index among its set's input footprints; padding past
 * the set's count up to the row length is NaN), and per kind fp_chi2_dev[m][k] = the sum of the finite
 * ((model - value)/sigma)^2 over the set's footprints of kind k, fp_count_dev[m][k] their number (may be NULL).
 * The model value of a footprint is the weighted mean of its points' model values (the operators of the point
 * observations), over the points whose value is finite, in a fixed order: the footprint's j-th kept point (input order)
 * goes to lane j % 32 of one warp, which adds w*v and w in order from 0.0; lane 0 collects both with the shuffle-down
 * tree 16, 8, 4, 2, 1; the mean is their quotient, NaN when no point was finite.  The footprint terms are summed as the
 * point terms (one kind's range, in input order within the set, thread i % 256 of one block).  Five launches: the
 * pre-pass (2), the season kernel, the footprint means, the epilogue.  While footprints are registered,
 * nesosim_run_season_misfit and nesosim_run_season_scores return NESOSIM_ERR_STATE (they would drop them).
 * NESOSIM_ERR_ARG: whatever nesosim_set_observations_ex rejects; fp_begin not starting at 0 or not increasing (an
 * empty footprint); a weight that is not finite and > 0; a kind, sigma or set tag as for point observations; a point
 * outside the grid or outside its set's season; a density point on day 0; a set's slots or points that do not fit
 * int indices; fp_model_stride < the footprint row length.  A rejected registration leaves the previous one in force;
 * the stale-layout rule of nesosim_set_observations_sets applies unchanged. */
int nesosim_set_observations_fp(nesosim_ctx *ctx, int64_t n_obs, const int32_t *obs_set_host,
                                const int32_t *obs_day_host, const int32_t *obs_row_host, const int32_t *obs_col_host,
                                const int32_t *obs_kind_host, const double *obs_value_host, const double *obs_sigma_host,
                                int64_t n_fp, const int32_t *fp_set_host, const int32_t *fp_kind_host,
                                const double *fp_value_host, const double *fp_sigma_host, const int64_t *fp_begin_host,
                                const int32_t *pt_day_host, const int32_t *pt_row_host, const int32_t *pt_col_host,
                                const double *pt_weight_host);
/* length of a member's footprint model row: the largest number of input footprints of one set (0: none) */
int nesosim_footprint_row_length(const nesosim_ctx *ctx, int64_t *row_len);
/* fp_chi2_dev [M][NESOSIM_OBS_KINDS]; fp_count_dev same shape or NULL; fp_model_dev [M][fp_model_stride] or NULL */
int nesosim_run_season_scores_fp(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                                 int ic_per_member, double *chi2_dev, int64_t *count_dev, double *model_dev,
                                 int64_t model_stride, double *fp_chi2_dev, int64_t *fp_count_dev,
                                 double *fp_model_dev, int64_t fp_model_stride, void *stream);

/* Asynchronous mode.  By default nesosim_run_season on the season-resident path synchronises `stream` once to read
 * the kernel's operand-range flag (see above).  With nesosim_set_async(ctx, 1) it never synchronises: the flag is copied
 * to pinned host memory behind the kernel and examined by nesosim_sync (which waits for every season enqueued so far on
 * this context, redoes with the general kernels any season whose flag is raised -- never on physical data -- and
 * reports how many) or, without waiting, by later calls.  Contract in this mode: a season's outputs, its IC buffer and
 * the forcing are final / reusable only after nesosim_sync; back-to-back seasons, the next forcing's upload and the
 * previous outputs' download then overlap freely on the caller's streams.  nesosim_set_async(ctx, 0) syncs first. */
int nesosim_set_async(nesosim_ctx *ctx, int on);
int nesosim_sync(nesosim_ctx *ctx, int *seasons_redone);

/* Kernel path of nesosim_run_season: 0 = automatic (default), 1 = general per-day kernel (any grid),
 * 2 = season-resident cluster kernel (grids up to 96x96, variable density, whole season; error otherwise).
 * Both paths produce identical values.  nesosim_last_path reports which one the last season used.
 * The path also chooses the producer of the calibration samples.  Observations registered (nesosim_set_observations,
 * _sets, _ex, _fp) under path 1 are compiled for the general path and scored (nesosim_run_season_misfit, _scores,
 * _scores_fp) on any grid by the scoring build of the day kernel: it advances only the two depth layers, in a two-slot
 * ring (32 bytes per member-cell; no accumulator or density is loaded or stored, nothing is written to caller arrays),
 * and copies the observed cells of each day into the samples; then the same epilogues run.  The scores, counts and
 * model rows are bit-identical to the season kernel's where it applies (the fixed order depends only on the (cell,
 * day) order of the observations).  The call takes T+2 launches (T+3 with footprints: init, T-1 day kernels, the
 * last-day samples, [footprint means,] epilogue) and never synchronises the stream (there is no operand-range flag).
 * Registration under path 1 also returns NESOSIM_ERR_ARG on a strip context (nesosim_strip_setup) and with
 * densityType='clim' (the density observation operator is densityCalc).  Under paths 0 and 2 registration needs the
 * season-resident kernel, as before.  Observations remember the path they were compiled for: after a change between
 * path 1 and paths 0/2 the scoring calls return NESOSIM_ERR_STATE until the observations are registered again. */
int nesosim_set_path(nesosim_ctx *ctx, int path);
int nesosim_last_path(const nesosim_ctx *ctx);

/* Calibration gradients (general path only): exact tangent-linear derivatives of the scores of
 * nesosim_run_season_scores(_fp) with respect to three parameters of every member.  The model is piecewise linear in
 * them for fixed forcing, so a tangent build of the scoring day kernel carries d(h0, h1)/dtheta through the season in the
 * same fixed orders as the primal (DESIGN.md §4.1): the pathwise derivative, with the kinks (clamps, NaN masks, the
 * density clamps) taken on the side the primal took.  windPackThresh enters only through the step W > thresh: its
 * derivative is 0 almost everywhere and undefined at the step, and it is not reported.
 * Outputs besides those of nesosim_run_season_scores_fp, which are bit-identical to that call's:
 *   grad_dev [M][NESOSIM_OBS_KINDS][NESOSIM_GRAD_DIRS]: per kind d chi2 / d theta_j = sum of 2 r (dv_j / sigma) over the
 *     terms chi2 counts, in chi2's order;
 *   jac_dev [M][NESOSIM_GRAD_DIRS][jac_stride] or NULL: dv_j at every input observation (NaN where v is not finite and
 *     for observations dropped at registration);
 *   fp_grad_dev, fp_jac_dev: the same for the footprints (d mean = sum w dv over the points with finite v / sum w).
 * Needs observations registered under path 1 (else NESOSIM_ERR_STATE); with footprints registered fp_chi2_dev and
 * fp_grad_dev are required (NESOSIM_ERR_STATE), without them the fp_* arguments are ignored.  NESOSIM_ERR_ARG: a NULL
 * grad_dev, a stride shorter than its row, more members or tile rows than a launch grid holds.  The tangent state
 * (96 bytes per member-cell) is allocated by the first call and freed with the observations.  T+2 launches (T+3 with
 * footprints), no stream synchronisation, as nesosim_run_season_scores_fp. */
#define NESOSIM_GRAD_DIRS 3   /* windPackFactor, leadLossFactor, atmLossFactor */
int nesosim_run_season_score_grads(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                                   int ic_per_member, double *chi2_dev, int64_t *count_dev, double *model_dev,
                                   int64_t model_stride, double *grad_dev, double *jac_dev, int64_t jac_stride,
                                   double *fp_chi2_dev, int64_t *fp_count_dev, double *fp_model_dev,
                                   int64_t fp_model_stride, double *fp_grad_dev, double *fp_jac_dev, int64_t fp_jac_stride,
                                   void *stream);

/* Calibration adjoint (general path only): reverse-mode derivatives of the objective
 *   J_m = sum_k weights_host[k] chi2[m][k] + sum_k fp_weights_host[k] fp_chi2[m][k]
 * of every member m with respect to its initial snow-depth field and to the three parameters of
 * nesosim_run_season_score_grads, by one backward sweep through the season (DESIGN.md §4.1): the same pathwise
 * derivative as the tangent build, with every kink on the side the primal took.  Outputs besides those of
 * nesosim_run_season_scores_fp, which are bit-identical to that call's:
 *   theta_grad_dev [M][NESOSIM_GRAD_DIRS]: dJ_m / d(windPackFactor, leadLossFactor, atmLossFactor);
 *   ic_grad_dev [M][ny][nx]: dJ_m / d ic, per member even when the IC is shared (sum over members for the total);
 *     exactly 0 where conc[0] < minConc (the IC is zeroed there), and possibly non-zero on land, whose finite IC the
 *     first day's dynamics read.
 * The weights are host arrays [NESOSIM_OBS_KINDS] and must be finite and >= 0 (NESOSIM_ERR_ARG).  Needs observations
 * registered under path 1 (else NESOSIM_ERR_STATE); with footprints registered fp_chi2_dev is required
 * (NESOSIM_ERR_STATE).  NESOSIM_ERR_ARG also for a NULL theta_grad_dev or ic_grad_dev, a stride shorter than its row and
 * more members or tile rows than a launch grid holds.  The adjoint state, allocated by the first call and freed with the
 * observations, is 17 T + 56 bytes per member-cell (the depth trajectory, one record byte per day, a two-slot ring of
 * the adjoint depths and the three parameter accumulators) plus 16 bytes per member and sample slot; when it does not
 * fit the call frees what it allocated, returns NESOSIM_ERR_NOMEM and the context stays usable.  The first call also
 * uploads the per-slot seed tables with synchronous copies (and cudaMalloc may synchronise the device); later calls
 * issue 2T+4 kernel launches (2T+5 with footprints; one fewer on a grid without ocean, which has no sample slot), one
 * memset (two with model_dev) and no stream synchronisation. */
int nesosim_run_season_score_adjoint(nesosim_ctx *ctx, const nesosim_member_params *params_host, const double *ic_dev,
                                     int ic_per_member, const double *weights_host, const double *fp_weights_host,
                                     double *chi2_dev, int64_t *count_dev, double *model_dev, int64_t model_stride,
                                     double *fp_chi2_dev, int64_t *fp_count_dev, double *fp_model_dev,
                                     int64_t fp_model_stride, double *theta_grad_dev, double *ic_grad_dev, void *stream);

/* Calibration adjoint with the forcing: nesosim_run_season_score_adjoint plus the derivatives of the same J_m with
 * respect to the snowfall, wind-speed and ice-concentration forcing f = 0 precip, 1 wind, 2 conc (DESIGN.md §4.1).  They
 * enter the day step point-wise, so the backward day kernel forms them per cell next to the parameter terms, pathwise as
 * the rest (the wind threshold and the IC zeroing where conc[0] < minConc are steps, not differentiated):
 *   forcing_scale_grad_dev [M][NESOSIM_FORCING_DIRS][ny][nx], required: sum over the member's days x (descending) of
 *     F(x) g_F(x) where F(x) is finite, from 0.0 -- dJ_m / d alpha for a per-cell factor F -> alpha F over the season;
 *   forcing_scale_total_dev [M][NESOSIM_FORCING_DIRS], required: each field summed over the cells in theta_grad's fixed
 *     order ([m][0]: the derivative with respect to one snowfall scaling factor);
 *   precip_day_dev, wind_day_dev, conc_day_dev [M][T][ny][nx], each NULL or written in full: g_F(x) = dJ_m / d F(x) of
 *     every day (0 after the member's last day, and for precip and wind on it); conc includes the depth observation
 *     operator's (h0 + h1) / C.
 * Chi2, counts, model rows, theta_grad and ic_grad are bit-identical to nesosim_run_season_score_adjoint's.  Errors as
 * that call's, and NESOSIM_ERR_ARG for a NULL forcing_scale_grad_dev or forcing_scale_total_dev.  The state is that of
 * nesosim_run_season_score_adjoint plus 24 bytes per member-cell (the three scale accumulators) and 8 bytes per member
 * and sample slot (the concentration seeds): 17 T + 80 bytes per member-cell and 24 per member-slot, allocated by the
 * first forcing call and freed with the observations (NESOSIM_ERR_NOMEM as there).  The same 2T+4 launches (2T+5 with
 * footprints), one memset more and no stream synchronisation after the first call. */
#define NESOSIM_FORCING_DIRS 3   /* precip, wind, conc */
int nesosim_run_season_score_adjoint_forcing(nesosim_ctx *ctx, const nesosim_member_params *params_host,
                                             const double *ic_dev, int ic_per_member, const double *weights_host,
                                             const double *fp_weights_host, double *chi2_dev, int64_t *count_dev,
                                             double *model_dev, int64_t model_stride, double *fp_chi2_dev,
                                             int64_t *fp_count_dev, double *fp_model_dev, int64_t fp_model_stride,
                                             double *theta_grad_dev, double *ic_grad_dev,
                                             double *forcing_scale_grad_dev, double *forcing_scale_total_dev,
                                             double *precip_day_dev, double *wind_day_dev, double *conc_day_dev,
                                             void *stream);

/* Calibration adjoint with the ice drift: nesosim_run_season_score_adjoint (and, optionally,
 * nesosim_run_season_score_adjoint_forcing) plus the derivatives of the same J_m with respect to the drift components
 * d = 0 u, 1 v (DESIGN.md §4.1).  The raw dynamics terms adv_l = -(ut gx(h_l) + vt gy(h_l)) and
 * div_l = -(h_l gx(ut) + h_l gy(vt)) (ut = u dT, vt = v dT, h_l the depth of day x, np.gradient's stencils) are
 * bilinear in depth and drift, so per day x below the member's last slot L, with nu_l the transposed 3x3 smoothing of
 * m_l = (kill_l ? 0 : lambda_l(x+1)) / divisor and A_l, D_l whether adv_l, div_l were finite:
 *   g_u(c) = -dT (sum_l [A_l(c)] nu_l(c) gx(h_l)(c) + Qx(c-1) - Qx(c+1) + E_x(c)),
 *   Qx(r) = sum_l [D_l(r)] nu_l(r) h_l(r) / d_x(r), d_x = dx on that axis's grid edge, else 2 dx,
 *   E_x = (last ? Qx(c) : 0) - (first ? Qx(c) : 0);  g_v alike along y;  g = 0 on days L..T-1 and without dynamics.
 * A land cell next to the ocean gets the Q of its neighbour through the drift gradient of the neighbour's div term.
 *   drift_scale_grad_dev [M][NESOSIM_DRIFT_DIRS][ny][nx], required: sum over the member's days x (descending) of
 *     F(x) g_F(x) where F(x) is finite, from 0.0 -- dJ_m / d alpha for a per-cell factor F -> alpha F over the season;
 *   drift_scale_total_dev [M][NESOSIM_DRIFT_DIRS], required: each field summed over the cells in theta_grad's fixed
 *     order; [m][0] + [m][1] is the derivative with respect to one drift speed factor (u, v) -> alpha (u, v);
 *   drift_day_dev [M][T][NESOSIM_DRIFT_DIRS][ny][nx] (the staged drift's layout), NULL or written in full: g_u, g_v of
 *     every day.
 * The forcing outputs are those of nesosim_run_season_score_adjoint_forcing, optional as a pair: with both
 * forcing_scale_grad_dev and forcing_scale_total_dev NULL no forcing term is formed (and precip_day_dev, wind_day_dev,
 * conc_day_dev must be NULL).  Chi2, counts, model rows, theta_grad and ic_grad are bit-identical to
 * nesosim_run_season_score_adjoint's, and the forcing outputs to nesosim_run_season_score_adjoint_forcing's.  Errors as
 * those calls', and NESOSIM_ERR_ARG for a NULL drift_scale_grad_dev or drift_scale_total_dev, for one of the forcing
 * pair without the other, or for a per-day forcing buffer without the pair.  The state is that of the call without the
 * drift plus 16 bytes per member-cell (the two drift scale accumulators), allocated by the first drift call and freed
 * with the observations (NESOSIM_ERR_NOMEM as there).  The same 2T+4 launches (2T+5 with footprints), one memset more
 * and no stream synchronisation after the first call. */
#define NESOSIM_DRIFT_DIRS 2   /* u, v */
int nesosim_run_season_score_adjoint_drift(nesosim_ctx *ctx, const nesosim_member_params *params_host,
                                           const double *ic_dev, int ic_per_member, const double *weights_host,
                                           const double *fp_weights_host, double *chi2_dev, int64_t *count_dev,
                                           double *model_dev, int64_t model_stride, double *fp_chi2_dev,
                                           int64_t *fp_count_dev, double *fp_model_dev, int64_t fp_model_stride,
                                           double *theta_grad_dev, double *ic_grad_dev,
                                           double *forcing_scale_grad_dev, double *forcing_scale_total_dev,
                                           double *precip_day_dev, double *wind_day_dev, double *conc_day_dev,
                                           double *drift_scale_grad_dev, double *drift_scale_total_dev,
                                           double *drift_day_dev, void *stream);

/* ---- Row-strip domain decomposition over peer memory (grids too large for one GPU: the 5 km case; the reference
 * has no counterpart -- its grid is one numpy array -- so the contract is that of calcBudget on the whole grid).
 * A context created on rows [lo-2, hi+2) of the full grid (mask and forcing sliced the same way; 2 = radius of
 * np.gradient followed by the 3x3 convolution, NESOSIM.py:204-213,184-185; no ghost rows at the global edges) is one
 * STRIP.  After nesosim_strip_setup + nesosim_strip_connect*, nesosim_run_season on the general path advances the
 * strip with ONE launch per day and nothing in between: the day kernel itself stores the new depths of its first /
 * last two owned rows into the neighbouring strip's mailbox (peer memory over NVLink when the neighbour is another
 * GPU) and raises that strip's flag; the next day's boundary CTAs wait for their own flag and take the ghost rows
 * from the mailbox.  The owned rows of every output come out identical to a single-context run of the whole grid;
 * the ghost rows of the outputs are scratch.  n_members must be 1.  All strips must run the same sequence of
 * nesosim_run_season calls (whole seasons, or the same first_step/num_steps pieces), and every strip's previous
 * season must have completed on its stream before any strip starts the next one (one barrier between seasons).
 * A neighbour that never delivers does not hang the GPU: waits give up after a time-out (default 5 s) and
 * nesosim_strip_status reports it. */
#define NESOSIM_IPC_HANDLE_BYTES 64
int nesosim_strip_setup(nesosim_ctx *ctx, int has_up_neighbour, int has_down_neighbour);
/* the strip's exchange block: as a cudaIpcMemHandle_t (64 bytes, for a neighbour in another process) ... */
int nesosim_strip_export(nesosim_ctx *ctx, void *handle64);
/* ... or as a device pointer (for a neighbour in the same process; other device: peer access must be enabled) */
int nesosim_strip_block(nesosim_ctx *ctx, void **block_dev, int64_t *bytes);
/* attach the neighbours' blocks (NULL where there is no neighbour) */
int nesosim_strip_connect(nesosim_ctx *ctx, const void *up_handle64, const void *down_handle64);
int nesosim_strip_connect_local(nesosim_ctx *ctx, void *up_block_dev, void *down_block_dev);
/* *timed_out = 1 if any wait for a neighbour gave up since nesosim_strip_setup (synchronous device read) */
int nesosim_strip_status(nesosim_ctx *ctx, int *timed_out);
int nesosim_strip_set_timeout(nesosim_ctx *ctx, double seconds);

/* Diagnostics for the exact constant-division path used for /dx, /(2.*dx), /rho and /kernel.sum()
 * (cell_math.cuh div_const): whether the 3-operation path was proven exact for divisor c, and a host
 * replica of the device routine (same branches, std::fma) so CPU tests can compare it with x / c. */
int    nesosim_const_div_is_fast(double c);
double nesosim_const_div_eval_host(double x, double c);

/* Seasons the season-resident path had to hand back to the general kernels (see nesosim_run_season). */
int64_t nesosim_rerun_count(const nesosim_ctx *ctx);

/* How the last nesosim_run_season_host drained its results: *compacted = 1 if only the ocean cells (and the land cells
 * of the first three time slots) of the member-dependent arrays crossed the link and host threads scattered them into
 * the caller's arrays; *full_chunks = (member, array) blocks (since creation) for which that was given up because their land
 * cells were not constant in time, and which were copied in full instead.  The caller's arrays are the same either way
 * (the reference's genEmptyArrays contract, NESOSIM.py:350-376). */
int nesosim_host_drain_info(const nesosim_ctx *ctx, int *compacted, int64_t *full_chunks);

/* The compacted drain shares the work between the host threads and the copy engine as it goes: whenever every slot of
 * the pinned ring is taken (the threads are the bottleneck), the link copies whole (member, array) blocks of the same
 * batch straight into the caller's arrays instead.  *packed / *plain = the blocks of the last call that went either
 * way (both 0 after a plain drain). */
int nesosim_host_drain_blocks(const nesosim_ctx *ctx, int64_t *packed, int64_t *plain);

/* Host half of that drain, on its own: one member's packed block of one array -- [planes_per_slot*num_days][n_ocean]
 * ocean values (cells with mask 1..10, ascending), then [planes_per_slot*min(3,num_days)][n_land] land values of the
 * first slots -- scattered into the full planes dst[planes_per_slot*num_days][plane]; later slots repeat the land cells
 * of the third.  No device involved. */
int nesosim_unpack_member_array(const uint8_t *mask, int64_t plane, int planes_per_slot, int num_days,
                                const double *packed, double *dst);

/* Device time of the season-resident kernel's launches so far (CUDA events on the launching stream) and their
 * number: what bench.py divides the algorithmic bytes per launch by for its roofline figure. */
int nesosim_season_kernel_time(const nesosim_ctx *ctx, double *total_ms, int64_t *launches);

/* Number of kernel launches this context has issued since creation (bench.py reports it). */
int64_t nesosim_launch_count(const nesosim_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* NESOSIM_B200_H */
