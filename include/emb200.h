/* emb200.h -- C ABI of libemb200.so, the B200-native sampler for the hot path of
 * Airspace-Encounter-Models/em-model-manned-bayes.
 *
 * The reference is pure MATLAB and has no FFI boundary of its own (SURVEY.md section 8b); the
 * boundary therefore sits at the MATLAB signatures that take a *batch* argument.  Each entry point
 * below names the reference interface it replaces (paths relative to /root/reference/).  A MATLAB
 * user reaches these through the MEX gateway in matlab/emb_mex.cpp; the tests and the Python
 * mirror (em_model_manned_bayes_b200/) reach them through ctypes.  INTEGRATION.md shows both.
 *
 * Conventions
 *  - plain C types only; every function returns 0 on success or a negative EMB_E_* code, and
 *    emb_last_error() returns a thread-local message whose text starts with the reference's error
 *    identifier/message where one exists (e.g. "Unknown field: ...", em_read.m:105).
 *  - bins are 1-based (MATLAB values); variable ids in arrays are 1-based too.
 *  - sample indices are 0-based *global* indices; the random stream is keyed by them, so any shard
 *    [first, first+n) of a job gives the same numbers on any GPU count (SURVEY.md 8e).
 *  - the caller owns every output buffer; `mem` says whether buffers are host or device pointers.
 *    Host buffers should be pinned (emb_host_alloc) for full PCIe speed.
 *  - there is NO CPU fallback: sampling entry points fail with EMB_E_CUDA if no sm_100 device or
 *    kernel image is available.
 */
#ifndef EMB200_H
#define EMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EMB_ABI_VERSION 2

/* status codes */
#define EMB_OK 0
#define EMB_E_IO (-1)        /* cannot open/read file */
#define EMB_E_PARSE (-2)     /* malformed model file ("Unknown field: %s", em_read.m:105) */
#define EMB_E_MODEL (-3)     /* inconsistent model ("Network could not be hierarchically sorted", bn_sort.m:23) */
#define EMB_E_ARG (-4)       /* bad argument ("Attempt to preset a dependent variable", bn_sample.m:47; "dynvar:empty", UncorEncounterModel.m:231) */
#define EMB_E_CUDA (-5)      /* CUDA error / no device */
#define EMB_E_LIMIT (-6)     /* model exceeds a compiled limit (EMB_MAX_*) */
#define EMB_E_REJECT (-7)    /* a sample exhausted the rejection budget */

#define EMB_MAX_VARS 24      /* initial-network variables */
#define EMB_MAX_DYN 8        /* dynamic variables */
#define EMB_MAX_PARENTS 8
#define EMB_MAX_GATED 16

/* memory kind of caller buffers */
#define EMB_MEM_HOST 0
#define EMB_MEM_DEVICE 1
/* or-ed with EMB_MEM_DEVICE, emb_sample_tracks / emb_sample_initial only: enqueue the pass on opts.stream and return without waiting for it, so
 * consecutive passes run back to back; emb_async_status(device) later synchronises and reports an exhausted rejection loop */
#define EMB_MEM_ASYNC 0x100

/* prior kinds: bn_dirichlet_prior.m:17-38 and setTransitionPriors.m:12-33 */
#define EMB_PRIOR_CONSTANT 0 /* alpha = value everywhere (EncounterModel.m:45 default 0) */
#define EMB_PRIOR_DBE 1      /* alpha = 1/(r*q) */
#define EMB_PRIOR_STAY 2     /* transition only: alpha = value where child bin == own previous bin */

typedef struct emb_model emb_model; /* opaque; immutable after load except emb_set_prior */

/* ---- model reader: replaces em_read.m:1-141 + bn_sort.m:14-24 + the packing the kernels need --- */
int emb_model_load(const char* parameters_filename, int is_overwrite_zero_boundaries,
                   const int32_t* idx_zero_boundaries, int32_t n_idx, emb_model** out);
/* Build a model from arrays (bn_sample.m:1 functional form and synthetic models).  G is row-major
 * n x n with G[parent*n + child]; N_* are the concatenated column-major count tables in variable
 * order (em_read.m:191-198); transition arguments may be NULL/0 for an initial-only network;
 * boundaries are concatenated, boundaries_len[i] entries each (0 = '*'). */
int emb_model_from_arrays(int32_t n_initial, const uint8_t* G_initial, const int32_t* r_initial,
                          const double* N_initial, int64_t len_N_initial,
                          int32_t n_transition, const uint8_t* G_transition, const int32_t* r_transition,
                          const double* N_transition, int64_t len_N_transition,
                          const int32_t* temporal_map /* k x 2, 1-based, row-major */, int32_t n_temporal,
                          const double* boundaries, const int32_t* boundaries_len,
                          const double* resample_rates, emb_model** out);
void emb_model_free(emb_model* m);

typedef struct emb_model_info {
    int32_t n_initial, n_transition, n_dyn, n_gated;
    int32_t is_dynvar_depend;   /* dbn_sample.m:55: 1 = "slow" branch, 0 = frozen-parent "fast" branch */
    int32_t n_timevarying;      /* variables whose continuous value can change over a track */
    int64_t len_N_initial, len_N_transition;
    int32_t r_initial[EMB_MAX_VARS];
    int32_t r_transition[EMB_MAX_VARS + EMB_MAX_DYN];
    int32_t order_initial[EMB_MAX_VARS];                       /* 1-based, bn_sort order */
    int32_t order_transition[EMB_MAX_VARS + EMB_MAX_DYN];
    int32_t temporal_map[EMB_MAX_DYN][2];                      /* 1-based [var(t), var(t+1|t-1)] */
    int32_t zero_bins[EMB_MAX_VARS];                           /* 0 = none (em_read.m:143-156) */
    int32_t boundaries_len[EMB_MAX_VARS];
    int32_t timevarying_vars[EMB_MAX_VARS];                    /* 1-based ids, ascending */
    double resample_rates[EMB_MAX_VARS];
    double bounds_initial[EMB_MAX_VARS][2];                    /* em_read.m:124-136 */
} emb_model_info;
int emb_model_get_info(const emb_model* m, emb_model_info* info);
/* copies; `which`: 0 initial, 1 transition.  Returns the needed length when buf is NULL. */
int64_t emb_model_get_labels(const emb_model* m, int which, char* buf, int64_t cap); /* '\n'-joined */
int64_t emb_model_get_G(const emb_model* m, int which, uint8_t* buf, int64_t cap);
int64_t emb_model_get_N(const emb_model* m, int which, double* buf, int64_t cap);
int64_t emb_model_get_boundaries(const emb_model* m, double* buf, int64_t cap);
/* packed word-space thresholds actually uploaded to the GPU (for tests): column-padded tables */
int64_t emb_model_get_packed(const emb_model* m, int which, uint32_t* buf, int64_t cap);

/* ---- priors: replaces EncounterModel.m:249-257 -> bn_dirichlet_prior.m, setTransitionPriors.m --- */
/* Repacks the model's threshold tables: must not run concurrently with a sampling call on the SAME model (distinct models,
 * and sampling calls among themselves, are independent). */
int emb_set_prior(emb_model* m, int which /*0 initial, 1 transition*/, int kind, double value);

/* ---- random stream --------------------------------------------------------------------------- */
typedef struct emb_rng {
    uint64_t seed;          /* replaces rng(seed,'twister') (UncorEncounterModel.m:213-216) */
    uint64_t first_sample;  /* global index of this call's sample 0 */
} emb_rng;
/* the keyed Philox4x32-10 word for tests / injection hooks (stream spec v1, DESIGN.md) */
uint32_t emb_rng_word(uint64_t seed, uint64_t sample, uint32_t attempt, uint32_t purpose,
                      uint32_t index, uint32_t sub, uint32_t lane);

/* ---- sampling options ------------------------------------------------------------------------ */
#define EMB_REJECT_NONE 0
#define EMB_REJECT_UNCOR 1 /* v*1.68781 > |dh|/60 (UncorEncounterModel.m:275) */
#define EMB_REJECT_BOX 2   /* lo <= value <= hi per variable (@CorTerminalModel/sample.m:45-70) */

typedef struct emb_sample_opts {
    int32_t start[EMB_MAX_VARS]; /* preset bins, 0 = free (bn_sample.m:45, `start` cell) */
    int32_t reject_mode;
    int32_t idx_v, idx_dh, idx_L;             /* 1-based variable ids for EMB_REJECT_UNCOR / layers */
    double box_lo[EMB_MAX_VARS], box_hi[EMB_MAX_VARS]; /* EMB_REJECT_BOX */
    int32_t is_quantize500;                   /* UncorEncounterModel.m:266-268 */
    int32_t n_layers;                         /* 0 = no layers; else rows of `layers` (UncorEncounterModel.m:259-263) */
    double layers[8][2];
    int32_t max_attempts;                     /* 0 -> 65535 */
    int32_t mem;                              /* EMB_MEM_HOST / EMB_MEM_DEVICE for all output buffers */
    int32_t device;                           /* CUDA device ordinal; -1 = current */
    void* stream;                             /* cudaStream_t or NULL */
    /* per-sample presets (the n_samples x n_initial `start` cell of @CorTerminalModel/InitStartTerminal.m:43-92, one row per
     * sample): int8 [n_initial][n], 1-based bins, 0 = free; NULL = use `start` for every sample.  Host or device memory
     * like the outputs (`mem`).  A preset variable with a free parent is refused like bn_sample.m:46-47 does (EMB_E_ARG). */
    const int8_t* start_per_sample;
    /* NOT the reference's behaviour (default 0): for a model without a dynamic -> dynamic edge dbn_sample.m:110-135 freezes
     * the parent configuration of every dynamic variable at t = 1 (SURVEY F6); 1 re-evaluates the parents every second, as
     * dbn_sample.m:66-79 does for the other models -- the Markov chain the transition tables were trained for. */
    int32_t correct_dbn;
} emb_sample_opts;
void emb_sample_opts_init(emb_sample_opts* o);

/* ---- initial network: replaces bn_sample.m:25-58 (batch over num_samples) followed by the
 *      initial half of dbn_hierarchical_sample.m:25-31 / @CorTerminalModel/sample.m:29-77 ------- */
/* bins   : int8  [n_initial][n]   (1-based bins)                 nullable
 * values : double[n_initial][n]   (dediscretised; bin for '*')   nullable
 * attempts: uint16[n]             (rejection attempts used)      nullable */
int emb_sample_initial(const emb_model* m, const emb_rng* rng, int64_t n, const emb_sample_opts* opts,
                       int8_t* bins, double* values, uint16_t* attempts);
/* the same with fp32 values [n_initial][n]: the compact contract (1 + 4 bytes per variable); within 1e-6 relative of the fp64
 * values (the de-discretisation uniform has 23 bits, its conversion is exact in fp32; emb_model.cpp: pack) */
int emb_sample_initial_f32(const emb_model* m, const emb_rng* rng, int64_t n, const emb_sample_opts* opts,
                           int8_t* bins, float* values, uint16_t* attempts);

/* ---- tracks: replaces UncorEncounterModel.m:244-307 loop around dbn_hierarchical_sample.m:9-37
 *      (dbn_sample.m both branches, resample_events.m, dediscretize.m, events2samples.m) ---------- */
typedef struct emb_track_out {
    /* dense, in tiles of 128 tracks x four seconds, all variables of a tile together, so that a warp stores
     * contiguous memory and a thread's stores sit at fixed offsets from one pointer:
     *     element (variable g, track s, second c) = [c/4][s/128][g][s%128][c%4]
     * column c (0-based) is the state during second c+1, i.e. out_samples{ii}(:, c+1) (events2samples.m:9-27);
     * padding seconds of the last group are 0, padding tracks of the last tile are never written.  Buffer
     * lengths (elements): emb_tracks_bins_len / emb_tracks_values_len */
    int8_t* bins;        /* [ceil(T/4)][ceil(n/128)][n_dyn][128][4]  1-based bins of the dynamic variables  nullable */
    float* values;       /* [ceil(T/4)][ceil(n/128)][n_timevarying][128][4] continuous values               nullable */
    /* per track */
    int8_t* init_bins;   /* [n_initial][n]                                                   nullable */
    double* init_values; /* [n_initial][n]  out_inits (after layers/quantize500)             nullable */
    uint16_t* attempts;  /* [n]                                                              nullable */
    /* verification histograms, accumulated (+=) on the device: counts[var][bin-1], stride 64 */
    unsigned long long* hist_initial;    /* [n_initial][64]                                  nullable */
    unsigned long long* hist_transition; /* [n_dyn][64] over all columns 2..T                nullable */
} emb_track_out;
int emb_sample_tracks(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T,
                      const emb_sample_opts* opts, const emb_track_out* out);
/* sizes (in elements) of the dense buffers for given n, T */
int64_t emb_tracks_bins_len(const emb_model* m, int64_t n, int32_t T);
int64_t emb_tracks_values_len(const emb_model* m, int64_t n, int32_t T);

/* ---- tracks as sparse event lists: the reference's own track representation, out_events{ii} of
 *      UncorEncounterModel.m:253-300 = dbn_hierarchical_sample.m:9-37 (dbn_sample.m:84-92/151-161 change
 *      rows, resample_events.m:17-36 re-emitted bins, closing row :15-19), already de-discretised ----- */
typedef struct emb_event {
    uint16_t dt;   /* seconds since the previous row (0 for further rows of the same second) */
    uint8_t var;   /* 1-based variable id, 0 in the closing row */
    uint8_t bin;   /* 1-based bin the value was drawn in (oracle extra), 0 in the closing row */
    float value;   /* de-discretised value (the bin itself for '*' variables) */
} emb_event;       /* 8 bytes; row k of track s is events[offsets[s] + k] */
/* Two device passes (count rows per track, prefix-sum, write).  offsets: int64 [n+1] (offsets[n] = total rows),
 * events: capacity rows.  *total_rows (host, nullable) always receives the number of rows; if it exceeds
 * `capacity` nothing is written to `events` and EMB_E_LIMIT is returned -- call again with a larger buffer
 * (the stream is keyed, the result is the same).  `init` (nullable) may carry init_bins / init_values /
 * attempts; its dense fields and histograms must be NULL.  Requires T <= 65535, <= 15 time-varying variables, <= 16 bins. */
int emb_sample_track_events(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                            int64_t capacity, emb_event* events, int64_t* offsets, const emb_track_out* init,
                            int64_t* total_rows);

/* The same lists as 5-byte packed rows -- what the device writes and what crosses PCIe (the 8-byte rows above are expanded
 * from these on the device):   row k of track s is (words[offsets[s] + k], dts[offsets[s] + k]) with
 *     word = frac | (bin - 1) << 23 | gord << 27 | (dt >> 8) << 30,    dts = dt & 255
 *   gord : 1-based ordinal of the variable in emb_model_get_gated (the time-varying variables), 0 in the closing row
 *   frac : 23 bits; the row's value is boundaries[bin] + (boundaries[bin+1] - boundaries[bin]) * (frac + 0.5) * 2^-23
 *          (dediscretize.m:39 with the uniform of stream spec v5), 0 in a zero bin, the bin itself for a '*' variable
 * Needs <= 7 time-varying variables with <= 16 bins and T <= 1023 (EMB_E_LIMIT otherwise); same two-pass protocol,
 * `capacity` in rows for both arrays. */
int emb_sample_track_events_packed(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                                   int64_t capacity, uint32_t* words, uint8_t* dts, int64_t* offsets,
                                   const emb_track_out* init, int64_t* total_rows);
/* 1-based ids of the time-varying ("gated") variables, ascending: resample rate > 0 or dynamic.  Returns their number. */
int64_t emb_model_get_gated(const emb_model* m, int32_t* buf, int64_t cap);

/* ---- every GPU of the box from ONE call (SURVEY 8e): one host thread per device, tracks sharded by global sample index (device
 *      d owns emb_shard_range(n, d, n_devices); the stream is keyed by the global index, so the union over the devices equals the
 *      single-device result), no traffic between the devices on the data path, and ONE collective at the end: the verification
 *      histograms are summed over the devices with ncclAllReduce (NCCL is bound at run time; the few KB go through the host when
 *      it is not there).  outs[d] describes the buffers of device d's shard (host memory, or device memory ON device d when
 *      opts->mem is EMB_MEM_DEVICE), sized for that shard (emb_tracks_bins_len(m, count_d, T), ...); their histogram fields are
 *      ignored: hist_initial [n_initial][64] / hist_transition [n_dyn][64] (host, nullable, accumulated +=) receive the global
 *      counts.  n_devices = 0: all visible devices.  opts->device, opts->stream and opts->start_per_sample are ignored. */
void emb_shard_range(int64_t n, int32_t shard, int32_t n_shards, int64_t* first, int64_t* count);
int emb_sample_tracks_multi(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                            int32_t n_devices, const emb_track_out* outs, unsigned long long* hist_initial,
                            unsigned long long* hist_transition);
/* counts[d]: `len` uint64 counters in device memory of devices[d] (NULL: device d); on return every buffer holds the sum */
int emb_allreduce_histograms(int32_t n_devices, const int32_t* devices, unsigned long long* const* counts, int64_t len);
int emb_nccl_available(void);              /* 1 when libnccl could be bound */
const char* emb_multi_last_error(void);    /* message of the first failing device of the last emb_sample_tracks_multi */

/* ---- terminal trajectory chains: replaces @CorTerminalModel/createEncounter.m:1-329 over a batch of encounters
 *      (PropagateTrajectory :93-265 = per state one dbn_sample.m:95-166 call with t_max = 2 and every initial
 *      variable preset by CreateStartDistribution :268-294, the dynamic-limit resample loop :192-243, the kinematic
 *      update :171-184/:246-256, CheckTrajectoryConditions :296-329) including the forward/backward concatenation
 *      and time sort of :74-84.  The em-core `local_smooth` of :88-89 is not part of this library. ------------------ */
typedef struct emb_dyn_limits {   /* @CorTerminalModel/getDynamicLimits.m:14-62 */
    double minVel_ft_s, maxVel_ft_s, maxTurnRate_deg_s, maxAltitude_ft, maxVertRate_ft_s;
} emb_dyn_limits;
/* "GENERIC", "RTCA228_A1", "RTCA228_A2", "RTCA228_A3", "TEST" (case-insensitive); EMB_E_ARG otherwise */
int emb_dyn_limits_named(const char* ac_type, emb_dyn_limits* out);

typedef struct emb_terminal_models {   /* @CorTerminalModel/CorTerminalModel.m:12-30; index = intent - 1 */
    const emb_model* own_fwd[2];       /* mdlFwd1_1 (landing), mdlFwd1_2 (takeoff) */
    const emb_model* own_bck[2];       /* mdlBck1_1, mdlBck1_2 */
    const emb_model* int_fwd[3];       /* mdlFwd2_1 (landing), mdlFwd2_2 (takeoff), mdlFwd2_3 (transit) */
    const emb_model* int_bck[3];       /* mdlBck2_1, mdlBck2_2, mdlBck2_3 */
} emb_terminal_models;
/* Every model must have labels_initial {"intent","distance","bearing","heading","altitude","speed"} with heading,
 * altitude, speed in positions 4-6 (createEncounter.m:107-116), exactly those three dynamic variables, no
 * dynamic->dynamic edge, and the stay prior of createEncounter.m:129 already set:
 * emb_set_prior(m, 1, EMB_PRIOR_STAY, 1.0).  The same emb_model may appear in several slots. */

#define EMB_TRAJ_FIELDS 5 /* x_nm, y_nm, z_ft, heading_deg, v_ft_s; t_s is the slot index */
typedef struct emb_traj_out {
    /* merged, time-sorted trajectories traj(1:2) of createEncounter.m:74-84:
     * traj[field][aircraft][slot][n] with slot k <-> t_s = k - floor(tmax_s), aircraft 0 = ownship, 1 = intruder;
     * NaN in the slots an aircraft does not reach */
    float* traj;     /* [EMB_TRAJ_FIELDS][2][2*floor(tmax_s)+1][n]                                  nullable */
    /* len[2*aircraft + 0][s] = numel(fwd.t_s), len[2*aircraft + 1][s] = numel(bck.t_s): the aircraft has states for
     * t_s = -(len_bck-1) .. len_fwd-1 */
    int16_t* len;    /* [4][n]                                                                      nullable */
} emb_traj_out;
/* geo: the encounter-geometry samples (outInits of @CorTerminalModel/sample.m), row-major [rows][geo_stride] doubles,
 * column s = encounter first_sample + s; geo_rows[12] = 0-based rows of own_intent, own_distance, own_bearing,
 * own_alt, own_heading, own_speed, int_intent, ... int_speed (sample_geo of createEncounter.m:14-49).  `geo` lives
 * in opts->mem like the outputs.  opts: mem, device, stream, max_attempts are used; limits[0] ownship, [1] intruder.
 * An intent outside 1..2 (own) / 1..3 (intruder) gives EMB_E_ARG "Unknown int_intent" after the call completes. */
int emb_terminal_propagate(const emb_terminal_models* models, const emb_rng* rng, int64_t n, const double* geo,
                           int64_t geo_stride, const int32_t* geo_rows, double tmax_s, const emb_dyn_limits* limits,
                           const emb_sample_opts* opts, const emb_traj_out* out);
int64_t emb_terminal_traj_len(int64_t n, double tmax_s); /* elements of emb_traj_out.traj */

/* ---- encounter screening on the output of emb_terminal_propagate: getGeneratedMissDistance
 *      (@CorTerminalModel/CorTerminalModel.m:117-133), the overlap length of @CorTerminalModel/track.m:88 and
 *      CheckRunwayProximity (CorTerminalModel.m:187-210).  traj / len as in emb_traj_out (same memory kind as the outputs). */
typedef struct emb_screen_out {
    double* hmd_ft;       /* [n]                                                                       nullable */
    double* vmd_ft;       /* [n]  z_int - z_own at the CPA                                             nullable */
    int16_t* tcpa;        /* [3][n]: tcpa_s, tcpa_index_own, tcpa_index_int (1-based, MATLAB indices)  nullable */
    int16_t* enc_time_s;  /* [n]  numel(intersect(traj(1).t_s, traj(2).t_s))                           nullable */
    uint8_t* runway;      /* [n]  bit0 is_close1, bit1 is_low1, bit2 is_close2, bit3 is_low2           nullable */
} emb_screen_out;
int emb_terminal_screen(const float* traj, const int16_t* len, int64_t n, double tmax_s, double thres_dist_ft,
                        double thres_altlow_ft, const emb_sample_opts* opts /* mem, device, stream */,
                        const emb_screen_out* out);

/* ---- first-order track integration: replaces the per-track loop of sample2track.m:188-244 (Euler update :199-218,
 *      CFIT and speed rejection :234-244) on the dense compact output of emb_sample_tracks ------------------------------ */
typedef struct emb_integrate_opts {
    int32_t idx_altitude, idx_speed;                      /* 1-based initial variables: 'L' (initial altitude, ft), 'v' */
    int32_t idx_acceleration, idx_vertrate, idx_turnrate; /* 1-based ids of the dynamic variables \dot v, \dot h, \dot\psi */
    double ur_speed, ur_vertrate, ur_heading;             /* unit ratios of sample2track.m:108-125 (kt->ft/s, ft/min->ft/s, 1) */
    double min_speed, max_speed;                          /* boundaries{v}([1 end]) * ur_speed (:98-99, :140-141) */
    int32_t mem, device;                                  /* EMB_MEM_*, CUDA ordinal (-1 = current) */
    void* stream;
} emb_integrate_opts;
/* init_values: double [n_initial][n] and values: float [ceil(T/4)][ceil(n/128)][n_timevarying][128][4] as written by emb_sample_tracks;
 * xyz: float [3][T+1][n] = x_ft, y_ft, z_ft at time_s = 0..T (nullable); is_good: uint8 [n] (nullable). */
int emb_tracks_integrate(const emb_model* m, int64_t n, int32_t T, const double* init_values, const float* values,
                         const emb_integrate_opts* opts, float* xyz, uint8_t* is_good);

/* Sampling and integration in ONE pass (sample2track.m:188-244 fused into the track kernel): the Euler loop runs on the values of
 * four seconds while they are in registers, so (x, y, z) leave the device without the dense tiles making a round trip through HBM.
 * `out` may be NULL or carry any of emb_sample_tracks' outputs except the histograms (dense bins / values are then written as well);
 * xyz, is_good as in emb_tracks_integrate, in opts->mem memory; iopts->mem / device / stream are ignored (opts' are used).
 * Identical results to emb_sample_tracks followed by emb_tracks_integrate.  Models without a specialised track kernel run
 * exactly that two-pass route internally. */
int emb_sample_tracks_xyz(const emb_model* m, const emb_rng* rng, int64_t n, int32_t T, const emb_sample_opts* opts,
                          const emb_integrate_opts* iopts, const emb_track_out* out, float* xyz, uint8_t* is_good);

/* ---- log-likelihood of given bins under a model: the inverse of the sampling entry points, for importance weights p(x)/q(x),
 *      model comparison and validation.  Nothing in the reference computes this; the conditionals are the reference's own.
 *
 * Every conditional probability is the model's, in fp64: log(w_m / W), w the column of N + alpha that select_random.m:17 selects
 * from (so emb_set_prior and emb_model_from_arrays weights apply exactly as they do to sampling), W = sum(w).  A zero-total column
 * gives bin 1 with probability 1 as the sampler does (log-prob 0 for bin 1, -inf otherwise); a zero-weight bin gives -inf.
 * These are the model's probabilities, not the sampler's word-space ones (emb_device.cuh), which differ by at most 2^-32 per bin.
 *
 * Initial network: log p(x) = sum_i log p(x_i | parents), parents addressed by asub2ind.m.
 * Tracks: the state at dense column c is the tile bins of the dynamic variables at c plus init_bins for the static variables.
 * The transition term sums over c = 1 .. T-1 and every dynamic variable; the parent configuration follows the branch the sampler
 * uses: frozen at column 0 for a model without a dynamic -> dynamic edge (dbn_sample.m:110-135, SURVEY F6), re-evaluated every
 * second otherwise or when opts->correct_dbn = 1 (dbn_sample.m:66-79).  Column 0 is the initial state: the initial term scores it.
 * Not included: the rejection truncation of EMB_REJECT_* (these are unnormalised model probabilities), within-bin value
 * densities (de-discretisation), and the resample gates (they change values, not bins).
 *
 * opts: only mem (EMB_MEM_HOST / EMB_MEM_DEVICE for every buffer; EMB_MEM_ASYNC is refused), device, stream and correct_dbn are
 * read.  Calls are synchronous.  EMB_E_ARG when a bin is outside 1..r, when tile column 0 differs from init_bins of the dynamic
 * variables, or (tracks) for a model without a transition network ("dynvar:empty").  Padding tracks and padding seconds of the
 * tiles are ignored; the tiles beyond column 0 are read only when `transition` is requested. */
/* log p of initial-network bins [n_initial][n] (emb_sample_initial's layout): total[n] and, nullable, per_var[n_initial][n]
 * (a caller who sampled with `start` presets drops the preset variables' rows to get the conditional) */
int emb_loglik_initial(const emb_model* m, int64_t n, const int8_t* bins, const emb_sample_opts* opts,
                       double* total, double* per_var);
/* log p of tracks: init_bins [n_initial][n] and the tiled dense bins of emb_sample_tracks (emb_tracks_bins_len(m, n, T)
 * elements); initial[n] / transition[n] nullable */
int emb_loglik_tracks(const emb_model* m, int64_t n, int32_t T, const int8_t* init_bins, const int8_t* bins,
                      const emb_sample_opts* opts, double* initial, double* transition);

/* ---- misc ------------------------------------------------------------------------------------- */
int emb_host_alloc(void** p, int64_t bytes); /* pinned host memory */
int emb_host_free(void* p);
int emb_device_count(void);
/* Per-call temporaries (staging buffers, event rows) are kept in the device's stream-ordered memory pool between calls so that
 * repeated calls do not pay cudaMalloc/cudaFree; this returns that memory to the driver (device < 0: the current device). */
int emb_trim_device_memory(int device);
/* waits for the device and returns EMB_E_REJECT if an EMB_MEM_ASYNC pass since the last call exhausted max_attempts, else 0 */
int emb_async_status(int device);
const char* emb_last_error(void);
int emb_abi_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t emb_launch_count(void);
/* test hooks: force the generic kernel (1) so the specialised and generic kernels can be compared;
 * whether the last emb_sample_tracks ran a specialised (1) or the generic (0) kernel */
void emb_debug_force_generic(int on);
int emb_debug_last_kernel_fast(void);

#ifdef __cplusplus
}
#endif
#endif /* EMB200_H */
