/* include/bsg.h -- C ABI of libbsg_b200.so: the B200-native batched BlueSky-Gym step path.
 *
 * The reference (svlaskin/bluesky-gym-sasha) is pure Python and has no FFI of its own; the boundary
 * its hot path sits behind is the gymnasium Env API (bluesky_gym/__init__.py:4-46 registration,
 * Env.reset / Env.step in bluesky_gym/envs/<env>.py).  Each entry point below therefore cites the
 * reference *Python* interface it replaces; INTEGRATION.md shows the ctypes stub a maintainer adds.
 *
 * Conventions: extern "C", plain pointers and sizes, no torch / CUDA types in the signatures
 * (streams travel as void* = cudaStream_t).  Every function returns 0 on success or a negative
 * BSG_E* code; bsg_last_error() returns a thread-local message.  No exceptions cross the boundary,
 * there is no global state, and one handle serves one (process, device).  Memory is owned by the
 * caller (torch tensors in the Python host); the library holds raw device pointers only between
 * bsg_bind_state() and bsg_destroy() and never frees them.  Calls on one handle are not
 * thread-safe; different handles may be driven from different threads or processes.
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with BSG_ECUDA.
 */
#ifndef BSG_H_
#define BSG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSG_ABI_VERSION 6

enum { BSG_OK = 0, BSG_EINVAL = -1, BSG_ECUDA = -2, BSG_ESTATE = -3, BSG_ENOMEM = -4 };

/* gym ids of bluesky_gym/__init__.py:7-46 that are on the accelerated path */
enum {
    BSG_ENV_DESCENT = 0,        /* DescentEnv-v0       descent_env.py       */
    BSG_ENV_HORIZONTAL_CR = 1,  /* HorizontalCREnv-v0  horizontal_cr_env.py */
    BSG_ENV_SECTOR_CR = 2,      /* SectorCREnv-v0      sector_cr_env.py     */
    BSG_ENV_MERGE = 3,          /* MergeEnv-v0         merge_env.py         */
    BSG_ENV_PLAN_WAYPOINT = 4,  /* PlanWaypointEnv-v0  plan_waypoint_env.py */
    BSG_ENV_VERTICAL_CR = 5,    /* VerticalCREnv-v0    vertical_cr_env.py   */
    BSG_ENV_STATIC_OBSTACLE = 6 /* StaticObstacleEnv-v0 static_obstacle_env.py */
};

/* vector autoreset behaviour (gymnasium.vector.AutoresetMode) */
enum { BSG_AUTORESET_DISABLED = 0, BSG_AUTORESET_NEXT_STEP = 1, BSG_AUTORESET_SAME_STEP = 2 };

/* OpenAP-lite envelope of the one aircraft type the reference flies ("A320", e.g.
 * horizontal_cr_env.py:91).  Data, not code: see oracle/perf.py::PerfTable. */
typedef struct bsg_perf {
    float vminto, vmaxic, vminer, vmaxer, vminap, vmaxap;   /* m/s CAS */
    float vsmin, vsmax;                                     /* m/s     */
    float hmax;                                             /* m       */
    float mmo;
    float axmax_gd, axmax_air;                              /* m/s^2   */
} bsg_perf;

typedef struct bsg_config {
    int32_t env_type;           /* BSG_ENV_*                                                        */
    int32_t num_envs;           /* E: env instances on this device                                   */
    int32_t n_intruders;        /* HorizontalCR only: reference 5 (horizontal_cr_env.py:17)          */
    int32_t cd_enabled;         /* run StateBased.detect every substep (off in the reference);        */
                                /* 2 = same results, candidate filter redone every substep (test knob) */
    int32_t autoreset_mode;     /* BSG_AUTORESET_*                                                   */
    int32_t max_episode_steps;  /* TimeLimit of the registration, bluesky_gym/__init__.py:9-45       */
    int32_t default_hdg_random; /* Traffic.cre(achdg=None) draws randint(1,360) when 1, else 0 deg   */
    int32_t device;             /* CUDA ordinal                                                      */
    uint64_t seed;              /* Philox key part; stream = (seed, env_id_offset + e, episode)      */
    int64_t env_id_offset;      /* global id of env 0 on this device (sharding is placement-free)    */
    float rpz, hpz, dtlookahead;/* ASAS zone [m], [m], [s]; <= 0 selects 5 NM / 1000 ft / 300 s      */
    bsg_perf perf;
    int32_t wind_obs;           /* WindFieldWrapper(augment_obs=True): append wind_u, wind_v to obs  */
    int32_t sector_density_uniform; /* SectorCREnv(ac_density_mode != "normal"): uniform(0.003, 0.007) traffic
                                     * density instead of normal(0.005, 0.001), sector_cr_env.py:98-103  */
    float init_alt;             /* HorizontalCR: altitude [m] every aircraft is created at.  Reference: 0
                                 * (horizontal_cr_env.py:91, cre without acalt => ground phase, CAS capped near
                                 * 88 m/s); SURVEY 8d also measures a 3000 m variant (aircraft keep 150 m/s CAS) */
    int32_t cd_pair_cap;        /* in-sim ASAS pair list: entries per env in tensor_table.cd_pairs / cd_attr
                                 * (0 = lists off; slots*(slots-1)/2 holds every pair)                         */
} bsg_config;

/* What the caller must allocate (all device memory, zero-initialised) for a given config. */
typedef struct bsg_layout {
    int32_t slots;              /* G: aircraft slots per env (1, 8, 16 or 32), slot index fastest    */
    int32_t obs_dim;            /* floats per env in obs / final_obs                                 */
    int32_t act_dim;            /* floats per env in actions                                         */
    int32_t info_dim;           /* floats per env in info                                            */
    int32_t n_sub;              /* simulator substeps per env step (ACTION_FREQUENCY)                */
    int32_t env_f64, env_f32, env_i32; /* per-env scalar record widths                               */
    int32_t poly_f64;           /* per-env polygon doubles (SectorCR: 2*32; StaticObstacle: 360), else 0 */
    float simdt;
} bsg_layout;

/* Device pointers of caller-owned tensors.  Per-aircraft arrays have E*G elements.                 */
typedef struct bsg_tensor_table {
    double *pos;        /* [E*G] double2 (lat, lon) deg            bs.traf.lat / lon                 */
    float *kin;         /* [E*G] float4  (alt m, tas m/s, hdg deg, vs m/s)    bs.traf.alt/tas/hdg/vs  */
    float *cmd;         /* [E*G] float4  (selspd, selalt, selvs, ap.trk)      bs.traf.sel*, ap.trk    */
    float *aux;         /* [E*G] float4  (ax, curlegdir, cas, reserved)                              */
    uint32_t *flags;    /* [E*G] bit0 alive, bit1 swlnav, bit2 swlastwp, bits 8.. active wp index    */
    float *tcpamax;     /* [E*G] ASAS tcpamax per aircraft (cd_enabled)                              */
    uint8_t *inconf;    /* [E*G] ASAS inconf per aircraft  (cd_enabled)                              */
    double *env_f64;    /* [E*env_f64]                                                               */
    float *env_f32;     /* [E*env_f32]                                                               */
    int32_t *env_i32;   /* [E*env_i32]                                                               */
    double *poly;       /* [E*poly_f64] or NULL                                                      */
    float *obs;         /* [E*obs_dim]   Env._get_obs, keys concatenated in declaration order        */
    float *final_obs;   /* [E*obs_dim]   SAME_STEP autoreset: terminal observations, COMPACT -- row k is the */
                        /*               terminal obs of env final_ids[k], k < final_count[final_count[2]]; may be NULL */
    int32_t *final_ids; /* [E]           env index of each compact final_obs row (needed with final_obs)    */
    int32_t *final_count;/* [4]          [2] = s in {0, 1}; [s] = number of envs that finished in the last step (two  */
                        /*               counters take turns so that no memset sits between two step launches) */
    float *reward;      /* [E]                                                                       */
    uint8_t *terminated;/* [E]                                                                       */
    uint8_t *truncated; /* [E]                                                                       */
    float *info;        /* [info_dim][E] Env._get_info values at the end of the step (pre-autoreset), key-major: */
                        /*               one contiguous row of E values per info key                          */
    float *actions_staging; /* [E*act_dim] device staging buffer used by bsg_step_host, may be NULL  */
    /* in-sim ASAS pair lists of the LAST simulator substep (bs.traf.cd.confpairs / lospairs and the per-conflict
     * qdr, dist, dcpa, tcpa, tinconf of upstream's detect()), cfg.cd_pair_cap entries per env, count in
     * env_i32[BSG_I32_NPAIRS] (true number found; entries beyond the capacity are dropped).  One entry per UNORDERED
     * pair i < j that is a conflict in either order or a LoS:
     *   cd_pairs: i | j << 8 | BSG_PAIR_CONF_IJ | BSG_PAIR_CONF_JI | BSG_PAIR_LOS
     *   cd_attr : BSG_PAIR_ATTR_COUNT floats (qdr i->j [deg], dist [m], dcpa [m], tcpa [s], tinconf (i,j), tinconf (j,i))
     * Both may be NULL (cd_attr alone may be NULL too). */
    uint32_t *cd_pairs;     /* [E*cd_pair_cap]                                                          */
    float *cd_attr;         /* [E*cd_pair_cap*BSG_PAIR_ATTR_COUNT]                                       */
} bsg_tensor_table;
enum { BSG_PAIR_CONF_IJ = 1 << 16, BSG_PAIR_CONF_JI = 1 << 17, BSG_PAIR_LOS = 1 << 18 };
enum { BSG_PAIR_ATTR_QDR = 0, BSG_PAIR_ATTR_DIST = 1, BSG_PAIR_ATTR_DCPA = 2, BSG_PAIR_ATTR_TCPA = 3,
       BSG_PAIR_ATTR_TINCONF_IJ = 4, BSG_PAIR_ATTR_TINCONF_JI = 5, BSG_PAIR_ATTR_COUNT = 6 };

/* indices into the per-env records (shared by all env types; unused slots stay zero) */
enum { BSG_F64_WPT_LAT = 0, BSG_F64_WPT_LON = 1, BSG_F64_TARGET_ALT = 2, BSG_F64_POLY_AREA = 3,
       BSG_F64_WPTS = 4 /* PlanWaypoint: 5 x (lat, lon) */, BSG_F64_COUNT = 16 };
enum { BSG_F32_TOTAL_REWARD = 0, BSG_F32_DRIFT_SUM = 1, BSG_F32_FINAL_ALT = 2, BSG_F32_LAST_HDG = 3,
       BSG_F32_LAST_WDIST = 4, BSG_F32_LAST_DRIFT = 5 /* StaticObstacle: values of the last _get_obs */, BSG_F32_COUNT = 8 };
enum {
    BSG_I32_STEP = 0, BSG_I32_EPISODE = 1, BSG_I32_SIMK = 2, BSG_I32_WPT_REACH = 3, BSG_I32_DRIFT_N = 4,
    BSG_I32_INTRUSIONS = 5, BSG_I32_NUM_AC = 6, BSG_I32_NVERT = 7, BSG_I32_NEEDS_RESET = 8,
    BSG_I32_FAF = 9, BSG_I32_NCONF = 10, BSG_I32_NLOS = 11, BSG_I32_RESET_FLAGS = 12, BSG_I32_NPAIRS = 13,
    BSG_I32_COUNT = 16
};

typedef struct bsg_handle bsg_handle;

int bsg_abi_version(void);
/* sizeof of the library's view of an interface structure (which: 0 bsg_config, 1 bsg_layout, 2 bsg_tensor_table,
 * 3 bsg_wind, 4 bsg_perf, 5 bsg_ac_state, 6 bsg_cd_lists, 7 bsg_traf_config, 8 bsg_traf_tensors, 9 bsg_traf_events; anything else -1): a binding in another language checks its own declarations against it */
int bsg_abi_struct_size(int which);
const char *bsg_last_error(void);
int bsg_device_count(void);

/* Fills the allocation plan for cfg.  Pure host logic: works without a GPU. */
int bsg_query_layout(const bsg_config *cfg, bsg_layout *out);

/* replaces: Env.__init__ (bs.init + 'DT n;FF'), e.g. horizontal_cr_env.py:41-80 */
int bsg_create(const bsg_config *cfg, bsg_handle **out);
void bsg_destroy(bsg_handle *h);
int bsg_bind_state(bsg_handle *h, const bsg_tensor_table *t);

/* replaces: Env.reset, e.g. horizontal_cr_env.py:82-101, sector_cr_env.py:87-115, merge_env.py:103-130,
 * descent_env.py:162-182.  d_mask: E bytes on the device, non-zero = reset that env; NULL = all. */
int bsg_reset(bsg_handle *h, const uint8_t *d_mask, void *stream);

/* replaces: Env.step, e.g. horizontal_cr_env.py:103-125 (action -> n_sub x bs.sim.step() -> obs ->
 * reward -> terminated/truncated -> info), plus the TimeLimit wrapper and vector autoreset.
 * d_actions: [E*act_dim] float32 on the device.  Asynchronous on `stream`. */
int bsg_step(bsg_handle *h, const float *d_actions, void *stream);

/* End-to-end form of bsg_step for host callers (SB3 / numpy): copies h_actions (pinned or pageable)
 * to the device, steps, copies obs / reward / terminated / truncated / info back and synchronises. */
int bsg_step_host(bsg_handle *h, const float *h_actions, float *h_obs, float *h_reward,
                  uint8_t *h_terminated, uint8_t *h_truncated, float *h_info, int32_t *h_final_count,
                  void *stream);

/* Same as bsg_step_host for callers that allocated the step outputs as ONE contiguous device block that
 * starts at tensor_table.obs and keep a pinned host mirror of it: copies h_actions in, steps, copies the
 * first `nbytes` bytes of that block to h_block and synchronises (one copy each way per env step).
 * Replaces the same reference call as bsg_step (Env.step, e.g. horizontal_cr_env.py:103-125). */
int bsg_step_host_block(bsg_handle *h, const float *h_actions, void *h_block, size_t nbytes, void *stream);

/* bsg_step_host_block that additionally copies the first `dst_bytes` bytes of the mirrored block (the
 * observations) from the pinned mirror into `dst`, the caller's own (pageable) result array, using the
 * library's host threads (BSG_HOST_THREADS; default 3/4 of the rank's share of the cores) and overlapping that copy with the device->host
 * transfer chunk by chunk.  dst may be NULL (then identical to bsg_step_host_block). */
int bsg_step_host_copy(bsg_handle *h, const float *h_actions, void *h_block, size_t nbytes,
                       void *dst, size_t dst_bytes, void *stream);

/* bsg_step_host_block in two halves, for callers that have work of their own to overlap with the step (SB3's
 * VecEnv.step_async / step_wait, stable_baselines3 as driven by the reference's main.py:36-55): _begin enqueues the
 * copy of h_actions, the step and the copy of the first `nbytes` bytes of the output block to h_block on `stream` and
 * returns without waiting; _wait blocks until that transfer has landed and, when dst is not NULL, copies the first
 * dst_bytes bytes of h_block into dst with the library's host threads.  One step may be in flight per handle
 * (BSG_ESTATE otherwise); h_actions and h_block must stay valid until _wait returns. */
int bsg_step_host_begin(bsg_handle *h, const float *h_actions, void *h_block, size_t nbytes, void *stream);
int bsg_step_host_wait(bsg_handle *h, const void *h_block, void *dst, size_t dst_bytes);

/* The host-thread copy bsg_step_host_copy uses, on its own (pure host code; works without a GPU). */
int bsg_host_copy(void *dst, const void *src, size_t nbytes);
/* dst[i] = (double)src[i], i < n, with the same host threads: the float64 observations of the reference's spaces
 * (e.g. horizontal_cr_env.py:49-62 declare np.float64) from the float32 block the device writes. */
int bsg_host_widen(double *dst, const float *src, size_t n);

/* replaces: Env.reset(seed=...) (gymnasium seeding, e.g. horizontal_cr_env.py:82-83 super().reset(seed=seed)):
 * re-keys the Philox streams of the scenario generators and of the observation noise; takes effect at the next
 * reset of each env (stream = (seed, env_id_offset + e, episode)). */
int bsg_set_seed(bsg_handle *h, uint64_t seed);

/* replaces: WindFieldWrapper (bluesky_gym/wrappers/wind.py:8-64) = bs.traf.wind.addpointvne(lat, lon, vnorth,
 * veast, alt) + the wind terms of upstream Traffic.update_groundspeed / APorASAS.update / Autopilot.selhdgcmd.
 * Wind vectors at n_points lat/lon points, interpolated with inverse-distance-squared weights; n_alt == 1: no
 * altitude dependence, else vn/ve hold n_alt rows (row k = altitude k * alt_step, upstream: 100 ft steps to
 * 45 000 ft) of n_points values.  All pointers are DEVICE memory owned by the caller and must stay valid until
 * the wind is cleared or the handle destroyed; d_gs is [E * slots * 2] floats (ground-speed north / east per
 * aircraft, persistent state that only exists with wind).  w == NULL or n_points == 0 switches the wind off. */
typedef struct bsg_wind {
    int32_t n_points, n_alt;
    float alt_step;             /* [m] */
    const float *d_lat, *d_lon; /* [n_points] deg */
    const float *d_vn, *d_ve;   /* [n_alt * n_points] m/s */
    float *d_gs;                /* [E * slots * 2] */
} bsg_wind;
int bsg_set_wind(bsg_handle *h, const bsg_wind *w);

/* replaces: NoisyObservationWrapper (bluesky_gym/wrappers/uncertainty.py:4-31): from now on every observation
 * written by bsg_reset / bsg_step* (terminal observations of same-step autoreset included) carries independent
 * Gaussian noise N(0, sigma) per element, drawn from a Philox stream keyed by (seed, global env id, call index).
 * sigma = 0 switches it off.  One extra elementwise kernel per call while it is on. */
int bsg_set_obs_noise(bsg_handle *h, float sigma);

/* The observation-noise stream's call index (number of reset / step calls made with noise on): part of a checkpoint,
 * because the stream is keyed by (seed, global env id, call index).  bsg_set_noise_calls restores it. */
int bsg_get_noise_calls(bsg_handle *h, uint32_t *out);
int bsg_set_noise_calls(bsg_handle *h, uint32_t calls);

/* replaces: the state a reference env holds after Env.reset() -- bs.traf.* arrays after bs.traf.cre / creconfs
 * (e.g. horizontal_cr_env.py:85-101) plus the env's own members (waypoint, polygon, counters) -- injected from HOST
 * arrays into env `env` of the batch, so a parity test can start the device simulator from a reference / oracle
 * post-reset state.  Arrays hold s->n aircraft (n <= layout.slots; the remaining slots are cleared).  NULL optional
 * arrays take the stated default; env_f64 / env_f32 / env_i32 / poly are WHOLE per-env records (layout.env_f64 ...
 * layout.poly_f64 elements) or NULL = left as they are.  Synchronises `stream` before returning. */
typedef struct bsg_ac_state {
    int32_t n;
    const double *lat, *lon;                        /* bs.traf.lat / lon [deg]                       */
    const double *alt, *tas, *hdg, *vs;             /* bs.traf.alt / tas / hdg / vs                  */
    const double *selspd, *selalt, *selvs, *ap_trk; /* bs.traf.selspd / selalt / selvs, ap.trk       */
    const double *cas;                              /* bs.traf.cas                                   */
    const double *ax;                               /* bs.traf.ax                    (NULL: 0)       */
    const double *curlegdir;                        /* actwp.curlegdir               (NULL: -999)    */
    const uint8_t *swlnav;                          /* bs.traf.swlnav                (NULL: off)     */
    const int32_t *iactwp;                          /* route.iactwp, >= 1 = last wp  (NULL: 0)       */
    const double *env_f64; const float *env_f32; const int32_t *env_i32; const double *poly;
} bsg_ac_state;
int bsg_load_state(bsg_handle *h, int32_t env, const bsg_ac_state *s, void *stream);

/* replaces: n_sub x bs.sim.step() alone (Traffic.update kinematics + autopilot, no obs/reward);
 * used by the trajectory parity tests. */
int bsg_traf_update(bsg_handle *h, int32_t n_sub, void *stream);

/* ---- single-airspace state-based conflict detection (StateBased.detect; CD record = 32 B) -------- */

/* CD record storage, tile-blocked: d_rec[tile][BSG_CD_REC_FIELDS][BSG_CD_TILE] floats, tile = aircraft index /
 * BSG_CD_TILE; field k of aircraft j is d_rec[(j / BSG_CD_TILE) * BSG_CD_TILE * BSG_CD_REC_FIELDS + k * BSG_CD_TILE +
 * j % BSG_CD_TILE].  Fields: x, y [m of arc from (lat0, lon0)], ch, sh (cos, sin of half the latitude), u, v [m/s east,
 * north], alt [m], vs [m/s].  Padding records are inert: ch = 1, alt = 3e9, every other field 0. */
enum { BSG_CD_TILE = 256,
       BSG_CD_REC_X = 0, BSG_CD_REC_Y = 1, BSG_CD_REC_CH = 2, BSG_CD_REC_SH = 3,
       BSG_CD_REC_U = 4, BSG_CD_REC_V = 5, BSG_CD_REC_ALT = 6, BSG_CD_REC_VS = 7, BSG_CD_REC_FIELDS = 8 };

/* Packs float64 SoA aircraft state (bs.traf.lat/lon/trk/gs/alt/vs) into 32-byte CD records (BSG_CD_REC_*).
 * d_rec must hold bsg_cd_padded(n) records; the padding of the last tile is filled with inert aircraft. */
int64_t bsg_cd_padded(int64_t n);
int bsg_cd_pack(const double *d_lat, const double *d_lon, const double *d_trk, const double *d_gs,
                const double *d_alt, const double *d_vs, int64_t n, double lat0, double lon0,
                float *d_rec, void *stream);

/* bsg_cd_pack with the aircraft laid out in a spatially coherent order chosen on the device (uniform grid over their
 * bounding box, strip by strip, alternate strips reversed; counting sort, no library call): what makes
 * bsg_cd_detect_culled effective.  d_perm [n] receives the order: record k holds aircraft d_perm[k] (indices in the
 * detection's outputs are record indices: map them back through d_perm).  The order inside a grid cell is unspecified;
 * the detection's outputs (sets, counts, maxima) do not depend on it.  d_work: 8-byte aligned device scratch of
 * bsg_cd_order_workspace(n) bytes.  Replaces: the sort of StateBasedCD.detect(cull=True) (formerly two library radix
 * sorts and six gathers). */
int64_t bsg_cd_order_workspace(int64_t n);
int bsg_cd_pack_ordered(const double *d_lat, const double *d_lon, const double *d_trk, const double *d_gs,
                        const double *d_alt, const double *d_vs, int64_t n, double lat0, double lon0,
                        float *d_rec, int32_t *d_perm, void *d_work, int64_t work_bytes, void *stream);

enum { BSG_CD_LON_WRAP = 1,     /* pairs may straddle the +-180 deg meridian relative to lon0        */
       BSG_CD_SYMMETRIC = 2,    /* bsg_cd_detect_culled: evaluate each unordered tile pair once and emit both
                                 * ordered results (needs n_rows == n_all); same outputs, half the work  */
       BSG_CD_CULL = 4,         /* bsg_cd_detect_peers: use the culled form (needs the workspace)    */
       BSG_CD_ALLTILES = 8 };   /* bsg_cd_detect_culled: keep every tile pair (no culling; with
                                 * BSG_CD_SYMMETRIC = brute force over unordered pairs)              */
/* bsg_cd_detect_culled over several GPUs that all hold every record (after an all-gather): GPU k of n evaluates the row
 * blocks (256 rows) whose index % n == k, the others' lists stay empty.  With BSG_CD_SYMMETRIC (row0 = 0, n_rows = n_all on
 * every GPU) the unordered tile pairs are thereby dealt round-robin -- the lists shrink with the row index, so this balances
 * -- and the per-row outputs of the GPUs add up: sum d_nconf_row / d_nlos_row / d_npairs and take the maximum of d_tcpamax
 * over the GPUs (one all-reduce each); d_inconf is nconf > 0 after the sum.  n, k <= 255. */
#define BSG_CD_DEAL(n, k) ((((uint32_t)(n)) & 0xffu) << 8 | (((uint32_t)(k)) & 0xffu) << 16)

/* Pair lists of a detection = what upstream's StateBased.detect returns besides the per-aircraft flags:
 * confpairs, lospairs and, per conflict, qdr / dist / dcpa / tcpa / tinconf.  All DEVICE memory owned by the caller;
 * any pointer may be NULL (that output is then only counted).  Entries are written in arbitrary order (upstream's
 * order is row-major np.where; sort on the host if needed); conf_attr row k belongs to conf_pairs row k.  When more
 * pairs exist than the capacity holds the lists are truncated, d_npairs keeps the true totals. */
enum { BSG_CD_ATTR_QDR = 0 /* deg [0, 360) own -> intruder */, BSG_CD_ATTR_DIST = 1 /* m */, BSG_CD_ATTR_DCPA = 2 /* m */,
       BSG_CD_ATTR_TCPA = 3 /* s */, BSG_CD_ATTR_TINCONF = 4 /* s */, BSG_CD_ATTR_COUNT = 5 };
typedef struct bsg_cd_lists {
    int32_t *d_conf_pairs;              /* [conf_cap][2] ordered (own, intruder) global indices             */
    float *d_conf_attr;                 /* [conf_cap][BSG_CD_ATTR_COUNT]                                    */
    int64_t conf_cap;
    int32_t *d_los_pairs;               /* [los_cap][2]                                                     */
    int64_t los_cap;
    unsigned long long *d_npairs;       /* [2]: conflicts found, LoS pairs found (required with any list)   */
} bsg_cd_lists;

/* Maps the outputs of a detection on reordered records (record k = aircraft d_perm[k], d_perm a permutation of [0, n))
 * back to aircraft order, on the device.  The rows of both pair lists of `lists` -- the first min(npairs, cap) of each,
 * npairs read on the device (no host synchronisation) -- are rewritten in place, (a, b) -> (d_perm[a], d_perm[b]); rows
 * past them are untouched, the attributes stay as they are.  Per-row outputs are scattered, out[d_perm[k]] = in[k], k < n;
 * each in / out pair may be NULL (both), and must not alias.  `lists` may be NULL.  One launch, O(pairs + n). */
int bsg_cd_unpermute(const int32_t *d_perm, int64_t n, const bsg_cd_lists *lists, const uint32_t *d_nconf_in,
                     const uint32_t *d_nlos_in, const float *d_tcpamax_in, const uint8_t *d_inconf_in,
                     uint32_t *d_nconf_out, uint32_t *d_nlos_out, float *d_tcpamax_out, uint8_t *d_inconf_out, void *stream);

/* Rows [row0, row0+n_rows) of d_rec against all n_all aircraft (row sharding for multi-GPU).
 * Outputs (caller-owned, device): per-row nconf / nlos counts and tcpamax, inconf flags, and the pair lists
 * (`lists` may be NULL).  Any output pointer except d_nconf_row may be NULL.
 * replaces: StateBased.detect(ownship, intruder, rpz, hpz, dtlookahead) -> confpairs, lospairs, inconf, tcpamax,
 * qdr, dist, dcpa, tcpa, tLOS (upstream bluesky/traffic/asas/statebased.py; SURVEY App. A.5). */
int bsg_cd_detect(const float *d_rec, int64_t n_all, int64_t row0, int64_t n_rows,
                  float rpz, float hpz, float dtlookahead, uint32_t flags,
                  uint32_t *d_nconf_row, uint32_t *d_nlos_row, float *d_tcpamax, uint8_t *d_inconf,
                  const bsg_cd_lists *lists, void *stream);

/* bsg_cd_detect with spatial culling: identical outputs, but column tiles that cannot contain a conflict or LoS
 * partner of a row block (farther apart at time 0 than rpz + (v_a + v_b) * dtlookahead, or vertically beyond
 * hpz + (|vs_a| + |vs_b|) * dtlookahead, from per-tile bounding boxes) are never evaluated.  It pays off when the
 * records are spatially coherent (sort the aircraft into compact tiles before bsg_cd_pack, as
 * StateBasedCD.detect(cull=True) does); on unsorted input every tile pair survives and it degenerates to
 * bsg_cd_detect plus three tiny kernels.  row0 must be a multiple of 256; no BSG_CD_LON_WRAP.
 * d_work: device scratch of at least bsg_cd_cull_workspace(n_all, n_rows) bytes. */
int64_t bsg_cd_cull_workspace(int64_t n_all, int64_t n_rows);
int bsg_cd_detect_culled(const float *d_rec, int64_t n_all, int64_t row0, int64_t n_rows, float rpz, float hpz,
                         float dtlookahead, uint32_t flags, uint32_t *d_nconf_row, uint32_t *d_nlos_row,
                         float *d_tcpamax, uint8_t *d_inconf, const bsg_cd_lists *lists,
                         void *d_work, int64_t work_bytes, void *stream);

/* Multi-GPU form without a gather: every GPU of the node packs its block of n_per_peer aircraft (a multiple of 256)
 * into a buffer that its peers can address (CUDA peer access / symmetric memory: torch.distributed._symmetric_memory
 * gives the pointers), and this call evaluates rank my_rank's rows against ALL columns, fetching column tile t
 * from h_peer_rec[t / (n_per_peer / 256)] directly over NVLink with the kernel's own TMA bulk copies -- the transfer
 * overlaps the pair arithmetic tile by tile and, with BSG_CD_CULL, only the tiles that survive culling ever cross the
 * link.  h_peer_rec is a HOST array of n_peers (<= 8) DEVICE pointers valid in this process.  The caller must make
 * sure all peers have finished packing before the call and keep their buffers unchanged until every rank's call has
 * completed (a barrier on each side; StateBasedCD.detect_sharded_p2p uses the symmetric-memory barrier).
 * Replaces: ncclAllGather + bsg_cd_detect(row0 = my_rank * n_per_peer, n_rows = n_per_peer). */
int bsg_cd_detect_peers(const float *const *h_peer_rec, int32_t n_peers, int32_t my_rank, int64_t n_per_peer,
                        float rpz, float hpz, float dtlookahead, uint32_t flags, uint32_t *d_nconf_row,
                        uint32_t *d_nlos_row, float *d_tcpamax, uint8_t *d_inconf, const bsg_cd_lists *lists,
                        void *d_work, int64_t work_bytes, void *stream);

/* ---- single-airspace traffic with routes, VNAV and ASAS resolution (SURVEY 8f-4) ---------------------------------
 * One airspace of n aircraft (the bs.traf of a BlueSky scenario at N = 1e5 instead of the handful a NumPy Traffic
 * can step): per simulator substep  bsg_traf_pack -> bsg_cd_detect[_culled] with pair lists -> bsg_traf_substep, which
 * indexes the conflict list by own aircraft and then fuses per aircraft: Autopilot.update (LNAV, update_fms over multi-waypoint
 * routes with altitude / speed constraints, ComputeVNAV, the continuous VNAV / speed guidance), ConflictResolution.update
 * (MVP.resolve over the aircraft's own conflicts in intruder order, resumenav with waypoint recovery), APorASAS.update,
 * perfoap.limits and Traffic.update_airspeed / update_groundspeed / update_pos.
 * Replaces upstream bluesky/traffic/{autopilot,route,aporasas}.py, asas/{resolution,mvp}.py as restated in
 * oracle/traffic_ext.py (the reference only ever says `reso off`, merge_env.py:157, and builds unconstrained two-waypoint
 * routes, merge_env.py:155-156).  Stateless: every call takes the configuration and the caller-owned DEVICE tensors. */
enum { BSG_TRAF_PARTNERS = 8 };         /* resopairs kept per aircraft (ConflictResolution.resopairs as rows)      */
enum { BSG_TF_ALIVE = 1, BSG_TF_LNAV = 2, BSG_TF_VNAV = 4, BSG_TF_VNAVSPD = 8, BSG_TF_LASTWP = 16, BSG_TF_ASAS = 32 /* cr.active */,
       BSG_TF_RESOOFF = 64, BSG_TF_PH_GD = 128 /* phase of the last perf.update: ground */, BSG_TF_PH_AP = 256 /* approach */,
       BSG_TF_ACTIVATE = 512 /* route uploaded, Route.direct(first waypoint) still to run */,
       BSG_TF_IWP_SHIFT = 16 /* active waypoint index, 8 bits */, BSG_TF_NWP_SHIFT = 24 /* waypoints in the route, 8 bits */ };
enum { BSG_TRAF_CTR_OVERFLOW = 0 /* resopairs that did not fit BSG_TRAF_PARTNERS */, BSG_TRAF_CTR_SWITCH = 1 /* waypoint switches */,
       BSG_TRAF_CTR_ACTIVE = 2 /* aircraft under ASAS command after the last substep */, BSG_TRAF_CTR_COUNT = 4 };
typedef struct bsg_traf_config {
    int64_t n;                  /* aircraft                                                               */
    int32_t max_wpts;           /* W: waypoint slots per route (<= 255)                                   */
    int32_t reso;               /* 0: detection only (RESO OFF); 1: MVP                                   */
    int32_t reso_mode;          /* 0: horizontal + vertical (upstream default); 1: horizontal only        */
    float simdt;
    float rpz, hpz, dtlookahead;
    float resofach, resofacv;   /* settings.asas_mar (1.01)                                               */
    bsg_perf perf;
    double lat0, lon0;          /* origin of the CD records                                               */
    int64_t row0;               /* airspace sharded over GPUs: index of this block's aircraft 0 in the records of the
                                 * whole airspace (a multiple of 256; 0 when the airspace is not sharded)  */
} bsg_traf_config;
typedef struct bsg_traf_tensors {
    double *pos;                /* [n][2] lat, lon [deg]                                                  */
    float *kin;                 /* [n][4] alt, tas, hdg, vs                                               */
    float *cmd;                 /* [n][4] selspd (CAS or Mach), selalt, selvs, ap.trk                     */
    float *aux;                 /* [n][4] ax, actwp.curlegdir, actwp.next_qdr, actwp.turndist             */
    double *actwp;              /* [n][2] active waypoint lat, lon                                        */
    float *vnav1;               /* [n][4] actwp.nextaltco, actwp.xtoalt, actwp.vs, ap.dist2vs             */
    float *vnav2;               /* [n][4] actwp.spd, actwp.nextspd, actwp.spdcon, ap.vnavvs               */
    float *asas;                /* [n][4] cr.trk, cr.tas, cr.vs, cr.alt                                   */
    uint32_t *flags;            /* [n] BSG_TF_*                                                           */
    int32_t *partners;          /* [n][BSG_TRAF_PARTNERS] intruder indices of the aircraft's resopairs, -1 = free */
    const double *rt_pos;       /* [n][W][2] route waypoints                                              */
    const float *rt_con;        /* [n][W][4] wpalt, wpspd (< 0: none), wptoalt, wpxtoalt (Route.calcfp)   */
    const float *rt_dir;        /* [n][W] direction of the leg from waypoint k to k + 1 [deg], -999 after the last */
    uint32_t *counters;         /* [BSG_TRAF_CTR_COUNT]                                                   */
} bsg_traf_tensors;
/* Traffic state -> CD records of bsg_cd_detect (trk = hdg, gs = tas: no wind); d_rec holds bsg_cd_padded(n) records. */
int bsg_traf_pack(const bsg_traf_config *cfg, const bsg_traf_tensors *t, float *d_rec, void *stream);
/* bsg_traf_pack with the records in a spatial order, for bsg_cd_detect_culled on an airspace whose index order is not
 * spatially coherent (created in any order, or flown for a long time).  reorder != 0: a fresh order of the n aircraft is
 * computed from their current positions into d_perm [n] (bsg_cd_pack_ordered's grid; dead slots stay out of the bounding
 * box); reorder == 0: the d_perm given is reused.  Record k of d_rec_ordered (bsg_cd_padded(n) records) is then aircraft
 * d_perm[k]'s record, bit for bit the one bsg_traf_pack writes, and padding is inert.  d_rec != NULL: the same launch also
 * writes the aircraft-order records of bsg_traf_pack (what bsg_traf_substep and bsg_traf_events_update read).  Map the
 * detection's outputs back with bsg_cd_unpermute.  d_work (needed with reorder != 0): 8-byte aligned device scratch of
 * bsg_traf_order_workspace(n) bytes.  Not for a sharded airspace (cfg->row0 must be 0).  Launches: 5 + 1 with reorder,
 * else 1. */
int64_t bsg_traf_order_workspace(int64_t n);
int bsg_traf_pack_ordered(const bsg_traf_config *cfg, const bsg_traf_tensors *t, int32_t reorder, int32_t *d_perm,
                          float *d_rec_ordered, float *d_rec, void *d_work, int64_t work_bytes, void *stream);
/* Route.direct(first waypoint) + ComputeVNAV for every aircraft flagged BSG_TF_ACTIVATE (after the route tables changed). */
int bsg_traf_activate(const bsg_traf_config *cfg, const bsg_traf_tensors *t, void *stream);
/* One simulator substep.  d_rec: the records bsg_traf_pack made of the state BEFORE this substep (what the detection saw);
 * d_conf_pairs [conf_cap][2], d_conf_attr [conf_cap][BSG_CD_ATTR_COUNT], d_npairs: the conflict list of that detection
 * exactly as bsg_cd_detect[_culled] wrote it (bsg_cd_lists: any order); all may be NULL with reso == 0.
 * d_work: device scratch of at least bsg_traf_workspace(n, conf_cap) bytes whose first n int32 are ZERO on entry (zero it
 * after allocation and whenever n changes: every call leaves them zero again).  fms_ready: the FMS timer fires in this substep (sim step
 * count % (10.5 // simdt) == 0).  Airspace sharded over GPUs (cfg->row0 = this block's first global index; SURVEY 8e: a rank
 * owns the kinematics of its block): d_rec holds the records of the WHOLE airspace (every rank's bsg_traf_pack output, all-gathered),
 * the conflict list that of bsg_cd_detect*(row0, n_rows = this block) with global indices, and d_nconf_all the number of
 * conflicts in the whole airspace (the all-reduced d_npairs[0]: upstream rewrites every aircraft's ASAS commands whenever ANY
 * conflict exists); d_nconf_all == NULL means d_npairs.  Launches: 3 small index kernels (count / allocate / scatter of the conflict list by own
 * aircraft; only with reso) + the fused per-aircraft kernel. */
int64_t bsg_traf_workspace(int64_t n, int64_t conf_cap);
int bsg_traf_substep(const bsg_traf_config *cfg, const bsg_traf_tensors *t, const float *d_rec, int32_t fms_ready,
                     const int32_t *d_conf_pairs, const float *d_conf_attr, const unsigned long long *d_npairs,
                     const unsigned long long *d_nconf_all, int64_t conf_cap, void *d_work, int64_t work_bytes, void *stream);

/* ---- conflict and loss-of-separation events of an airspace -------------------------------------------------------
 * Replaces the bookkeeping of upstream's ConflictDetection.update (bluesky/traffic/asas/detection.py): confpairs_all /
 * lospairs_all, i.e. the number of conflicts and LoS of an experiment, plus per event its start / end and, for LoS, its
 * severity.  Call bsg_traf_events_update once per detection, after bsg_cd_detect[_culled] on the same stream, with that
 * detection's lists.  An event is an UNORDERED pair (a < b) that is in the detection's conflict (LoS) list in either order;
 * it starts at the first detection that lists it after one that did not and ends (end = nstep) at the first later
 * detection that does not.  LoS events keep the minimum horizontal distance and |dalt| [m] over their detections, from
 * d_rec with cd_pair.cuh's algebra.  Totals count every event even when its log is full (rows beyond the capacity are
 * dropped and counted in BSG_EV_CTR_LOG_OVERFLOW); a detection with npairs > cap (lists incomplete) increments
 * BSG_EV_CTR_TRUNCATED, after which the log is unreliable.  Lists of one airspace on one GPU with global indices (not the
 * row-sharded form: there the two orders of a pair sit on different GPUs).  Asynchronous: no host synchronisation.
 * Stateless: everything lives in the caller-owned DEVICE memory below. */
enum { BSG_EV_CTR_NCONF_TOTAL = 0, BSG_EV_CTR_NLOS_TOTAL = 1 /* events so far (= log rows claimed) */,
       BSG_EV_CTR_NCONF_ACTIVE = 2, BSG_EV_CTR_NLOS_ACTIVE = 3 /* events open after the last detection */,
       BSG_EV_CTR_LOG_OVERFLOW = 4 /* events not logged (log full) */, BSG_EV_CTR_TRUNCATED = 5 /* detections with npairs > cap */,
       BSG_EV_CTR_COUNT = 8 };
typedef struct bsg_traf_events {
    void *d_cur;                /* set of this detection: set_bytes, 16-byte aligned                                      */
    void *d_prev;               /* set of the previous detection.  Both ZERO before the first call; the call leaves d_prev
                                 * zero again, so the caller swaps d_cur and d_prev after every call                       */
    int64_t set_bytes;          /* >= bsg_traf_events_workspace(conf_cap, los_cap) of the lists (the same caps every call) */
    int32_t *d_conf_log;        /* [conf_log_cap][4] a, b, start nstep, end nstep (-1 while open); row = event number      */
    int32_t *d_los_log;         /* [los_log_cap][4] the same for LoS events                                                */
    float *d_los_sev;           /* [los_log_cap][2] dmin, dalt_min [m]                                                     */
    int64_t conf_log_cap, los_log_cap;
    unsigned long long *d_counters; /* [BSG_EV_CTR_COUNT], zero before the first call                                   */
} bsg_traf_events;
/* Bytes of ONE set (a hash table of >= 2 x (conf_cap + los_cap) 16-byte slots and the dense list of its occupied slots). */
int64_t bsg_traf_events_workspace(int64_t conf_cap, int64_t los_cap);
/* d_rec: the records the detection ran on (needed with a LoS list); nstep: the simulator step of the detection, stored as
 * start / end.  Launches a memset and two kernels. */
int bsg_traf_events_update(const bsg_traf_events *ev, const float *d_rec, const bsg_cd_lists *lists, int64_t nstep, void *stream);

/* ---- rgb_array frames (SURVEY 8f-4) --------------------------------------------------------------------------------
 * Paints a list of draw calls into an RGB frame on the device: d_prims [n_prims][BSG_PRIM_FLOATS] float32 records
 * (type, x0, y0, x1, y1, width, colour as the bits of r | g << 8 | b << 16, unused), later records over earlier ones,
 * d_rgb [height][width][3] uint8.  LINE: (x0, y0) - (x1, y1), pixels within max(width, 1) / 2 of the segment; RING: centre
 * (x0, y0), radius x1, ring width `width` drawn inwards (0 = filled disc); RECT: filled [x0, x1) x [y0, y1); a polygon is
 * a run of EDGE records closed by one EDGE_END record, filled by the even-odd rule.
 * Replaces: the pygame draw calls of the reference's _render_frame (e.g. horizontal_cr_env.py:277-395), which only ever
 * reach a window; bluesky_gym_sasha_b200/render.py builds the list per env type. */
enum { BSG_PRIM_LINE = 1, BSG_PRIM_RING = 2, BSG_PRIM_RECT = 3, BSG_PRIM_EDGE = 4, BSG_PRIM_EDGE_END = 5, BSG_PRIM_FLOATS = 8 };
int bsg_render(const float *d_prims, int32_t n_prims, int32_t width, int32_t height, uint32_t background_rgb,
               uint8_t *d_rgb, void *stream);

/* ---- roofline denominators measured on the spot (bench.py) ------------------------------------- */
/* Dense FP32 FMA throughput [FLOP/s] of this device, timed with CUDA events. */
int bsg_probe_fp32(int32_t device, double *flops_out);

#ifdef __cplusplus
}
#endif
#endif /* BSG_H_ */
