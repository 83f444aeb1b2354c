// api.cu -- the extern "C" surface of libbsg_b200.so declared in include/bsg.h (handles, layout,
// bind/reset/step plumbing, error strings, the FP32 peak probe).  No compute happens on the host and
// there is no CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <new>
#include <string.h>

#include "env_kernels.cuh"

int bsg_launch_env(const bsg::EnvParams& P, int slots, cudaStream_t st);   // env_step.cu
int bsg_upload_tas150_table(const double* h_tab);   // env_step.cu
int bsg_launch_obs_noise(const bsg::EnvParams& P, float sigma, uint32_t call, bool with_final, cudaStream_t st);   // obs_noise.cu
namespace bsg { void host_copy_mt(void* dst, const void* src, size_t n, bool widen = false); void host_pool_prewake(); }   // host_pool.cu

static thread_local char g_err[512] = "";

int bsg_fail(int code, const char* msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}
int bsg_cuda_check(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return BSG_OK;
    snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return BSG_ECUDA;
}

// Entry points run on the handle's device and leave the caller's current device as they found it.
struct DeviceGuard {
    int prev = -1, dev;
    explicit DeviceGuard(int d) : dev(d) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
};

struct bsg_handle {
    bsg_config cfg;
    bsg_layout lay;
    bsg_tensor_table t;
    bool bound;
    bsg::EnvParams P;
    cudaEvent_t ev[4];      // chunk-arrival events of bsg_step_host_copy (created on first use)
    bool have_ev;
    bool pending;           // a bsg_step_host_begin without its bsg_step_host_wait
    int fc_slot;            // final_count slot of the last step launch (two counters take turns, see env_kernel)
    float obs_noise;        // NoisyObservationWrapper sigma (0 = off)
    uint32_t noise_calls;   // reset / step calls so far: the noise stream's call index
};

extern "C" int bsg_abi_version(void) { return BSG_ABI_VERSION; }
extern "C" int bsg_abi_struct_size(int which) {
    switch (which) {
        case 0: return (int)sizeof(bsg_config);
        case 1: return (int)sizeof(bsg_layout);
        case 2: return (int)sizeof(bsg_tensor_table);
        case 3: return (int)sizeof(bsg_wind);
        case 4: return (int)sizeof(bsg_perf);
        case 5: return (int)sizeof(bsg_ac_state);
        case 6: return (int)sizeof(bsg_cd_lists);
        case 7: return (int)sizeof(bsg_traf_config);
        case 8: return (int)sizeof(bsg_traf_tensors);
        case 9: return (int)sizeof(bsg_traf_events);
    }
    return -1;
}
extern "C" const char* bsg_last_error(void) { return g_err; }
extern "C" int bsg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static int pow2_slots(int n) { return n <= 1 ? 1 : (n <= 8 ? 8 : (n <= 16 ? 16 : 32)); }

extern "C" int bsg_query_layout(const bsg_config* cfg, bsg_layout* out) {
    if (!cfg || !out) return bsg_fail(BSG_EINVAL, "bsg_query_layout: null argument");
    if (cfg->num_envs < 0) return bsg_fail(BSG_EINVAL, "num_envs must be >= 0");
    memset(out, 0, sizeof(*out));
    out->info_dim = 6;
    out->env_f64 = BSG_F64_COUNT; out->env_f32 = BSG_F32_COUNT; out->env_i32 = BSG_I32_COUNT;
    switch (cfg->env_type) {
        case BSG_ENV_DESCENT:            // descent_env.py:29,53-62,72
            out->slots = 1; out->obs_dim = 4; out->act_dim = 1; out->n_sub = 30; out->simdt = 1.0f; break;
        case BSG_ENV_HORIZONTAL_CR: {    // horizontal_cr_env.py:17,30,49-62,72
            if (cfg->n_intruders < 1 || cfg->n_intruders > 31)
                return bsg_fail(BSG_EINVAL, "HorizontalCR: n_intruders must be in [1, 31]");
            out->slots = pow2_slots(cfg->n_intruders + 1);
            out->obs_dim = 5 * cfg->n_intruders + 3; out->act_dim = 1; out->n_sub = 10; out->simdt = 5.0f; break;
        }
        case BSG_ENV_SECTOR_CR:          // sector_cr_env.py:32,52-67,77
            out->slots = 32; out->obs_dim = 3 + 7 * 4; out->act_dim = 2; out->n_sub = 5; out->simdt = 1.0f;
            out->poly_f64 = 64; break;
        case BSG_ENV_MERGE:              // merge_env.py:34-36,59-76,86
            out->slots = 32; out->obs_dim = 5 + 7 * 5; out->act_dim = 2; out->n_sub = 10; out->simdt = 5.0f; break;
        case BSG_ENV_PLAN_WAYPOINT:      // plan_waypoint_env.py:15,22,49-58,69
            out->slots = 1; out->obs_dim = 20; out->act_dim = 1; out->n_sub = 10; out->simdt = 1.0f; break;
        case BSG_ENV_VERTICAL_CR:        // vertical_cr_env.py:40,42,64-82,95
            out->slots = 8; out->obs_dim = 4 + 7 * 5; out->act_dim = 1; out->n_sub = 30; out->simdt = 1.0f; break;
        case BSG_ENV_STATIC_OBSTACLE:    // static_obstacle_env.py:31,33,45-55,83
            out->slots = 16; out->obs_dim = 3 + 4 * 10; out->act_dim = 2; out->n_sub = 10; out->simdt = 1.0f;
            out->poly_f64 = 360; break;
        default:
            return bsg_fail(BSG_EINVAL, "unknown env_type");
    }
    if (cfg->wind_obs) out->obs_dim += 2;        // wrappers/wind.py:17-23: wind_u, wind_v appended
    return BSG_OK;
}

extern "C" int bsg_create(const bsg_config* cfg, bsg_handle** out) {
    if (!cfg || !out) return bsg_fail(BSG_EINVAL, "bsg_create: null argument");
    bsg_layout lay;
    int rc = bsg_query_layout(cfg, &lay);
    if (rc != BSG_OK) return rc;
    if (cfg->autoreset_mode < 0 || cfg->autoreset_mode > 2) return bsg_fail(BSG_EINVAL, "bad autoreset_mode");
    if (cfg->cd_pair_cap < 0) return bsg_fail(BSG_EINVAL, "cd_pair_cap must be >= 0");
    if ((long long)cfg->num_envs * lay.slots > 0x7fffff00LL) return bsg_fail(BSG_EINVAL, "num_envs * slots exceeds the 32-bit thread index");
    int ndev = bsg_device_count();
    if (ndev <= 0) return bsg_fail(BSG_ECUDA, "no CUDA device: libbsg_b200 has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) return bsg_fail(BSG_EINVAL, "device ordinal out of range");
    bsg_handle* h = new (std::nothrow) bsg_handle;
    if (!h) return bsg_fail(BSG_ENOMEM, "out of host memory");
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg;
    h->lay = lay;
    bsg::EnvParams& P = h->P;
    P.env_type = cfg->env_type; P.E = cfg->num_envs; P.n_int = cfg->n_intruders; P.cd_enabled = cfg->cd_enabled;
    P.autoreset = cfg->autoreset_mode; P.max_steps = cfg->max_episode_steps; P.hdg_random = cfg->default_hdg_random;
    P.n_sub = lay.n_sub; P.simdt = lay.simdt;
    int rel = (int)floor(10.5 / (double)lay.simdt);          // settings.fms_dt // simdt  (core/simtime.py Timer)
    P.fms_rel_freq = rel < 1 ? 1 : rel;
    P.obs_dim = lay.obs_dim; P.act_dim = lay.act_dim; P.info_dim = lay.info_dim; P.wind_obs = cfg->wind_obs; P.sector_uniform = cfg->sector_density_uniform;
    float rpz = cfg->rpz > 0.0f ? cfg->rpz : 5.0f * 1852.0f;
    P.R2 = rpz * rpz;
    P.rpz = rpz;
    P.init_alt = cfg->init_alt;
    {   // TAS every aircraft of the scenario generator is created with -- vcas2tas(cas, alt) of bluesky/tools/aero.py as
        // restated in oracle/aero.py -- for the envs that create them at a fixed altitude and speed: evaluated once, here
        double hh = (double)cfg->init_alt, cas = 150.0;              // HorizontalCR (horizontal_cr_env.py:91; init_alt: 0)
        switch (cfg->env_type) {
            case BSG_ENV_SECTOR_CR: case BSG_ENV_STATIC_OBSTACLE: hh = 350.0; break;     // sector_cr_env.py:211, static_obstacle_env.py:106
            case BSG_ENV_MERGE: hh = 10000.0; cas = 100.0; break;                        // merge_env.py:119
            case BSG_ENV_PLAN_WAYPOINT: hh = 0.0; break;                                 // plan_waypoint_env.py:162
            default: break;
        }
        const double T = fmax(288.15 - 0.0065 * hh, 216.65);
        const double rhotrop = 1.225 * pow(T / 288.15, 4.256848030018761);
        const double rho = rhotrop * exp(-fmax(0.0, hh - 11000.0) / 6341.552161), p = rho * 287.05287 * T;
        const double q = 101325.0 * (pow(1.0 + 1.225 * cas * cas / (7.0 * 101325.0), 3.5) - 1.0);
        P.init_tas0 = sqrt(7.0 * p / rho * (pow(q / p + 1.0, 2.0 / 7.0) - 1.0));
    }
    if (cfg->env_type == BSG_ENV_DESCENT || cfg->env_type == BSG_ENV_VERTICAL_CR) {
        // descent_env.py:165,173 / vertical_cr_env.py:263,270: alt_init = randint(2000, 4000), cre(..., acspd=150): the TAS for
        // every altitude the generator can draw, in float64, for this device's copy of the table
        static double tab[2001];
        const double q = 101325.0 * (pow(1.0 + 1.225 * 150.0 * 150.0 / (7.0 * 101325.0), 3.5) - 1.0);
        for (int k = 0; k <= 2000; ++k) {
            const double hh = 2000.0 + k, T = fmax(288.15 - 0.0065 * hh, 216.65);
            const double rho = 1.225 * pow(T / 288.15, 4.256848030018761), p = rho * 287.05287 * T;
            tab[k] = sqrt(7.0 * p / rho * (pow(q / p + 1.0, 2.0 / 7.0) - 1.0));
        }
        DeviceGuard guard(cfg->device);
        const int rc2 = bsg_upload_tas150_table(tab);
        if (rc2 != BSG_OK) { delete h; return rc2; }
    }
    P.hpz = cfg->hpz > 0.0f ? cfg->hpz : 1000.0f * 0.3048f;
    P.dtlook = cfg->dtlookahead > 0.0f ? cfg->dtlookahead : 300.0f;
    P.seed = cfg->seed; P.gid0 = cfg->env_id_offset; P.perf = cfg->perf;
    P.inv_axmax_gd = 1.0f / cfg->perf.axmax_gd; P.inv_axmax_air = 1.0f / cfg->perf.axmax_air;
    {   // merge_env.py:43-46: FIX = get_point_at_distance(RWY, 200 km, bearing 0)
        const double d2r = 0.017453292519943295;
        double la = bsg::kRwyLat * d2r, lo = bsg::kRwyLon * d2r, ang = 200.0 / 6371.0;
        double l2 = asin(sin(la) * cos(ang) + cos(la) * sin(ang));
        double o2 = lo + atan2(0.0, cos(ang) - sin(la) * sin(l2));
        P.fix_lat = l2 / d2r; P.fix_lon = o2 / d2r;
    }
    *out = h;
    return BSG_OK;
}

extern "C" void bsg_destroy(bsg_handle* h) {
    if (!h) return;
    if (h->have_ev) {
        cudaSetDevice(h->cfg.device);
        for (int k = 0; k < 4; ++k) cudaEventDestroy(h->ev[k]);
    }
    delete h;
}

extern "C" int bsg_bind_state(bsg_handle* h, const bsg_tensor_table* t) {
    if (!h || !t) return bsg_fail(BSG_EINVAL, "bsg_bind_state: null argument");
    if (!t->pos || !t->kin || !t->cmd || !t->aux || !t->flags || !t->env_f64 || !t->env_f32 || !t->env_i32 ||
        !t->obs || !t->reward || !t->terminated || !t->truncated || !t->info)
        return bsg_fail(BSG_EINVAL, "bsg_bind_state: a required tensor pointer is null");
    if (h->cfg.cd_enabled && (!t->tcpamax || !t->inconf)) return bsg_fail(BSG_EINVAL, "cd_enabled needs tcpamax and inconf");
    if (h->lay.poly_f64 && !t->poly) return bsg_fail(BSG_EINVAL, "this env type needs the poly tensor");
    if (t->final_obs && (!t->final_ids || !t->final_count)) return bsg_fail(BSG_EINVAL, "final_obs needs final_ids and final_count");
    h->t = *t;
    bsg::EnvParams& P = h->P;
    P.pos = (double2*)t->pos; P.kin = (float4*)t->kin; P.cmd = (float4*)t->cmd; P.aux = (float4*)t->aux;
    P.flags = t->flags; P.tcpamax = t->tcpamax; P.inconf = t->inconf;
    P.ef64 = t->env_f64; P.ef32 = t->env_f32; P.ei32 = t->env_i32; P.poly = t->poly;
    P.obs = t->obs; P.final_obs = t->final_obs; P.final_ids = t->final_ids; P.final_count = t->final_count; P.reward = t->reward; P.term = t->terminated; P.trunc = t->truncated;
    P.info = t->info;
    if (h->cfg.cd_pair_cap > 0 && h->cfg.cd_enabled && !t->cd_pairs) return bsg_fail(BSG_EINVAL, "cd_pair_cap > 0 needs tensor_table.cd_pairs");
    P.cd_pairs = (h->cfg.cd_pair_cap > 0 && h->cfg.cd_enabled) ? t->cd_pairs : nullptr;
    P.cd_attr = P.cd_pairs ? t->cd_attr : nullptr;
    P.cd_pair_cap = h->cfg.cd_pair_cap;
    h->bound = true;
    return BSG_OK;
}

static int run_mode(bsg_handle* h, int mode, const float* d_actions, const uint8_t* d_mask, int n_sub, void* stream) {
    if (!h) return bsg_fail(BSG_EINVAL, "null handle");
    if (!h->bound) return bsg_fail(BSG_ESTATE, "bsg_bind_state has not been called");
    DeviceGuard guard(h->cfg.device);
    bsg::EnvParams P = h->P;
    P.mode = mode; P.actions = d_actions; P.reset_mask = d_mask;
    if (n_sub > 0) P.n_sub = n_sub;
    if (mode == bsg::kModeStep) h->fc_slot ^= 1;
    P.fc_slot = h->fc_slot;
    int rc = bsg_launch_env(P, h->lay.slots, (cudaStream_t)stream);
    if (rc != BSG_OK || mode == bsg::kModeTraf || !(h->obs_noise > 0.0f)) return rc;
    return bsg_launch_obs_noise(P, h->obs_noise, h->noise_calls++, mode == bsg::kModeStep, (cudaStream_t)stream);
}

extern "C" int bsg_set_seed(bsg_handle* h, uint64_t seed) {
    if (!h) return bsg_fail(BSG_EINVAL, "null handle");
    h->cfg.seed = seed;
    h->P.seed = seed;
    return BSG_OK;
}

extern "C" int bsg_set_wind(bsg_handle* h, const bsg_wind* w) {
    if (!h) return bsg_fail(BSG_EINVAL, "null handle");
    bsg::EnvParams& P = h->P;
    if (!w || w->n_points == 0) {
        P.wind_n = 0; P.wind_nalt = 0; P.wind_lat = P.wind_lon = P.wind_vn = P.wind_ve = nullptr; P.gsv = nullptr;
        return BSG_OK;
    }
    if (w->n_points < 0 || w->n_points > 64) return bsg_fail(BSG_EINVAL, "bsg_set_wind: n_points must be in [0, 64]");
    if (w->n_alt < 1 || (w->n_alt > 1 && !(w->alt_step > 0.0f))) return bsg_fail(BSG_EINVAL, "bsg_set_wind: bad altitude axis");
    if (!w->d_lat || !w->d_lon || !w->d_vn || !w->d_ve || !w->d_gs) return bsg_fail(BSG_EINVAL, "bsg_set_wind: null pointer");
    P.wind_n = w->n_points; P.wind_nalt = w->n_alt; P.wind_altstep = w->alt_step;
    P.wind_lat = w->d_lat; P.wind_lon = w->d_lon; P.wind_vn = w->d_vn; P.wind_ve = w->d_ve;
    P.gsv = (float2*)w->d_gs;
    return BSG_OK;
}

extern "C" int bsg_set_obs_noise(bsg_handle* h, float sigma) {
    if (!h) return bsg_fail(BSG_EINVAL, "null handle");
    if (!(sigma >= 0.0f)) return bsg_fail(BSG_EINVAL, "bsg_set_obs_noise: noise level must be >= 0");
    h->obs_noise = sigma;
    return BSG_OK;
}

extern "C" int bsg_get_noise_calls(bsg_handle* h, uint32_t* out) {
    if (!h || !out) return bsg_fail(BSG_EINVAL, "bsg_get_noise_calls: null argument");
    *out = h->noise_calls;
    return BSG_OK;
}
extern "C" int bsg_set_noise_calls(bsg_handle* h, uint32_t calls) {
    if (!h) return bsg_fail(BSG_EINVAL, "null handle");
    h->noise_calls = calls;
    return BSG_OK;
}

extern "C" int bsg_load_state(bsg_handle* h, int32_t env, const bsg_ac_state* s, void* stream) {
    if (!h || !s) return bsg_fail(BSG_EINVAL, "bsg_load_state: null argument");
    if (!h->bound) return bsg_fail(BSG_ESTATE, "bsg_bind_state has not been called");
    const int G = h->lay.slots, n = s->n;
    if (env < 0 || env >= h->cfg.num_envs) return bsg_fail(BSG_EINVAL, "bsg_load_state: env index out of range");
    if (n < 0 || n > G) return bsg_fail(BSG_EINVAL, "bsg_load_state: more aircraft than slots");
    if (n > 0 && (!s->lat || !s->lon || !s->alt || !s->tas || !s->hdg || !s->vs || !s->selspd || !s->selalt || !s->selvs ||
                  !s->ap_trk || !s->cas))
        return bsg_fail(BSG_EINVAL, "bsg_load_state: a required aircraft array is null");
    cudaStream_t st = (cudaStream_t)stream;
    DeviceGuard guard(h->cfg.device);
    double pos[32 * 2];
    float kin[32 * 4], cmd[32 * 4], aux[32 * 4];
    uint32_t fl[32];
    memset(pos, 0, sizeof(pos)); memset(kin, 0, sizeof(kin)); memset(cmd, 0, sizeof(cmd)); memset(aux, 0, sizeof(aux));
    memset(fl, 0, sizeof(fl));
    for (int i = 0; i < n; ++i) {
        pos[2 * i] = s->lat[i]; pos[2 * i + 1] = s->lon[i];
        kin[4 * i] = (float)s->alt[i]; kin[4 * i + 1] = (float)s->tas[i]; kin[4 * i + 2] = (float)s->hdg[i]; kin[4 * i + 3] = (float)s->vs[i];
        cmd[4 * i] = (float)s->selspd[i]; cmd[4 * i + 1] = (float)s->selalt[i]; cmd[4 * i + 2] = (float)s->selvs[i]; cmd[4 * i + 3] = (float)s->ap_trk[i];
        aux[4 * i] = s->ax ? (float)s->ax[i] : 0.0f;
        aux[4 * i + 1] = s->curlegdir ? (float)s->curlegdir[i] : -999.0f;
        aux[4 * i + 2] = (float)s->cas[i];
        uint32_t f = bsg::kFlAlive;
        if (s->swlnav && s->swlnav[i]) f |= bsg::kFlLnav;
        if (s->iactwp) {
            const int ia = s->iactwp[i] > 0 ? s->iactwp[i] : 0;
            f |= ((uint32_t)ia << bsg::kFlWpShift) | (ia >= 1 ? bsg::kFlLastWp : 0u);
        }
        fl[i] = f;
    }
    const size_t o = (size_t)env * G;
    BSG_CUDA(cudaMemcpyAsync(h->t.pos + 2 * o, pos, sizeof(double) * 2 * G, cudaMemcpyHostToDevice, st));
    BSG_CUDA(cudaMemcpyAsync(h->t.kin + 4 * o, kin, sizeof(float) * 4 * G, cudaMemcpyHostToDevice, st));
    BSG_CUDA(cudaMemcpyAsync(h->t.cmd + 4 * o, cmd, sizeof(float) * 4 * G, cudaMemcpyHostToDevice, st));
    BSG_CUDA(cudaMemcpyAsync(h->t.aux + 4 * o, aux, sizeof(float) * 4 * G, cudaMemcpyHostToDevice, st));
    BSG_CUDA(cudaMemcpyAsync(h->t.flags + o, fl, sizeof(uint32_t) * G, cudaMemcpyHostToDevice, st));
    if (s->env_f64) BSG_CUDA(cudaMemcpyAsync(h->t.env_f64 + (size_t)env * h->lay.env_f64, s->env_f64, sizeof(double) * h->lay.env_f64, cudaMemcpyHostToDevice, st));
    if (s->env_f32) BSG_CUDA(cudaMemcpyAsync(h->t.env_f32 + (size_t)env * h->lay.env_f32, s->env_f32, sizeof(float) * h->lay.env_f32, cudaMemcpyHostToDevice, st));
    if (s->env_i32) BSG_CUDA(cudaMemcpyAsync(h->t.env_i32 + (size_t)env * h->lay.env_i32, s->env_i32, sizeof(int32_t) * h->lay.env_i32, cudaMemcpyHostToDevice, st));
    if (s->poly) {
        if (!h->lay.poly_f64 || !h->t.poly) return bsg_fail(BSG_EINVAL, "bsg_load_state: this env type has no polygon record");
        BSG_CUDA(cudaMemcpyAsync(h->t.poly + (size_t)env * h->lay.poly_f64, s->poly, sizeof(double) * h->lay.poly_f64, cudaMemcpyHostToDevice, st));
    }
    BSG_CUDA(cudaStreamSynchronize(st));         // the staging arrays above live on this stack frame
    return BSG_OK;
}

extern "C" int bsg_reset(bsg_handle* h, const uint8_t* d_mask, void* stream) {
    return run_mode(h, bsg::kModeReset, nullptr, d_mask, 0, stream);
}
extern "C" int bsg_step(bsg_handle* h, const float* d_actions, void* stream) {
    if (!d_actions) return bsg_fail(BSG_EINVAL, "bsg_step: null actions");
    return run_mode(h, bsg::kModeStep, d_actions, nullptr, 0, stream);
}
extern "C" int bsg_traf_update(bsg_handle* h, int32_t n_sub, void* stream) {
    if (n_sub < 0) return bsg_fail(BSG_EINVAL, "bsg_traf_update: n_sub < 0");
    if (n_sub == 0) return BSG_OK;
    return run_mode(h, bsg::kModeTraf, nullptr, nullptr, n_sub, stream);
}

extern "C" int bsg_step_host(bsg_handle* h, const float* h_actions, float* h_obs, float* h_reward,
                             uint8_t* h_terminated, uint8_t* h_truncated, float* h_info, int32_t* h_final_count,
                             void* stream) {
    if (!h || !h_actions) return bsg_fail(BSG_EINVAL, "bsg_step_host: null argument");
    if (!h->bound) return bsg_fail(BSG_ESTATE, "bsg_bind_state has not been called");
    if (!h->t.actions_staging) return bsg_fail(BSG_ESTATE, "bsg_step_host needs tensor_table.actions_staging");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t E = (size_t)h->cfg.num_envs;
    DeviceGuard guard(h->cfg.device);
    BSG_CUDA(cudaMemcpyAsync(h->t.actions_staging, h_actions, E * h->lay.act_dim * sizeof(float), cudaMemcpyHostToDevice, st));
    int rc = run_mode(h, bsg::kModeStep, h->t.actions_staging, nullptr, 0, stream);
    if (rc != BSG_OK) return rc;
    // Outputs that are laid out in ONE contiguous block on the device (obs | reward | info | final_count[4] |
    // terminated | truncated, as BlueSkyVectorEnv allocates them) and mirrored with the same offsets on
    // the host go back in a single copy instead of six.
    {
        const char* d0 = (const char*)h->t.obs;
        char* h0 = (char*)h_obs;
        const size_t n_obs = E * h->lay.obs_dim * sizeof(float), n_rew = E * sizeof(float);
        const size_t n_info = E * h->lay.info_dim * sizeof(float), n_cnt = 4 * sizeof(int32_t);
        const size_t o_rew = n_obs, o_info = o_rew + n_rew, o_cnt = o_info + n_info, o_term = o_cnt + n_cnt, o_trunc = o_term + E;
        const bool packed = h_obs && h_reward && h_info && h_terminated && h_truncated && h_final_count &&
                            (const char*)h->t.reward == d0 + o_rew && (char*)h_reward == h0 + o_rew &&
                            (const char*)h->t.info == d0 + o_info && (char*)h_info == h0 + o_info &&
                            (const char*)h->t.final_count == d0 + o_cnt && (char*)h_final_count == h0 + o_cnt &&
                            (const char*)h->t.terminated == d0 + o_term && (char*)h_terminated == h0 + o_term &&
                            (const char*)h->t.truncated == d0 + o_trunc && (char*)h_truncated == h0 + o_trunc;
        if (packed) {
            BSG_CUDA(cudaMemcpyAsync(h0, d0, o_trunc + E, cudaMemcpyDeviceToHost, st));
        } else {
            if (h_obs) BSG_CUDA(cudaMemcpyAsync(h_obs, h->t.obs, n_obs, cudaMemcpyDeviceToHost, st));
            if (h_reward) BSG_CUDA(cudaMemcpyAsync(h_reward, h->t.reward, n_rew, cudaMemcpyDeviceToHost, st));
            if (h_terminated) BSG_CUDA(cudaMemcpyAsync(h_terminated, h->t.terminated, E, cudaMemcpyDeviceToHost, st));
            if (h_truncated) BSG_CUDA(cudaMemcpyAsync(h_truncated, h->t.truncated, E, cudaMemcpyDeviceToHost, st));
            if (h_info) BSG_CUDA(cudaMemcpyAsync(h_info, h->t.info, n_info, cudaMemcpyDeviceToHost, st));
            if (h_final_count && h->t.final_count)
                BSG_CUDA(cudaMemcpyAsync(h_final_count, h->t.final_count + h->fc_slot, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        }
    }
    BSG_CUDA(cudaStreamSynchronize(st));
    return BSG_OK;
}

// Single-mirror form: the caller laid the step outputs out as ONE contiguous device block starting at
// tensor_table.obs (obs | reward | info | final_count[4] | terminated | truncated | pad | final_ids |
// final_obs rows ...) and mirrors its first `nbytes` bytes in pinned host memory.  One H2D copy, one
// launch, one D2H copy, one synchronise per env step.
extern "C" int bsg_step_host_block(bsg_handle* h, const float* h_actions, void* h_block, size_t nbytes, void* stream) {
    if (!h || !h_actions || !h_block) return bsg_fail(BSG_EINVAL, "bsg_step_host_block: null argument");
    if (!h->bound) return bsg_fail(BSG_ESTATE, "bsg_bind_state has not been called");
    if (!h->t.actions_staging) return bsg_fail(BSG_ESTATE, "bsg_step_host_block needs tensor_table.actions_staging");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t E = (size_t)h->cfg.num_envs;
    DeviceGuard guard(h->cfg.device);
    BSG_CUDA(cudaMemcpyAsync(h->t.actions_staging, h_actions, E * h->lay.act_dim * sizeof(float), cudaMemcpyHostToDevice, st));
    int rc = run_mode(h, bsg::kModeStep, h->t.actions_staging, nullptr, 0, stream);
    if (rc != BSG_OK) return rc;
    BSG_CUDA(cudaMemcpyAsync(h_block, h->t.obs, nbytes, cudaMemcpyDeviceToHost, st));
    BSG_CUDA(cudaStreamSynchronize(st));
    return BSG_OK;
}

// bsg_step_host_block + the copy of the block's first `dst_bytes` bytes (the observations) into the caller's
// own result array, pipelined: the device->host transfer is issued in chunks, and while chunk k+1 is still
// crossing PCIe the host threads (host_pool.cu) move chunk k from the pinned mirror into `dst`.
extern "C" int bsg_step_host_copy(bsg_handle* h, const float* h_actions, void* h_block, size_t nbytes,
                                  void* dst, size_t dst_bytes, void* stream) {
    if (!h || !h_actions || !h_block) return bsg_fail(BSG_EINVAL, "bsg_step_host_copy: null argument");
    if (!h->bound) return bsg_fail(BSG_ESTATE, "bsg_bind_state has not been called");
    if (!h->t.actions_staging) return bsg_fail(BSG_ESTATE, "bsg_step_host_copy needs tensor_table.actions_staging");
    if (dst_bytes > nbytes) return bsg_fail(BSG_EINVAL, "bsg_step_host_copy: dst_bytes exceeds the mirrored block");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t E = (size_t)h->cfg.num_envs;
    DeviceGuard guard(h->cfg.device);
    if (!h->have_ev) {
        for (int k = 0; k < 4; ++k) BSG_CUDA(cudaEventCreateWithFlags(&h->ev[k], cudaEventDisableTiming));
        h->have_ev = true;
    }
    BSG_CUDA(cudaMemcpyAsync(h->t.actions_staging, h_actions, E * h->lay.act_dim * sizeof(float), cudaMemcpyHostToDevice, st));
    int rc = run_mode(h, bsg::kModeStep, h->t.actions_staging, nullptr, 0, stream);
    if (rc != BSG_OK) return rc;
    const char* d0 = (const char*)h->t.obs;
    char* h0 = (char*)h_block;
    if (dst) bsg::host_pool_prewake();     // the copy threads wake up while the GPU is busy
    // chunks: small transfers go in one piece; otherwise 2 pieces of the copied region, the tail with the last
    // (1, 2 and 4 pieces measured equal once the copy threads are pre-woken: DESIGN §4)
    const int nchunk = (dst && dst_bytes >= (512u << 10)) ? 2 : 1;
    size_t bounds[3];
    for (int k = 0; k <= nchunk; ++k) bounds[k] = (dst_bytes * k / nchunk) & ~(size_t)255;
    bounds[0] = 0;
    bounds[nchunk] = nbytes;
    for (int k = 0; k < nchunk; ++k) {
        BSG_CUDA(cudaMemcpyAsync(h0 + bounds[k], d0 + bounds[k], bounds[k + 1] - bounds[k], cudaMemcpyDeviceToHost, st));
        BSG_CUDA(cudaEventRecord(h->ev[k], st));
    }
    for (int k = 0; k < nchunk; ++k) {
        BSG_CUDA(cudaEventSynchronize(h->ev[k]));
        if (dst) {
            size_t lo = bounds[k], hi = bounds[k + 1] < dst_bytes ? bounds[k + 1] : dst_bytes;
            if (hi > lo) bsg::host_copy_mt((char*)dst + lo, h0 + lo, hi - lo);
        }
    }
    return BSG_OK;
}

extern "C" int bsg_step_host_begin(bsg_handle* h, const float* h_actions, void* h_block, size_t nbytes, void* stream) {
    if (!h || !h_actions || !h_block) return bsg_fail(BSG_EINVAL, "bsg_step_host_begin: null argument");
    if (!h->bound) return bsg_fail(BSG_ESTATE, "bsg_bind_state has not been called");
    if (!h->t.actions_staging) return bsg_fail(BSG_ESTATE, "bsg_step_host_begin needs tensor_table.actions_staging");
    if (h->pending) return bsg_fail(BSG_ESTATE, "bsg_step_host_begin: the previous step has not been waited for");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t E = (size_t)h->cfg.num_envs;
    DeviceGuard guard(h->cfg.device);
    if (!h->have_ev) {
        for (int k = 0; k < 4; ++k) BSG_CUDA(cudaEventCreateWithFlags(&h->ev[k], cudaEventDisableTiming));
        h->have_ev = true;
    }
    BSG_CUDA(cudaMemcpyAsync(h->t.actions_staging, h_actions, E * h->lay.act_dim * sizeof(float), cudaMemcpyHostToDevice, st));
    int rc = run_mode(h, bsg::kModeStep, h->t.actions_staging, nullptr, 0, stream);
    if (rc != BSG_OK) return rc;
    BSG_CUDA(cudaMemcpyAsync(h_block, h->t.obs, nbytes, cudaMemcpyDeviceToHost, st));
    BSG_CUDA(cudaEventRecord(h->ev[0], st));
    h->pending = true;
    return BSG_OK;
}

extern "C" int bsg_step_host_wait(bsg_handle* h, const void* h_block, void* dst, size_t dst_bytes) {
    if (!h) return bsg_fail(BSG_EINVAL, "bsg_step_host_wait: null handle");
    if (!h->pending) return bsg_fail(BSG_ESTATE, "bsg_step_host_wait without bsg_step_host_begin");
    if (dst && !h_block) return bsg_fail(BSG_EINVAL, "bsg_step_host_wait: null block");
    DeviceGuard guard(h->cfg.device);
    if (dst) bsg::host_pool_prewake();
    h->pending = false;
    BSG_CUDA(cudaEventSynchronize(h->ev[0]));
    if (dst && dst_bytes) bsg::host_copy_mt((char*)dst, (const char*)h_block, dst_bytes);
    return BSG_OK;
}

extern "C" int bsg_host_copy(void* dst, const void* src, size_t nbytes) {
    if ((!dst || !src) && nbytes) return bsg_fail(BSG_EINVAL, "bsg_host_copy: null argument");
    bsg::host_pool_prewake();
    bsg::host_copy_mt(dst, src, nbytes);
    return BSG_OK;
}

extern "C" int bsg_host_widen(double* dst, const float* src, size_t n) {
    if ((!dst || !src) && n) return bsg_fail(BSG_EINVAL, "bsg_host_widen: null argument");
    bsg::host_pool_prewake();
    bsg::host_copy_mt(dst, src, n * sizeof(float), true);
    return BSG_OK;
}

// ---- FP32 FMA peak probe (roofline denominator for the CD kernels; SURVEY.md section 6) -------------
__global__ void __launch_bounds__(256) fma_probe_kernel(float* out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.0f, a2 = a0 + 2.0f, a3 = a0 + 3.0f;
    float a4 = a0 + 4.0f, a5 = a0 + 5.0f, a6 = a0 + 6.0f, a7 = a0 + 7.0f;
    const float m = 0.999f + blockIdx.x * 1e-9f, c = 1e-3f * (threadIdx.x & 3);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
            a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
        }
    }
    float r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (r == 123.456f) out[0] = r;        // never true; keeps the chain alive
}

extern "C" int bsg_probe_fp32(int32_t device, double* flops_out) {
    if (!flops_out) return bsg_fail(BSG_EINVAL, "bsg_probe_fp32: null output");
    if (bsg_device_count() <= 0) return bsg_fail(BSG_ECUDA, "no CUDA device");
    BSG_CUDA(cudaSetDevice(device));
    int sms = 0;
    BSG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    float* d = nullptr;
    BSG_CUDA(cudaMalloc(&d, 256));
    cudaEvent_t e0, e1;
    BSG_CUDA(cudaEventCreate(&e0));
    BSG_CUDA(cudaEventCreate(&e1));
    const int iters = 4096, blocks = sms * 8;
    fma_probe_kernel<<<blocks, 256>>>(d, 64);           // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        fma_probe_kernel<<<blocks, 256>>>(d, iters);
        cudaEventRecord(e1);
        BSG_CUDA(cudaEventSynchronize(e1));
        float ms = 0.0f;
        cudaEventElapsedTime(&ms, e0, e1);
        double fl = 2.0 * 8.0 * 16.0 * (double)iters * 256.0 * (double)blocks / (ms * 1e-3);
        if (fl > best) best = fl;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *flops_out = best;
    return BSG_OK;
}
