// C ABI of libjiminy_b200.so (declared in include/jiminy_b200.h): batch life-cycle, uploads,
// kernel launches and env-major host views.  No CPU compute path exists: every entry point that
// needs the device fails with JB_ERR_CUDA when CUDA is unavailable.
#ifndef JB_HOST_EMUL
#include <cuda_runtime.h>
#endif

#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <random>
#include <string>
#include <vector>

#include "../../include/jiminy_b200.h"
#include "jb_kernel.cuh"
#include "jb_plan.h"

using namespace jb;

#ifndef JB_HOST_EMUL
#define JB_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif

#ifdef JB_HOST_EMUL
namespace jb { KParams g_kp_host; }
#else
static std::mutex g_launch_mutex;
static cudaEvent_t g_last_launch[64] = {};
#endif
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return fail(JB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));  \
    } while (0)

struct JbBatch {
    int device = 0;
    int n_env = 0, n_pad = 0;
    Plan plan;
    KParams kp{};
    cudaStream_t stream = nullptr;
    int nq = 0, nv = 0, nmotors = 0, njoints = 0, width = 0;
    std::vector<double> q_lower, q_upper;
    std::vector<void*> allocs;
    // device buffers
    double *d_q = nullptr, *d_v = nullptr, *d_a = nullptr, *d_sched = nullptr;
    long long* d_iters = nullptr;
    int32_t* d_status = nullptr;
    double *d_cmd = nullptr, *d_sensors = nullptr, *d_qv = nullptr;
    // jb_state_ptrs: pinned host mirrors refreshed behind every start / step launch (stable addresses, zero-copy views)
    double *h_mirror = nullptr, *hm_t = nullptr, *hm_qv = nullptr, *hm_a = nullptr, *hm_sensors = nullptr, *d_a_aos = nullptr;
    double *d_qin = nullptr, *d_vin = nullptr, *d_aout = nullptr, *d_fext = nullptr, *d_u = nullptr, *d_umotor = nullptr;
    double* d_springs = nullptr;
    double *d_pd = nullptr, *d_cmd_torque = nullptr, *d_pdf = nullptr, *d_pdf_state = nullptr, *d_mahony = nullptr;
    double *d_pdf_snap = nullptr, *d_mahony_snap = nullptr;
    // sensor measurement pipeline (jb_set_sensor_options / jb_set_seeds)
    std::vector<SensorDesc> sdesc;
    std::vector<uint32_t> seeds;
    bool sp_dirty = false;
    int sp_cap_alloc = 0;
    SensorDesc* d_sdesc = nullptr;
    unsigned long long *d_sp_rng = nullptr, *d_sp_rng_init = nullptr, *d_sp_snap_rng = nullptr;
    int32_t *d_sp_count = nullptr, *d_sp_snap_count = nullptr;
    double *d_sp_times = nullptr, *d_sp_ring = nullptr, *d_sens_true = nullptr;
    double *d_cmd_dyn = nullptr, *d_cstate_save = nullptr;   // jb_compute_dynamics: command of the evaluation, saved constraint state
    int nimu = 0;
    uint8_t* d_mask = nullptr;
    double* d_stage = nullptr;  // staging for SoA -> AoS getters
    // pinned host staging
    double* h_stage = nullptr;
    size_t h_stage_bytes = 0;
    int64_t launches = 0, param_uploads = 0;
    bool any_started = false;
    bool no_fast_kernel = false;   // JB_NO_FAST_KERNEL: always the full kernel (development / tests)
    size_t smem_bytes = 0;
    int base_fields = 0;           // plan fields + constraint bookkeeping, before the external-force slots
    int32_t* d_needs_full = nullptr;
    std::vector<int32_t> jc_joint;  // joint of each joint-bound constraint (constraint path)
    // observation exchange over peer memory
    int peer_world = 0, peer_rank = 0;
    char* d_peer_buf = nullptr;                 // [2][world][n_env][width] doubles, then flags [2][world] int64
    size_t peer_obs_doubles = 0;                // doubles of ONE parity buffer
    std::vector<void*> peer_opened;             // mapped buffers of the other ranks
    char* peer_base[8] = {nullptr};
    int* h_peer_timeout = nullptr;             // host-mapped: set by the wait kernel when a rank never signalled
    int* d_peer_timeout = nullptr;             // device alias of the same word
    double peer_timeout_s = 2.0;
    long long peer_timeout_cycles = 4000000000LL;
    long long step_id = 0;
    bool peer_enabled = true;                   // jb_peer_obs_enable
    // external forces: frames (slots), impulse table mirror, profile periods
    struct ExtFrame { int joint; double p[3]; };
    std::vector<ExtFrame> eframes;
    std::vector<double> h_imp;      // [MAX_IMPULSE][IMPULSE_ROWS][n_pad]
    ExtSlot* d_eslots = nullptr;
    double *d_imp = nullptr, *d_prof_pending = nullptr, *d_prof_latched = nullptr;
};

// The dynamic shared-memory opt-in is a per-function, per-device attribute: only ever raise it.
static std::mutex g_smem_mutex;
static size_t g_smem_attr[64] = {0};
static int raise_smem_attr(int device, size_t bytes) {
#ifndef JB_HOST_EMUL
    std::lock_guard<std::mutex> lock(g_smem_mutex);
    if (bytes <= g_smem_attr[device]) return JB_OK;
    cudaError_t e = cudaFuncSetAttribute(env_step_kernel_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(env_step_kernel_t<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
    if (e != cudaSuccess) return fail(JB_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    g_smem_attr[device] = bytes;
#endif
    return JB_OK;
}

// After a stream synchronisation: did a peer-exchange wait give up?  (the wait kernel writes the host-mapped word)
static int check_peer_timeout(JbBatch* b) {
    if (b->h_peer_timeout && *b->h_peer_timeout != 0) {
        const int who = *b->h_peer_timeout - 1;
        return fail(JB_ERR_PEER_TIMEOUT, "observation exchange: rank " + std::to_string(who) + " never signalled step " +
                    std::to_string(b->step_id) + " within " + std::to_string(b->peer_timeout_s) + " s (rank dead, or steps out of lockstep)");
    }
    return JB_OK;
}

template <typename T>
static int dev_alloc(JbBatch* b, T** p, size_t count) {
    void* raw = nullptr;
    CU(cudaMalloc(&raw, std::max<size_t>(count, 1) * sizeof(T)));
    CU(cudaMemsetAsync(raw, 0, std::max<size_t>(count, 1) * sizeof(T), b->stream));
    b->allocs.push_back(raw);
    *p = static_cast<T*>(raw);
    return JB_OK;
}

// SoA [k][n_pad] -> AoS [env][width]
__global__ void soa_to_aos_kernel(const double* __restrict__ in, double* __restrict__ out, int n_env, int n_pad, int width) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i >= static_cast<size_t>(n_env) * width) return;
    const size_t env = i / width, k = i % width;
    out[i] = in[k * n_pad + env];
}

// AoS [env][width] -> SoA [k][n_pad] (padding envs replicate the last one)
__global__ void aos_to_soa_kernel(const double* __restrict__ in, double* __restrict__ out, int n_env, int n_pad, int width) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i >= static_cast<size_t>(n_pad) * width) return;
    const size_t k = i / n_pad, env = i % n_pad;
    out[i] = in[(env < static_cast<size_t>(n_env) ? env : static_cast<size_t>(n_env - 1)) * width + k];
}

static int ensure_host_stage(JbBatch* b, size_t bytes) {
    if (bytes <= b->h_stage_bytes) return JB_OK;
    if (b->h_stage) cudaFreeHost(b->h_stage);
    b->h_stage = nullptr; b->h_stage_bytes = 0;
    CU(cudaMallocHost(reinterpret_cast<void**>(&b->h_stage), bytes));
    b->h_stage_bytes = bytes;
    return JB_OK;
}

// One launch of the step kernel.  The persistent parameter block lives in constant memory, one per device: it is
// re-uploaded only when it differs from what the device holds (another batch launched in between, or a setter
// changed it), ordered after every earlier launch on that device.  What changes at every launch (mode, step size,
// peer-exchange step) travels as the kernel parameter.
#ifndef JB_HOST_EMUL
static KParams g_kp_on_device[64];
static bool g_kp_valid[64] = {};
#endif
static int launch(JbBatch* b, int mode, double step_dt, const uint8_t* d_mask = nullptr, const double* d_command = nullptr) {
    KParams kp = b->kp;
    // static plan signatures carry no external-force code
    if (kp.n_eslot > 0) kp.sig_id = 0;
    LaunchArgs la{};
    la.mode = mode; la.step_dt = step_dt; la.mask = d_mask; la.command = d_command;
    if (mode == MODE_STEP && b->peer_world > 1 && !b->peer_opened.empty() && b->peer_enabled) {
        ++b->step_id;
        la.peer_on = 1;
        la.peer_parity = static_cast<int32_t>(b->step_id & 1);
        la.peer_step = b->step_id;
    }
    // the hot-path kernel hands envs that leave the hot path over to the full body inside the same launch
    const bool fast = mode == MODE_STEP && kp.n_eslot == 0 && kp.opt.contact_model == JB_CONTACT_SPRING_DAMPER &&
                      kp.opt.ode_solver != JB_SOLVER_RUNGE_KUTTA_DOPRI && !b->no_fast_kernel;
    const int epw = 32 / b->plan.L;
    const int nblocks = (b->n_env + epw - 1) / epw;
#ifdef JB_HOST_EMUL
    emul::current_L = b->plan.L;
    g_kp_host = kp;
    if (fast) JB_LAUNCH(env_step_kernel_t<true>, nblocks, 32, b->smem_bytes, b->stream, la);
    else JB_LAUNCH(env_step_kernel_t<false>, nblocks, 32, b->smem_bytes, b->stream, la);
#else
    {
        std::lock_guard<std::mutex> lock(g_launch_mutex);
        cudaEvent_t& evt = g_last_launch[b->device];
        if (!evt) CU(cudaEventCreateWithFlags(&evt, cudaEventDisableTiming));
        if (!g_kp_valid[b->device] || std::memcmp(&g_kp_on_device[b->device], &kp, sizeof kp) != 0) {
            if (g_kp_valid[b->device]) CU(cudaStreamWaitEvent(b->stream, evt, 0));
            g_kp_valid[b->device] = false;
            // (the copy is staged by the runtime before the call returns: `kp` may live on this stack)
            CU(cudaMemcpyToSymbolAsync(g_kp, &kp, sizeof kp, 0, cudaMemcpyHostToDevice, b->stream));
            std::memcpy(&g_kp_on_device[b->device], &kp, sizeof kp);
            g_kp_valid[b->device] = true;
            ++b->param_uploads;
        }
        if (fast) JB_LAUNCH(env_step_kernel_t<true>, nblocks, 32, b->smem_bytes, b->stream, la);
        else JB_LAUNCH(env_step_kernel_t<false>, nblocks, 32, b->smem_bytes, b->stream, la);
        CU(cudaEventRecord(evt, b->stream));
    }
#endif
    CU(cudaGetLastError());
    ++b->launches;
    if (b->h_mirror && (mode == MODE_STEP || mode == MODE_START)) {
        // behind the step on the same stream: the views hold the new state once the stream has been synchronised
        CU(cudaMemcpyAsync(b->hm_t, b->d_sched + static_cast<size_t>(SCH_T) * b->n_pad, sizeof(double) * b->n_env, cudaMemcpyDeviceToHost, b->stream));
        CU(cudaMemcpyAsync(b->hm_qv, b->d_qv, sizeof(double) * b->n_env * (b->nq + b->nv), cudaMemcpyDeviceToHost, b->stream));
        const size_t na = static_cast<size_t>(b->n_env) * b->nv;
        if (na) {
            JB_LAUNCH(soa_to_aos_kernel, static_cast<unsigned>((na + 255) / 256), 256, 0, b->stream, b->d_a, b->d_a_aos, b->n_env, b->n_pad, b->nv);
            CU(cudaGetLastError());
            ++b->launches;
            CU(cudaMemcpyAsync(b->hm_a, b->d_a_aos, sizeof(double) * na, cudaMemcpyDeviceToHost, b->stream));
        }
        if (b->width) CU(cudaMemcpyAsync(b->hm_sensors, b->d_sensors, sizeof(double) * b->n_env * b->width, cudaMemcpyDeviceToHost, b->stream));
    }
    return JB_OK;
}

extern "C" {

const char* jb_last_error(void) { return g_err.c_str(); }
const char* jb_version(void) { return "jiminy_b200 0.1 (sm_100a, fp64 lane-planned ABA)"; }

void jb_default_options(JbOptions* o) {
    std::memset(o, 0, sizeof *o);
    o->ode_solver = JB_SOLVER_RUNGE_KUTTA_DOPRI;
    o->successive_iter_failed_max = 1000;
    o->iter_max = 0;
    o->tol_abs = 1e-5; o->tol_rel = 1e-4; o->dt_max = 0.02; o->dt_restore_threshold_rel = 0.2;
    o->sensors_update_period = 0.0; o->controller_update_period = 0.0;
    o->contact_stiffness = 1e6; o->contact_damping = 2e3; o->contact_friction = 1.0;
    o->contact_transition_eps = 1e-3; o->contact_transition_velocity = 1e-2;
    o->gravity[2] = -9.81;
    o->contact_model = JB_CONTACT_SPRING_DAMPER;
    o->contact_torsion = 0.0; o->contact_stabilization_freq = 20.0; o->constraint_regularization = 1e-3;
}

static int check_options(const JbOptions* o) {
    if (o->contact_model != JB_CONTACT_SPRING_DAMPER && o->contact_model != JB_CONTACT_CONSTRAINT)
        return fail(JB_ERR_INVALID_ARGUMENT, "unknown contact model");
    if (o->contact_torsion < 0.0 || o->contact_stabilization_freq < 0.0 || o->constraint_regularization < 0.0)
        return fail(JB_ERR_INVALID_ARGUMENT, "contact / constraint options must be positive");
    if (o->ode_solver < JB_SOLVER_EULER_EXPLICIT || o->ode_solver > JB_SOLVER_RUNGE_KUTTA_DOPRI)
        return fail(JB_ERR_INVALID_ARGUMENT, "unknown ODE solver");
    if (!(o->dt_max >= 1e-6 - 1e-16 && o->dt_max <= 0.02 + 1e-16)) return fail(JB_ERR_INVALID_ARGUMENT, "'dtMax' option is out of range.");
    for (double p : {o->sensors_update_period, o->controller_update_period})
        if ((p > 2.3e-16 && p < 1e-6) || p > 0.02) return fail(JB_ERR_INVALID_ARGUMENT, "update period out of range");
    if (o->contact_transition_velocity < 2.3e-16) return fail(JB_ERR_INVALID_ARGUMENT, "'transitionVelocity' must be strictly positive.");
    if (o->contact_transition_eps < 0.0) return fail(JB_ERR_INVALID_ARGUMENT, "'transitionEps' must be positive.");
    const double sp = o->sensors_update_period, cp = o->controller_update_period;
    if (sp > 2.3e-16 && cp > 2.3e-16) {
        const double lo = std::min(sp, cp), hi = std::max(sp, cp);
        const double r = std::fmod(hi, lo);
        if (std::min(r, lo - r) > 1e-12) return fail(JB_ERR_INVALID_ARGUMENT, "controller and sensor update periods must be multiple of each other");
    }
    return JB_OK;
}

static void apply_options(JbBatch* b, const JbOptions* o) {
    b->kp.opt = *o;
    double supd = INFINITY;
    if (o->sensors_update_period > 2.3e-16) supd = std::min(supd, o->sensors_update_period);
    if (o->controller_update_period > 2.3e-16) supd = std::min(supd, o->controller_update_period);
    // profile forces with a finite update period add breakpoints (engine.cc:2551-2562)
    for (int j = 0; j < b->kp.n_prof; ++j)
        if (b->kp.prof_period[j] > 2.3e-16) supd = std::min(supd, b->kp.prof_period[j]);
    b->kp.stepper_update_period = std::isfinite(supd) ? supd : 1e308;
}

int jb_batch_destroy(JbBatch* b) {
    if (!b) return JB_OK;
    cudaSetDevice(b->device);
    if (b->stream) cudaStreamSynchronize(b->stream);
#ifndef JB_HOST_EMUL
    for (void* p : b->peer_opened) cudaIpcCloseMemHandle(p);
#endif
    for (void* p : b->allocs) cudaFree(p);
    if (b->h_stage) cudaFreeHost(b->h_stage);
    if (b->h_mirror) cudaFreeHost(b->h_mirror);
#ifndef JB_HOST_EMUL
    if (b->h_peer_timeout) cudaFreeHost(b->h_peer_timeout);
#endif
    if (b->stream) cudaStreamDestroy(b->stream);
    delete b;
    return JB_OK;
}

int jb_batch_create(const JbModelDesc* m, const JbOptions* opt, int32_t n_env, int32_t device, JbBatch** out) {
    if (!m || !opt || !out) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (n_env < 1) return fail(JB_ERR_INVALID_ARGUMENT, "n_env must be >= 1");
    int rc = check_options(opt);
    if (rc) return rc;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(JB_ERR_CUDA, std::string("no CUDA device available (") + cudaGetErrorString(e) + "); jiminy_b200 has no CPU path");
    if (device < 0 || device >= ndev) return fail(JB_ERR_INVALID_ARGUMENT, "invalid device index");
    CU(cudaSetDevice(device));
    JbBatch* b = new JbBatch;
    b->device = device;
    b->n_env = n_env;
    b->n_pad = (n_env + 31) / 32 * 32;
    try {
        int lanes = 0;
        if (const char* s = std::getenv("JB_LANES")) lanes = std::atoi(s);
        b->plan = build_plan(*m, lanes, opt->ode_solver == JB_SOLVER_RUNGE_KUTTA_DOPRI ? 7 : 0);
    } catch (const std::exception& ex) {
        delete b;
        return fail(JB_ERR_INVALID_ARGUMENT, std::string("lane planner: ") + ex.what());
    }
    const Plan& P = b->plan;
    if (P.nrec > MAX_REC) { delete b; return fail(JB_ERR_NOT_IMPLEMENTED, "too many records per lane"); }
    b->nq = m->nq; b->nv = m->nv; b->nmotors = m->nmotors; b->njoints = m->njoints; b->nimu = m->nimu;
    b->q_lower.assign(m->q_lower, m->q_lower + m->nq);
    b->q_upper.assign(m->q_upper, m->q_upper + m->nq);
    if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess) { delete b; return fail(JB_ERR_CUDA, "stream creation failed"); }

    KParams& kp = b->kp;
    kp.n_env = n_env; kp.n_pad = b->n_pad;
    kp.L = P.L; kp.nrec = P.nrec; kp.ntrunk = P.ntrunk; kp.npool = P.npool; kp.ncslot = P.ncslot; kp.nimuslot = P.nimuslot;
    kp.nfields = P.nfields; kp.pool_off = P.pool_off; kp.cslot_off = P.cslot_off; kp.imu_off = P.imu_off; kp.sph_off = P.sph_off;
    kp.nq = m->nq; kp.nv = m->nv; kp.nmotors = m->nmotors; kp.njoints = m->njoints; kp.n_hist = (opt->ode_solver == JB_SOLVER_RUNGE_KUTTA_DOPRI) ? 7 : 0;
    kp.nimu = m->nimu; kp.nforce = m->nforce; kp.nenc = m->nencoder; kp.neff = m->neffort; kp.ncs = m->ncontact_sensor;
    for (int r = 0; r < P.nrec; ++r) { kp.rec_off[r] = P.rec_off[r]; kp.rec_free[r] = P.rec_free[r]; kp.trunk_reduce[r] = P.trunk_reduce[r]; }
    // lane-uniform descriptors: usable when everything the dynamics evaluation branches on is identical on all lanes
    kp.all_uniform = 1;
    for (int r = 0; r < P.nrec; ++r) {
        const RecInt& a = P.rint[static_cast<size_t>(r) * P.L];
        for (int s = 1; s < P.L; ++s) {
            const RecInt& o = P.rint[static_cast<size_t>(r) * P.L + s];
            if (a.kind != o.kind || a.parent_rec != o.parent_rec || a.carry_in != o.carry_in || a.pool != o.pool ||
                a.parent_pool != o.parent_pool || a.carry_out != o.carry_out || a.take_carry != o.take_carry ||
                (a.motor >= 0) != (o.motor >= 0) || a.motor_flags != o.motor_flags || a.ncontact != o.ncontact ||
                a.contact0 != o.contact0 || a.imu_slot != o.imu_slot || a.has_limit != o.has_limit)
                kp.all_uniform = 0;
        }
        kp.rint_u[r] = a;
        kp.kind_u[r] = static_cast<uint8_t>(a.kind);
        for (int s = 1; s < P.L; ++s) if (P.rint[static_cast<size_t>(r) * P.L + s].kind != a.kind) kp.kind_u[r] = 0;
    }
    if (const char* s = std::getenv("JB_FORCE_PER_LANE")) if (std::atoi(s)) kp.all_uniform = 0;
    kp.sig_id = 0;
    JbSensorLayout& L = kp.lay;
    L.imu_offset = 0;
    L.force_offset = 6 * m->nimu;
    L.encoder_offset = L.force_offset + 6 * m->nforce;
    L.effort_offset = L.encoder_offset + 2 * m->nencoder;
    L.contact_offset = L.effort_offset + m->neffort;
    L.width = L.contact_offset + 3 * m->ncontact_sensor;
    b->width = L.width;
    // one force sensor per joint at most (the per-contact table keeps a single sensor index)
    for (int f = 0; f < m->nforce; ++f)
        for (int g = f + 1; g < m->nforce; ++g)
            if (m->force_joint[f] == m->force_joint[g]) { jb_batch_destroy(b); return fail(JB_ERR_NOT_IMPLEMENTED, "several force sensors on one joint"); }
    apply_options(b, opt);

#define ALLOC(ptr, count) do { int rc_ = dev_alloc(b, &(ptr), (count)); if (rc_) { jb_batch_destroy(b); return rc_; } } while (0)
    RecInt* d_rint; RecDbl* d_rdbl; ContactSlot* d_cs; double* d_imu;
    ALLOC(d_rint, P.rint.size()); ALLOC(d_rdbl, P.rdbl.size()); ALLOC(d_cs, P.cslots.size()); ALLOC(d_imu, 12 * static_cast<size_t>(m->nimu));
    const size_t N = b->n_pad;
    ALLOC(b->d_q, N * m->nq); ALLOC(b->d_v, N * m->nv); ALLOC(b->d_a, N * m->nv); ALLOC(b->d_sched, N * SCH_N);
    ALLOC(b->d_iters, 2 * N); ALLOC(b->d_status, N);
    ALLOC(b->d_cmd, static_cast<size_t>(n_env) * m->nmotors); ALLOC(b->d_sensors, static_cast<size_t>(n_env) * L.width);
    ALLOC(b->d_qv, static_cast<size_t>(n_env) * (m->nq + m->nv));
    ALLOC(b->d_qin, static_cast<size_t>(n_env) * m->nq); ALLOC(b->d_vin, static_cast<size_t>(n_env) * m->nv);
    ALLOC(b->d_aout, static_cast<size_t>(n_env) * m->nv); ALLOC(b->d_fext, static_cast<size_t>(n_env) * m->njoints * 6);
    ALLOC(b->d_u, static_cast<size_t>(n_env) * m->nv); ALLOC(b->d_umotor, static_cast<size_t>(n_env) * m->nmotors);
    ALLOC(b->d_springs, 2 * static_cast<size_t>(m->nv)); ALLOC(b->d_mask, n_env);
    ALLOC(b->d_pd, 2 * static_cast<size_t>(m->nmotors)); ALLOC(b->d_cmd_torque, static_cast<size_t>(n_env) * m->nmotors);
    ALLOC(b->d_stage, static_cast<size_t>(n_env) * std::max(std::max(m->nq, m->nv), SCH_N + 0));
#define ALLOC2 ALLOC
    cudaMemcpyAsync(d_rint, P.rint.data(), P.rint.size() * sizeof(RecInt), cudaMemcpyHostToDevice, b->stream);
    cudaMemcpyAsync(d_rdbl, P.rdbl.data(), P.rdbl.size() * sizeof(RecDbl), cudaMemcpyHostToDevice, b->stream);
    if (!P.cslots.empty()) cudaMemcpyAsync(d_cs, P.cslots.data(), P.cslots.size() * sizeof(ContactSlot), cudaMemcpyHostToDevice, b->stream);
    if (m->nimu) cudaMemcpyAsync(d_imu, m->imu_placement, 12 * sizeof(double) * m->nimu, cudaMemcpyHostToDevice, b->stream);
    std::vector<int32_t> st(N, JB_ENV_NOT_STARTED);
    cudaMemcpyAsync(b->d_status, st.data(), N * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream);
    kp.rint = d_rint; kp.rdbl = d_rdbl; kp.cslots = d_cs; kp.imu_placement = d_imu; kp.springs = nullptr;
    kp.pd_gains = nullptr; kp.cmd_torque = b->d_cmd_torque; kp.pdf = nullptr; kp.pdf_state = nullptr; kp.pdf_safety = 0; kp.mahony = nullptr; kp.mahony_kp = 1.0; kp.mahony_ki = 0.1;
    kp.q = b->d_q; kp.v = b->d_v; kp.a = b->d_a; kp.sched = b->d_sched; kp.iters = b->d_iters; kp.status = b->d_status;
    kp.command = b->d_cmd; kp.sensors = b->d_sensors; kp.qv_out = b->d_qv;
    kp.q_in = b->d_qin; kp.v_in = b->d_vin;
    kp.a_out = b->d_aout; kp.fext_out = b->d_fext; kp.u_out = b->d_u;
    kp.eff_u = b->d_u; kp.eff_umotor = b->d_umotor; kp.eff_fext = b->d_fext;
    {
        double *d_en, *d_ea, *d_ef;
        ALLOC2(d_en, 2 * static_cast<size_t>(n_env)); ALLOC2(d_ea, static_cast<size_t>(n_env) * m->njoints * 6);
        ALLOC2(d_ef, static_cast<size_t>(n_env) * m->njoints * 6);
        kp.extra_energy = d_en; kp.extra_a = d_ea; kp.extra_f = d_ef;
        double *d_y, *d_c, *d_vc, *d_hg;
        ALLOC2(d_y, static_cast<size_t>(n_env) * m->njoints * 10); ALLOC2(d_c, static_cast<size_t>(n_env) * m->njoints * 3);
        ALLOC2(d_vc, static_cast<size_t>(n_env) * m->njoints * 3); ALLOC2(d_hg, static_cast<size_t>(n_env) * 12);
        kp.extra_ycrb = d_y; kp.extra_com = d_c; kp.extra_vcom = d_vc; kp.extra_hg = d_hg; kp.total_mass = P.total_mass;
    }

    if (SigQuadruped::matches(kp) && !std::getenv("JB_NO_STATIC_PLAN")) kp.sig_id = SigQuadruped::ID;
    kp.rhs_variant = (std::getenv("JB_QUADRUPED_ABA") && std::atoi(std::getenv("JB_QUADRUPED_ABA"))) ? 0 : 1;
    kp.fast_bounds = 0;   // set below, once the constraint tables exist
    // ---- constraint path: lookup tables, persistent state and workspace (jb_constraints.cuh)
    {
        std::vector<JointMap> jmap(m->njoints);
        std::vector<int32_t> jc_joint, jc_of_joint(m->njoints, -1);
        for (int j = 0; j < m->njoints; ++j) {
            JointMap& jm = jmap[j];
            jm = JointMap{-1, 0, j ? m->parent[j] : 0, j ? m->idx_q[j] : 0, j ? m->idx_v[j] : 0, 0, REC_PAD, 0};
            if (!j) continue;
            int found = 0;
            for (int r = 0; r < P.nrec; ++r)
                for (int s = 0; s < P.L; ++s) {
                    const RecInt& ri = P.rint[static_cast<size_t>(r) * P.L + s];
                    if (ri.kind == REC_PAD || ri.joint != j) continue;
                    if (!found) { jm.rec = r; jm.sub = s; jm.kind = ri.kind; jm.nvj = ri.kind == REC_FREE ? 6 : (ri.kind == REC_SPH ? 3 : 1); }
                    ++found;
                }
            jm.trunk = found > 1;
            if (m->joint_type[j] != JB_JOINT_FREEFLYER && m->joint_type[j] != JB_JOINT_SPHERICAL) { jc_of_joint[j] = static_cast<int32_t>(jc_joint.size()); jc_joint.push_back(j); }
        }
        std::vector<ContactMap> cmap(std::max(m->ncontacts, 1));
        for (int k = 0; k < m->ncontacts; ++k) {
            ContactMap& cm = cmap[k];
            cm.joint = m->contact_joint[k]; cm.sub = 0; cm.cslot = 0; cm.trunk = 0;
            std::memcpy(cm.placement, m->contact_placement + 12 * k, sizeof cm.placement);
            int found = 0;
            for (int cs = 0; cs < P.ncslot; ++cs)
                for (int s = 0; s < P.L; ++s)
                    if (P.cslots[static_cast<size_t>(cs) * P.L + s].contact == k) { if (!found) { cm.cslot = cs; cm.sub = s; } ++found; }
            cm.trunk = found > 1;
        }
        kp.n_jc = static_cast<int32_t>(jc_joint.size()); kp.n_cc = m->ncontacts;
        kp.m_max = kp.n_jc + 4 * kp.n_cc;
        bool has_spherical = false;
        for (int j = 1; j < m->njoints; ++j) has_spherical = has_spherical || m->joint_type[j] == JB_JOINT_SPHERICAL;
        // the structured solvers (quadruped, body space, lane blocks) walk 1-dof and free-flyer records only: a model with
        // flexibility joints goes through the generic solver (jb_constraints.cuh)
        kp.cons_on = (m->nv <= 64) ? 1 : 0;
        kp.cons_off = P.nfields;
        kp.cq_off = P.nfields + 1;
        kp.cq_on = (kp.cons_on && opt->contact_model == JB_CONTACT_CONSTRAINT && cons_quadruped_matches(kp, P, *m) &&
                    !(std::getenv("JB_NO_STRUCTURED_CONS") && std::atoi(std::getenv("JB_NO_STRUCTURED_CONS")))) ? 1 : 0;
        b->base_fields = P.nfields + 1 + (kp.cq_on ? CQ_SIZE : 0);
        // body-space contact solver (jb_constraints_bodies.cuh): the distinct parent joints of the contact frames;
        // its sweep keeps a = Omega F in shared memory (not reserved when the quadruped solver covers the case)
        std::vector<int32_t> body_of(std::max(m->ncontacts, 1), 0), body_joint;
        for (int k = 0; k < m->ncontacts; ++k) {
            size_t bi = 0;
            while (bi < body_joint.size() && body_joint[bi] != cmap[k].joint) ++bi;
            if (bi == body_joint.size()) body_joint.push_back(cmap[k].joint);
            body_of[k] = static_cast<int32_t>(bi);
        }
        const char* offb = std::getenv("JB_NO_BODY_CONS");
        const bool bd_candidate = kp.cons_on && !kp.cq_on && !has_spherical && P.L > 1 && P.L <= 8 && m->ncontacts > 0 && m->ncontacts <= BD_MAX_CONTACTS &&
                                  body_joint.size() <= BD_MAX_BODIES && opt->contact_model == JB_CONTACT_CONSTRAINT && !(offb && std::atoi(offb));
        kp.bd_off = b->base_fields; kp.bd_lsh = 0;
        while ((1 << kp.bd_lsh) < P.L) ++kp.bd_lsh;
        if (bd_candidate) b->base_fields += 2 * ((6 * static_cast<int>(body_joint.size()) + P.L - 1) / P.L);
        if (kp.cons_on) {
            JointMap* d_jmap; ContactMap* d_cmap; int32_t *d_jcj, *d_jcof; double *d_cst, *d_cwk;
            const int cs_fields = CS_JOINT0 + CS_JOINT_SIZE * kp.n_jc + CS_CONTACT_SIZE * kp.n_cc;
            const CwLayout w = cw_layout(m->njoints, m->nv, kp.m_max);
            ALLOC(d_jmap, jmap.size()); ALLOC(d_cmap, cmap.size()); ALLOC(d_jcj, std::max<size_t>(jc_joint.size(), 1)); ALLOC(d_jcof, jc_of_joint.size());
            // the workspace is scratch of one dynamics evaluation, one row per block of the launch
            int n_sm = 1, blocks_per_sm = 1;
            {
                const int epw_ = 32 / P.L;
                n_sm = (n_env + epw_ - 1) / epw_;      // (historical names: rows = n_sm * blocks_per_sm blocks)
            }
            const size_t cw_rows = std::min<size_t>(N, static_cast<size_t>(n_sm) * blocks_per_sm * (32 / P.L));
            unsigned int* d_slots;
            ALLOC(d_slots, n_sm);
            kp.cw_slots = d_slots; kp.cw_blocks_per_sm = blocks_per_sm; kp.cw_n_sm = n_sm;
            ALLOC(d_cst, static_cast<size_t>(cs_fields) * N); ALLOC(d_cwk, static_cast<size_t>(w.total) * std::max<size_t>(cw_rows, static_cast<size_t>(n_sm) * blocks_per_sm * (32 / P.L)));
            cudaMemcpyAsync(d_jmap, jmap.data(), jmap.size() * sizeof(JointMap), cudaMemcpyHostToDevice, b->stream);
            cudaMemcpyAsync(d_cmap, cmap.data(), cmap.size() * sizeof(ContactMap), cudaMemcpyHostToDevice, b->stream);
            if (!jc_joint.empty()) cudaMemcpyAsync(d_jcj, jc_joint.data(), jc_joint.size() * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream);
            cudaMemcpyAsync(d_jcof, jc_of_joint.data(), jc_of_joint.size() * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream);
            kp.cs_total = cs_fields; kp.cw_total = w.total;
            // lane-block solver: dof numbering inside the trunk block and each lane's private block, row budget per lane
            kp.lb_on = 0;
            if (P.L > 1 && !has_spherical) {
                std::vector<int32_t> dof0(static_cast<size_t>(P.nrec) * P.L, 0);
                int nt = 0, nl = 0, ml = 0;
                for (int s = 0; s < P.L; ++s) {
                    int t = 0, l = 0, rows = 0;
                    for (int r = 0; r < P.nrec; ++r) {
                        const RecInt& ri = P.rint[static_cast<size_t>(r) * P.L + s];
                        if (ri.kind == REC_PAD) continue;
                        const int nd = ri.kind == REC_FREE ? 6 : 1;
                        int& n = r < P.ntrunk ? t : l;
                        dof0[static_cast<size_t>(r) * P.L + s] = n;
                        n += nd;
                    }
                    for (size_t k = 0; k < jc_joint.size(); ++k) { const JointMap& jm = jmap[jc_joint[k]]; if ((jm.trunk ? 0 : jm.sub) == s) rows += 1; }
                    for (int k = 0; k < m->ncontacts; ++k) if ((cmap[k].trunk ? 0 : cmap[k].sub) == s) rows += 4;
                    nt = t; nl = std::max(nl, l); ml = std::max(ml, rows);
                    kp.lb_nl_of[s] = l;
                }
                const char* off = std::getenv("JB_NO_BLOCK_CONS");
                kp.bd_on = 0;
                if (nt <= LB_MAX_NT && P.L <= 8 && !(off && std::atoi(off))) {
                    const LbLayout lw = lb_layout(P.nrec, P.ntrunk, nl, nt, ml, kp.n_jc + kp.n_cc);
                    int lw_total = lw.total;
                    if (bd_candidate) {
                        int per_lane[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ncar = 0;
                        kp.bd_n = static_cast<int32_t>(body_joint.size());
                        for (int bi = 0; bi < kp.bd_n; ++bi) {
                            const JointMap& jm = jmap[body_joint[bi]];
                            kp.bd_rec[bi] = jm.rec; kp.bd_owner[bi] = jm.trunk ? 0 : jm.sub;
                            kp.bd_slot[bi] = per_lane[kp.bd_owner[bi]]++;
                            ncar = std::max(ncar, per_lane[kp.bd_owner[bi]]);
                        }
                        kp.bd_ncar = ncar;
                        const BdLane bl = bd_lane_layout(lw.total, ncar, nl, nt, m->ncontacts, kp.bd_n);
                        const BdLayout bs = bd_layout(kp.bd_n, nt, m->ncontacts);
                        if (bs.total <= kp.cw_total) {   // the env's row of the generic workspace doubles as the shared area
                            int32_t* d_bof;
                            ALLOC(d_bof, body_of.size());
                            cudaMemcpyAsync(d_bof, body_of.data(), body_of.size() * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream);
                            kp.bd_of_contact = d_bof; kp.bd_on = 1; lw_total = bl.total;
                        }
                    }
                    int32_t* d_dof0; double* d_lwk;
                    ALLOC(d_dof0, dof0.size());
                    ALLOC(d_lwk, static_cast<size_t>(lw_total) * 32 * std::max<size_t>(1, static_cast<size_t>(n_sm) * blocks_per_sm));
                    cudaMemcpyAsync(d_dof0, dof0.data(), dof0.size() * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream);
                    kp.lb_on = 1; kp.lb_nt = nt; kp.lb_nl = nl; kp.lb_ml = ml; kp.lw_total = lw_total; kp.lb_dof0 = d_dof0; kp.lwork = d_lwk;
                }
            }
            b->jc_joint = jc_joint;
            kp.jmap = d_jmap; kp.cmap = d_cmap; kp.jc_joint = d_jcj; kp.jc_of_joint = d_jcof; kp.cstate = d_cst; kp.cwork = d_cwk;
        }
    }
    kp.fast_bounds = (kp.sig_id == SigQuadruped::ID && kp.rhs_variant == 1 && kp.cons_on &&
                      !(std::getenv("JB_NO_FAST_BOUNDS") && std::atoi(std::getenv("JB_NO_FAST_BOUNDS")))) ? 1 : 0;
    kp.fast_bounds_io = kp.fast_bounds;
    static_assert(CONS_PGS_MAX_ITER == sizeof(kp.pgs_relax) / sizeof(double), "relaxation table");
    for (int iter = 0; iter < CONS_PGS_MAX_ITER; ++iter) {
        const double ratio = (static_cast<double>(CONS_PGS_MAX_ITER - CONS_RELAX_MIN_ITER) - iter) /
                             (CONS_PGS_MAX_ITER - CONS_RELAX_MIN_ITER - CONS_RELAX_MAX_ITER);
        double wr = CONS_RELAX_MAX;
        if (ratio < 1.0) {
            wr = CONS_RELAX_MIN;
            if (ratio > 0.0) wr += (CONS_RELAX_MAX - CONS_RELAX_MIN) * (ratio * ratio);
        }
        kp.pgs_relax[iter] = wr;
    }
    kp.uniform_solver = (std::getenv("JB_NO_UNIFORM_SOLVER") && std::atoi(std::getenv("JB_NO_UNIFORM_SOLVER"))) ? 0 : 1;
    if (const char* e = std::getenv("JB_FAST_BOUNDS_MODE")) { const int m_ = std::atoi(e); if (m_ == 2) kp.fast_bounds = 0; if (m_ == 3) kp.fast_bounds_io = 0; }
    kp.n_eslot = 0; kp.n_imp = 0; kp.n_prof = 0; kp.ext_off = b->base_fields;
    b->smem_bytes = static_cast<size_t>(b->base_fields) * 32 * sizeof(double);
    if (b->smem_bytes > 227 * 1024) { jb_batch_destroy(b); return fail(JB_ERR_NOT_IMPLEMENTED, "robot too large: per-warp working set exceeds shared memory (" + P.describe() + ")"); }
    ALLOC(b->d_needs_full, N);
    kp.needs_full = b->d_needs_full;
    if (const char* s = std::getenv("JB_NO_FAST_KERNEL")) b->no_fast_kernel = std::atoi(s) != 0;
    if (raise_smem_attr(device, b->smem_bytes)) { jb_batch_destroy(b); return JB_ERR_CUDA; }
    e = cudaStreamSynchronize(b->stream);
    if (e != cudaSuccess) { jb_batch_destroy(b); return fail(JB_ERR_CUDA, std::string("upload failed: ") + cudaGetErrorString(e)); }
    *out = b;
    return JB_OK;
}

int jb_describe(JbBatch* b, char* buf, int32_t len) {
    if (!b || !buf) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    // (names every switch of the evaluation path, so that a test or an A/B run can check which one it measured)
    const char* hot = b->no_fast_kernel ? "none, every step runs the full kernel"
                      : b->kp.sig_id == SigQuadruped::ID ? (b->kp.rhs_variant == 1 ? "quadruped signature, composite-rigid-body evaluation" : "quadruped signature, ABA sweeps")
                      : (b->kp.all_uniform ? "ABA sweeps (dynamic plan, lane-uniform descriptors)" : "ABA sweeps (dynamic plan, per-lane descriptors)");
    std::snprintf(buf, len, "%s; hot path: %s%s; constraints: %s", b->plan.describe().c_str(), hot,
                  b->kp.fast_bounds ? ", joint bounds solved in the evaluation" : "",
                  !b->kp.cons_on ? "flag only" : (b->kp.cq_on ? (b->kp.lb_on ? "structured quadruped solver + lane-block solver" : "structured quadruped solver + generic")
                                                 : (b->kp.bd_on ? "body-space contact solver + lane-block solver" : (b->kp.lb_on ? "lane-block solver" : "generic solver"))));
    return JB_OK;
}

int jb_set_options(JbBatch* b, const JbOptions* o) {
    if (!b || !o) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    int rc = check_options(o);
    if (rc) return rc;
    if (o->ode_solver == JB_SOLVER_RUNGE_KUTTA_DOPRI && b->kp.n_hist == 0)
        return fail(JB_ERR_BAD_CONTROL_FLOW, "switching to 'runge_kutta_dopri' changes the working-set layout: create a new batch");
    if (o->contact_model == JB_CONTACT_CONSTRAINT && !b->kp.cons_on)
        return fail(JB_ERR_NOT_IMPLEMENTED, "contacts.model = 'constraint' is not available for this robot (more than 64 degrees of freedom)");
    apply_options(b, o);
    return JB_OK;
}

// Model randomisation (Model::addBiasedToExtendedModel, core/src/robot/model.cc:1166-1236): a reset of the reference
// re-draws the inertias and joint placements of ONE robot; a batch holds n_variants such draws of the same kinematic tree
// and every group of envs that shares a warp uses one of them (a table base per block: nothing on the hot path changes).
int jb_set_model_variants(JbBatch* b, int32_t n_variants, const JbModelDesc* models, const int32_t* variant_of_group) {
    if (!b || !models || !variant_of_group || n_variants < 1) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    const Plan& P0 = b->plan;
    const int epw = 32 / P0.L, ngroups = (b->n_env + epw - 1) / epw;
    std::vector<RecDbl> rows;
    std::vector<double> mass(n_variants);
    for (int v = 0; v < n_variants; ++v) {
        Plan P;
        try { P = build_plan(models[v], P0.L, b->kp.n_hist); }
        catch (const std::exception& ex) { return fail(JB_ERR_INVALID_ARGUMENT, std::string("lane planner (variant): ") + ex.what()); }
        // same tree, same hardware: everything but the numbers in the double tables must be what the batch was built with
        bool same = P.L == P0.L && P.nrec == P0.nrec && P.nfields == P0.nfields && P.rint.size() == P0.rint.size() &&
                    P.cslots.size() == P0.cslots.size() && models[v].nq == b->nq && models[v].nv == b->nv && models[v].nmotors == b->nmotors;
        if (same) same = std::memcmp(P.rint.data(), P0.rint.data(), P.rint.size() * sizeof(RecInt)) == 0;
        if (same && !P.cslots.empty()) same = std::memcmp(P.cslots.data(), P0.cslots.data(), P.cslots.size() * sizeof(ContactSlot)) == 0;
        if (!same) return fail(JB_ERR_INVALID_ARGUMENT, "a model variant must have the kinematic tree, hardware and frames of the batch's model (only inertias and joint placements may differ)");
        rows.insert(rows.end(), P.rdbl.begin(), P.rdbl.end());
        mass[v] = P.total_mass;
    }
    std::vector<int32_t> vob(ngroups);
    std::vector<double> bm(ngroups);
    for (int g = 0; g < ngroups; ++g) {
        if (variant_of_group[g] < 0 || variant_of_group[g] >= n_variants) return fail(JB_ERR_INVALID_ARGUMENT, "variant index out of range");
        vob[g] = variant_of_group[g]; bm[g] = mass[vob[g]];
    }
    RecDbl* d_rows; int32_t* d_vob; double* d_bm;
    int rc;
    if ((rc = dev_alloc(b, &d_rows, rows.size())) || (rc = dev_alloc(b, &d_vob, vob.size())) || (rc = dev_alloc(b, &d_bm, bm.size()))) return rc;
    CU(cudaMemcpyAsync(d_rows, rows.data(), rows.size() * sizeof(RecDbl), cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(d_vob, vob.data(), vob.size() * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(d_bm, bm.data(), bm.size() * sizeof(double), cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));   // the host vectors go away
    b->kp.rdbl = d_rows; b->kp.n_variants = n_variants > 1 ? n_variants : 2;   // (a single variant still replaces the table: keep the indirection on)
    b->kp.rdbl_rows = static_cast<int32_t>(P0.rdbl.size());
    b->kp.variant_of_block = d_vob; b->kp.block_mass = d_bm;
    return JB_OK;
}

int jb_envs_per_group(JbBatch* b) { return b ? 32 / b->plan.L : 0; }

// Linear internal dynamics u_custom = -k q - d v on 1-dof joints: the device-side stand-in for the
// `internalDynamics` functor of FunctionalController (controller_functor.h:27-80).
int jb_set_joint_springs(JbBatch* b, const double* k, const double* d) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (!k || !d) { b->kp.springs = nullptr; return JB_OK; }
    CU(cudaMemcpyAsync(b->d_springs, k, sizeof(double) * b->nv, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(b->d_springs + b->nv, d, sizeof(double) * b->nv, cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    b->kp.springs = b->d_springs;
    return JB_OK;
}

// Device-side PD controller block (see update_pd_commands in jb_kernel.cuh).
int jb_set_pd_controller(JbBatch* b, const double* kp, const double* kd) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (!kp || !kd) { b->kp.pd_gains = nullptr; return JB_OK; }
    if (!b->nmotors) return fail(JB_ERR_INVALID_ARGUMENT, "the robot has no motor");
    const JbOptions& o = b->kp.opt;
    if (!(o.controller_update_period > 2.3e-16))
        return fail(JB_ERR_NOT_IMPLEMENTED, "the device PD controller needs a discrete controllerUpdatePeriod");
    if (o.sensors_update_period > 2.3e-16 && std::fabs(o.sensors_update_period - o.controller_update_period) > 1e-12)
        return fail(JB_ERR_NOT_IMPLEMENTED, "the device PD controller needs sensorsUpdatePeriod == controllerUpdatePeriod (or 0)");
    CU(cudaMemcpyAsync(b->d_pd, kp, sizeof(double) * b->nmotors, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(b->d_pd + b->nmotors, kd, sizeof(double) * b->nmotors, cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    b->kp.pd_gains = b->d_pd;
    return JB_OK;
}

int jb_set_pd_controller_full(JbBatch* b, const double* kp, const double* kd, const double* lower, const double* upper, const double* safety) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (!kp) { b->kp.pdf = nullptr; return JB_OK; }
    if (!kd || !lower || !upper) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->nmotors) return fail(JB_ERR_INVALID_ARGUMENT, "the robot has no motor");
    const JbOptions& o = b->kp.opt;
    if (!(o.controller_update_period > 2.3e-16))
        return fail(JB_ERR_NOT_IMPLEMENTED, "the device PD controller needs a discrete controllerUpdatePeriod");
    if (o.sensors_update_period > 2.3e-16 && std::fabs(o.sensors_update_period - o.controller_update_period) > 1e-12)
        return fail(JB_ERR_NOT_IMPLEMENTED, "the device PD controller needs sensorsUpdatePeriod == controllerUpdatePeriod (or 0)");
    const size_t nm = b->nmotors;
    for (size_t k = 0; k < 3 * nm; ++k) if (!(lower[k] <= upper[k])) return fail(JB_ERR_INVALID_ARGUMENT, "state_lower must not exceed state_upper");
    if (!b->d_pdf) {
        int rc = dev_alloc(b, &b->d_pdf, 13 * nm);
        if (rc) return rc;
        rc = dev_alloc(b, &b->d_pdf_state, static_cast<size_t>(b->n_env) * 3 * nm);
        if (rc) return rc;
        rc = dev_alloc(b, &b->d_pdf_snap, static_cast<size_t>(b->n_env) * 3 * nm);
        if (rc) return rc;
    }
    std::vector<double> h(13 * nm, 0.0);
    std::memcpy(h.data(), kp, sizeof(double) * nm);
    std::memcpy(h.data() + nm, kd, sizeof(double) * nm);
    std::memcpy(h.data() + 2 * nm, lower, sizeof(double) * 3 * nm);
    std::memcpy(h.data() + 5 * nm, upper, sizeof(double) * 3 * nm);
    if (safety) {
        std::memcpy(h.data() + 8 * nm, safety, sizeof(double) * 5 * nm);
        for (size_t k = 0; k < nm; ++k) if (!(safety[4 * nm + k] >= 0.0)) return fail(JB_ERR_INVALID_ARGUMENT, "the soft velocity limit must be positive");
    }
    CU(cudaMemcpyAsync(b->d_pdf, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    b->kp.pdf = b->d_pdf; b->kp.pdf_state = b->d_pdf_state; b->kp.pdf_snap = b->d_pdf_snap; b->kp.pdf_safety = safety ? 1 : 0;
    b->kp.pd_gains = nullptr;
    return JB_OK;
}

int jb_get_pd_controller_state(JbBatch* b, double* state) {
    if (!b || !state) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->kp.pdf) return fail(JB_ERR_BAD_CONTROL_FLOW, "the PDController block is not enabled (jb_set_pd_controller_full)");
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpyAsync(state, b->d_pdf_state, sizeof(double) * b->n_env * 3 * b->nmotors, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_set_pd_controller_state(JbBatch* b, const double* state) {
    if (!b || !state) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->kp.pdf) return fail(JB_ERR_BAD_CONTROL_FLOW, "the PDController block is not enabled (jb_set_pd_controller_full)");
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpyAsync(b->d_pdf_state, state, sizeof(double) * b->n_env * 3 * b->nmotors, cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_set_mahony_filter(JbBatch* b, double kp, double ki) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (kp < 0.0) { b->kp.mahony = nullptr; return JB_OK; }
    if (!b->nimu) return fail(JB_ERR_INVALID_ARGUMENT, "the robot has no IMU sensor");
    if (b->nimu > 1) return fail(JB_ERR_NOT_IMPLEMENTED, "the device Mahony filter handles one IMU per robot");
    if (!(b->kp.opt.sensors_update_period > 2.3e-16)) return fail(JB_ERR_NOT_IMPLEMENTED, "the Mahony filter needs a discrete sensorsUpdatePeriod");
    if (ki < 0.0) return fail(JB_ERR_INVALID_ARGUMENT, "ki must be positive");
    if (!b->d_mahony) {
        int rc = dev_alloc(b, &b->d_mahony, static_cast<size_t>(b->n_env) * b->nimu * 10);
        if (rc) return rc;
        rc = dev_alloc(b, &b->d_mahony_snap, static_cast<size_t>(b->n_env) * b->nimu * 10);
        if (rc) return rc;
        CU(cudaStreamSynchronize(b->stream));
    }
    b->kp.mahony = b->d_mahony; b->kp.mahony_snap = b->d_mahony_snap; b->kp.mahony_kp = kp; b->kp.mahony_ki = ki;
    return JB_OK;
}

int jb_get_mahony_filter(JbBatch* b, double* out) {
    if (!b || !out) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->kp.mahony) return fail(JB_ERR_BAD_CONTROL_FLOW, "the Mahony filter is not enabled");
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpyAsync(out, b->d_mahony, sizeof(double) * b->n_env * b->nimu * 10, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_get_constraints(JbBatch* b, uint8_t* joint_enabled, double* joint_lambda, uint8_t* contact_enabled, double* contact_lambda) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->kp.cons_on) return fail(JB_ERR_NOT_IMPLEMENTED, "no constraint state for this robot (more than 64 degrees of freedom)");
    CU(cudaSetDevice(b->device));
    const size_t cs = b->kp.cs_total, n = b->n_env;
    std::vector<double> h(cs * n);
    CU(cudaMemcpyAsync(h.data(), b->kp.cstate, sizeof(double) * cs * n, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    const int nj = b->njoints, ncc = b->kp.n_cc;
    if (joint_enabled) std::memset(joint_enabled, 0, n * nj);
    if (joint_lambda) std::fill(joint_lambda, joint_lambda + n * nj, 0.0);
    for (size_t e = 0; e < n; ++e) {
        const double* row = h.data() + e * cs;
        for (size_t k = 0; k < b->jc_joint.size(); ++k) {
            const double* c = row + CS_JOINT0 + CS_JOINT_SIZE * k;
            if (joint_enabled) joint_enabled[e * nj + b->jc_joint[k]] = c[0] != 0.0;
            if (joint_lambda) joint_lambda[e * nj + b->jc_joint[k]] = c[3];
        }
        for (int k = 0; k < ncc; ++k) {
            const double* c = row + CS_JOINT0 + CS_JOINT_SIZE * b->jc_joint.size() + CS_CONTACT_SIZE * k;
            if (contact_enabled) contact_enabled[e * ncc + k] = c[0] != 0.0;
            if (contact_lambda) std::memcpy(contact_lambda + (e * ncc + k) * 4, c + 1, 4 * sizeof(double));
        }
    }
    return JB_OK;
}

// ---- sensor measurement pipeline ---------------------------------------------------------------------------
static const int kSensorFields[5] = {6, 6, 2, 1, 3};

int jb_set_sensor_options(JbBatch* b, int32_t type, int32_t index, const double* noise_std, const double* bias, double delay,
                          double jitter, int32_t delay_interpolation_order) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (b->any_started) return fail(JB_ERR_BAD_CONTROL_FLOW, "Robot already locked, probably because a simulation is running. Please stop it before setting sensor options.");
    const int counts[5] = {b->kp.nimu, b->kp.nforce, b->kp.nenc, b->kp.neff, b->kp.ncs};
    const int offs[5] = {b->kp.lay.imu_offset, b->kp.lay.force_offset, b->kp.lay.encoder_offset, b->kp.lay.effort_offset, b->kp.lay.contact_offset};
    if (type < 0 || type > 4 || index < 0 || index >= counts[type]) return fail(JB_ERR_INVALID_ARGUMENT, "unknown sensor");
    if (delay < 0.0 || jitter < 0.0) return fail(JB_ERR_INVALID_ARGUMENT, "delay and jitter must be positive");
    if (delay_interpolation_order != 0 && delay_interpolation_order != 1) return fail(JB_ERR_NOT_IMPLEMENTED, "`delayInterpolationOrder` must be either 0 or 1.");
    if (!(b->kp.opt.sensors_update_period > 2.3e-16))
        return fail(JB_ERR_NOT_IMPLEMENTED, "the device measurement pipeline needs a discrete sensorsUpdatePeriod (the delay buffer is sized from it)");
    if (b->sdesc.empty()) {
        for (int ty = 0; ty < 5; ++ty)
            for (int k = 0; k < counts[ty]; ++k) {
                SensorDesc d{};
                d.type = ty; d.index = k; d.nf = kSensorFields[ty]; d.ns = counts[ty]; d.offset = offs[ty]; d.order = 1;
                b->sdesc.push_back(d);
            }
    }
    for (SensorDesc& d : b->sdesc) {
        if (d.type != type || d.index != index) continue;
        d.has_noise = noise_std != nullptr; d.has_bias = bias != nullptr;
        for (int f = 0; f < d.nf; ++f) { d.noise_std[f] = noise_std ? noise_std[f] : 0.0; d.bias[f] = bias ? bias[f] : 0.0; }
        d.delay = delay; d.jitter = jitter; d.order = delay_interpolation_order;
    }
    b->sp_dirty = true;
    return JB_OK;
}

int jb_set_seeds(JbBatch* b, const uint32_t* seeds) {
    if (!b || !seeds) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    b->seeds.assign(seeds, seeds + b->n_env);
    return JB_OK;
}

// Tables, buffers and start states of the pipeline, (re)built at jb_start when options changed
static int prepare_sensor_pipeline(JbBatch* b, const uint8_t* mask) {
    if (b->sdesc.empty()) return JB_OK;
    KParams& kp = b->kp;
    const int ns = static_cast<int>(b->sdesc.size());
    if (b->sp_dirty || !kp.sp_on) {
        double dmax_all = 0.0;
        for (int ty = 0; ty < 5; ++ty) kp.sp_delay_max[ty] = 0.0;
        for (const SensorDesc& d : b->sdesc) {
            kp.sp_delay_max[d.type] = std::max(kp.sp_delay_max[d.type], d.delay + d.jitter);
            dmax_all = std::max(dmax_all, d.delay + d.jitter);
        }
        const int cap = static_cast<int>(std::floor((dmax_all + 0.02) / kp.opt.sensors_update_period)) + 8;
        if (cap > 4096) return fail(JB_ERR_NOT_IMPLEMENTED, "sensor delay too long for the sensor update period (more than 4096 samples)");
        if (!b->d_sdesc) {
            int rc;
            if ((rc = dev_alloc(b, &b->d_sdesc, ns))) return rc;
            if ((rc = dev_alloc(b, &b->d_sp_rng, static_cast<size_t>(b->n_env) * ns))) return rc;
            if ((rc = dev_alloc(b, &b->d_sp_rng_init, static_cast<size_t>(b->n_env) * ns))) return rc;
            if ((rc = dev_alloc(b, &b->d_sp_snap_rng, static_cast<size_t>(b->n_env) * ns))) return rc;
            if ((rc = dev_alloc(b, &b->d_sp_count, static_cast<size_t>(b->n_env) * 6))) return rc;
            if ((rc = dev_alloc(b, &b->d_sp_snap_count, static_cast<size_t>(b->n_env) * 6))) return rc;
            // ziggurat tables of the normal sampler (random.cc:62-98), computed with the host's libm like the reference does
            std::vector<uint32_t> kn(128, 0); std::vector<float> fn(128, 0.f), wn(128, 0.f);
            {
                const double m1 = 2147483648.0, vn = 9.91256303526217e-03;
                double dn = 3.442619855899, tn = dn;
                const double q = vn / std::exp(-0.5 * dn * dn);
                kn[0] = static_cast<uint32_t>((dn / q) * m1); kn[1] = 0;
                wn[0] = static_cast<float>(q / m1); wn[127] = static_cast<float>(dn / m1);
                fn[0] = 1.0F; fn[127] = static_cast<float>(std::exp(-0.5 * dn * dn));
                for (int i = 126; 1 <= i; i--) {
                    dn = std::sqrt(-2.0 * std::log(vn / dn + std::exp(-0.5 * dn * dn)));
                    kn[i + 1] = static_cast<uint32_t>((dn / tn) * m1);
                    tn = dn;
                    fn[i] = static_cast<float>(std::exp(-0.5 * dn * dn));
                    wn[i] = static_cast<float>(dn / m1);
                }
            }
            uint32_t* d_kn; float *d_fn, *d_wn;
            if ((rc = dev_alloc(b, &d_kn, 128)) || (rc = dev_alloc(b, &d_fn, 128)) || (rc = dev_alloc(b, &d_wn, 128))) return rc;
            CU(cudaMemcpyAsync(d_kn, kn.data(), 128 * sizeof(uint32_t), cudaMemcpyHostToDevice, b->stream));
            CU(cudaMemcpyAsync(d_fn, fn.data(), 128 * sizeof(float), cudaMemcpyHostToDevice, b->stream));
            CU(cudaMemcpyAsync(d_wn, wn.data(), 128 * sizeof(float), cudaMemcpyHostToDevice, b->stream));
            CU(cudaStreamSynchronize(b->stream));
            kp.zig_kn = d_kn; kp.zig_fn = d_fn; kp.zig_wn = d_wn;
        }
        if (cap > b->sp_cap_alloc) {
            int rc;
            if ((rc = dev_alloc(b, &b->d_sp_times, static_cast<size_t>(b->n_env) * cap))) return rc;
            if ((rc = dev_alloc(b, &b->d_sp_ring, static_cast<size_t>(b->n_env) * cap * std::max(b->width, 1)))) return rc;
            b->sp_cap_alloc = cap;
        }
        CU(cudaMemcpyAsync(b->d_sdesc, b->sdesc.data(), sizeof(SensorDesc) * ns, cudaMemcpyHostToDevice, b->stream));
        CU(cudaStreamSynchronize(b->stream));
        kp.sp_on = 1; kp.sp_cap = cap; kp.sp_nsens = ns; kp.sp_desc = b->d_sdesc;
        kp.sp_rng = b->d_sp_rng; kp.sp_rng_init = b->d_sp_rng_init; kp.sp_snap_rng = b->d_sp_snap_rng;
        kp.sp_count = b->d_sp_count; kp.sp_snap_count = b->d_sp_snap_count; kp.sp_times = b->d_sp_times; kp.sp_ring = b->d_sp_ring;
        b->sp_dirty = false;
    }
    // Start states of the generators: Engine::reset seeds the engine's PCG32 from stepper.randomSeedSeq (engine.cc:756-757),
    // Robot::reset draws one seed per sensor type (robot.cc:137-144; fixed type order Imu, Force, Encoder, Effort, Contact here,
    // the reference iterates an unordered_map), resetAll expands it with a seed_seq into one seed per sensor
    // (abstract_sensor.hxx:213-226) and PCG32(seed) sets state = seed | 3 (random.cc:10-13).
    if (b->seeds.empty()) b->seeds.assign(b->n_env, 0u);
    std::vector<unsigned long long> init(static_cast<size_t>(b->n_env) * ns, 0ULL);
    const int counts[5] = {kp.nimu, kp.nforce, kp.nenc, kp.neff, kp.ncs};
    for (int e = 0; e < b->n_env; ++e) {
        if (mask && !mask[e]) continue;
        std::seed_seq seq{b->seeds[e]};
        uint32_t buf[2];
        seq.generate(buf, buf + 2);
        unsigned long long st = (static_cast<unsigned long long>(buf[0]) | (static_cast<unsigned long long>(buf[1]) << 32)) | 3ULL;
        size_t col = 0;
        for (int ty = 0; ty < 5; ++ty) {
            if (!counts[ty]) continue;
            st *= 6364136223846793005ULL;
            unsigned long long sx = st;
            const unsigned rshift = static_cast<unsigned>(sx >> 61) & 7u;
            sx ^= sx >> 22;
            const uint32_t type_seed = static_cast<uint32_t>(sx >> (22 + rshift));
            std::seed_seq tseq{type_seed};
            std::vector<uint32_t> sub(counts[ty]);
            tseq.generate(sub.begin(), sub.end());
            for (int k = 0; k < counts[ty]; ++k) init[static_cast<size_t>(e) * ns + col++] = static_cast<unsigned long long>(sub[k]) | 3ULL;
        }
    }
    if (mask) {
        // rows of the envs that are not restarted keep what the device holds
        for (int e = 0; e < b->n_env; ++e)
            if (mask[e]) CU(cudaMemcpyAsync(b->d_sp_rng_init + static_cast<size_t>(e) * ns, init.data() + static_cast<size_t>(e) * ns, sizeof(unsigned long long) * ns, cudaMemcpyHostToDevice, b->stream));
    } else CU(cudaMemcpyAsync(b->d_sp_rng_init, init.data(), sizeof(unsigned long long) * init.size(), cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

__global__ void gather_true_sensors_kernel(const double* __restrict__ ring, const int32_t* __restrict__ count, double* __restrict__ out,
                                           int n_env, int cap, int width) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i >= static_cast<size_t>(n_env) * width) return;
    const size_t env = i / width, k = i % width;
    out[i] = ring[(env * cap + count[env * 6]) * width + k];
}

int jb_get_sensor_data(JbBatch* b, double* out) {
    if (!b || !out) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->kp.sp_on) return jb_get_sensors(b, out);
    CU(cudaSetDevice(b->device));
    const size_t total = static_cast<size_t>(b->n_env) * b->width;
    if (!total) return JB_OK;
    if (!b->d_sens_true) { int rc = dev_alloc(b, &b->d_sens_true, total); if (rc) return rc; }
    JB_LAUNCH(gather_true_sensors_kernel, static_cast<unsigned>((total + 255) / 256), 256, 0, b->stream, b->d_sp_ring, b->d_sp_count, b->d_sens_true,
              b->n_env, b->kp.sp_cap, b->width);
    CU(cudaGetLastError());
    ++b->launches;
    CU(cudaMemcpyAsync(out, b->d_sens_true, total * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_start(JbBatch* b, const uint8_t* mask, const double* q0, const double* v0) {
    if (!b || !q0 || !v0) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    // Engine::start input validation (engine.cc:1007-1037)
    for (int i = 0; i < b->n_env; ++i) {
        if (mask && !mask[i]) continue;
        for (int k = 0; k < b->nq; ++k) {
            const double x = q0[static_cast<size_t>(i) * b->nq + k];
            if (!(x == x)) return fail(JB_ERR_INVALID_ARGUMENT, "Initial configuration contains NaN (env " + std::to_string(i) + ").");
            if (2.220446049250313e-16 < x - b->q_upper[k] || 2.220446049250313e-16 < b->q_lower[k] - x)
                return fail(JB_ERR_INVALID_ARGUMENT, "Initial configuration out-of-bounds (env " + std::to_string(i) + ").");
        }
        for (int k = 0; k < b->nv; ++k) {
            const double x = v0[static_cast<size_t>(i) * b->nv + k];
            if (!(x == x)) return fail(JB_ERR_INVALID_ARGUMENT, "Initial velocity contains NaN (env " + std::to_string(i) + ").");
        }
    }
    CU(cudaMemcpyAsync(b->d_qin, q0, sizeof(double) * b->n_env * b->nq, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(b->d_vin, v0, sizeof(double) * b->n_env * b->nv, cudaMemcpyHostToDevice, b->stream));
    if (mask) CU(cudaMemcpyAsync(b->d_mask, mask, b->n_env, cudaMemcpyHostToDevice, b->stream));
    int rc = prepare_sensor_pipeline(b, mask);
    if (rc) return rc;
    rc = launch(b, MODE_START, 0.0, mask ? b->d_mask : nullptr);
    if (rc) return rc;
    CU(cudaStreamSynchronize(b->stream));
    b->any_started = true;
    return JB_OK;
}

// ---- external forces --------------------------------------------------------------------------
int jb_stop(JbBatch* b) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    std::vector<int32_t> st(b->n_pad, JB_ENV_NOT_STARTED);
    CU(cudaMemcpyAsync(b->d_status, st.data(), st.size() * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    b->any_started = false;
    return JB_OK;
}

static int ext_slot_for(JbBatch* b, int joint, const double* p, int* slot_out) {
    if (joint <= 0 || joint >= b->njoints) return fail(JB_ERR_INVALID_ARGUMENT, "Impossible to apply external forces to the universe itself (or unknown joint).");
    for (size_t e = 0; e < b->eframes.size(); ++e) {
        const auto& f = b->eframes[e];
        if (f.joint == joint && f.p[0] == p[0] && f.p[1] == p[1] && f.p[2] == p[2]) { *slot_out = static_cast<int>(e); return JB_OK; }
    }
    if (b->eframes.size() >= MAX_ESLOT) return fail(JB_ERR_NOT_IMPLEMENTED, "too many distinct frames carrying external forces");
    const Plan& P = b->plan;
    const size_t N = b->n_pad;
    if (!b->d_eslots) {
        int rc;
        if ((rc = dev_alloc(b, &b->d_eslots, static_cast<size_t>(MAX_ESLOT) * P.L))) return rc;
        if ((rc = dev_alloc(b, &b->d_imp, static_cast<size_t>(MAX_IMPULSE) * IMPULSE_ROWS * N))) return rc;
        if ((rc = dev_alloc(b, &b->d_prof_pending, static_cast<size_t>(MAX_PROFILE) * 6 * N))) return rc;
        if ((rc = dev_alloc(b, &b->d_prof_latched, static_cast<size_t>(MAX_PROFILE) * 6 * N))) return rc;
        b->h_imp.assign(static_cast<size_t>(MAX_IMPULSE) * IMPULSE_ROWS * N, 0.0);
        b->kp.eslots = b->d_eslots; b->kp.imp_data = b->d_imp;
        b->kp.prof_pending = b->d_prof_pending; b->kp.prof_latched = b->d_prof_latched;
    }
    const size_t smem = static_cast<size_t>(b->base_fields + ESLOT_SIZE * (b->eframes.size() + 1)) * 32 * sizeof(double);
    if (smem > 227 * 1024) return fail(JB_ERR_NOT_IMPLEMENTED, "no shared memory left for an external-force slot");
    int rc = raise_smem_attr(b->device, smem);
    if (rc) return rc;
    JbBatch::ExtFrame f{joint, {p[0], p[1], p[2]}};
    b->eframes.push_back(f);
    std::vector<ExtSlot> rows(b->eframes.size() * P.L);
    for (size_t e = 0; e < b->eframes.size(); ++e)
        for (int s = 0; s < P.L; ++s) {
            ExtSlot& x = rows[e * P.L + s];
            x.p[0] = b->eframes[e].p[0]; x.p[1] = b->eframes[e].p[1]; x.p[2] = b->eframes[e].p[2];
            x.joint = b->eframes[e].joint; x.rec = -1;
            for (int r = 0; r < P.nrec; ++r) {
                const RecInt& ri = P.rint[static_cast<size_t>(r) * P.L + s];
                if (ri.kind != REC_PAD && ri.joint == x.joint) x.rec = r;
            }
        }
    CU(cudaMemcpyAsync(b->d_eslots, rows.data(), rows.size() * sizeof(ExtSlot), cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    b->smem_bytes = smem;
    b->kp.n_eslot = static_cast<int32_t>(b->eframes.size());
    *slot_out = b->kp.n_eslot - 1;
    return JB_OK;
}

static int upload_impulse(JbBatch* b, int k, const uint8_t* mask, const double* t, const double* dt, const double* wrench) {
    const size_t N = b->n_pad;
    double* rows = b->h_imp.data() + static_cast<size_t>(k) * IMPULSE_ROWS * N;
    for (int i = 0; i < b->n_env; ++i) {
        if (mask && !mask[i]) continue;
        if (dt[i] < 1e-10) return fail(JB_ERR_INVALID_ARGUMENT, "Force duration cannot be smaller than 1e-10s.");
        if (t[i] < 0.0) return fail(JB_ERR_INVALID_ARGUMENT, "Force application time must be positive.");
        rows[i] = t[i]; rows[N + i] = dt[i];
        for (int c = 0; c < 6; ++c) rows[(2 + c) * N + i] = wrench[static_cast<size_t>(i) * 6 + c];
    }
    for (size_t i = b->n_env; i < N; ++i) { rows[i] = rows[b->n_env - 1]; rows[N + i] = rows[N + b->n_env - 1]; }
    CU(cudaMemcpyAsync(b->d_imp + static_cast<size_t>(k) * IMPULSE_ROWS * N, rows, sizeof(double) * IMPULSE_ROWS * N, cudaMemcpyHostToDevice, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_register_impulse_force(JbBatch* b, int32_t joint, const double* frame_translation, const double* t, const double* dt,
                              const double* wrench, int32_t* index_out) {
    if (!b || !frame_translation || !t || !dt || !wrench) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (b->any_started) return fail(JB_ERR_BAD_CONTROL_FLOW, "Simulation already running. Please stop it before registering new forces.");
    if (b->kp.n_imp >= MAX_IMPULSE) return fail(JB_ERR_NOT_IMPLEMENTED, "too many impulse forces");
    CU(cudaSetDevice(b->device));
    int slot = 0;
    int rc = ext_slot_for(b, joint, frame_translation, &slot);
    if (rc) return rc;
    const int k = b->kp.n_imp;
    rc = upload_impulse(b, k, nullptr, t, dt, wrench);
    if (rc) return rc;
    b->kp.imp_slot[k] = slot;
    b->kp.n_imp = k + 1;
    if (index_out) *index_out = k;
    return JB_OK;
}

int jb_set_impulse_force(JbBatch* b, int32_t index, const uint8_t* mask, const double* t, const double* dt, const double* wrench) {
    if (!b || !t || !dt || !wrench) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (index < 0 || index >= b->kp.n_imp) return fail(JB_ERR_INVALID_ARGUMENT, "unknown impulse force");
    CU(cudaSetDevice(b->device));
    return upload_impulse(b, index, mask, t, dt, wrench);
}

int jb_register_profile_force(JbBatch* b, int32_t joint, const double* frame_translation, double update_period, int32_t* slot_out) {
    if (!b || !frame_translation) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (b->any_started) return fail(JB_ERR_BAD_CONTROL_FLOW, "Simulation already running. Please stop it before registering new forces.");
    if (b->kp.n_prof >= MAX_PROFILE) return fail(JB_ERR_NOT_IMPLEMENTED, "too many profile forces");
    if (update_period > 2.3e-16 && update_period < 1e-6)
        return fail(JB_ERR_INVALID_ARGUMENT, "Cannot register external force profile with update period smaller than 1e-06s.");
    if (update_period > 2.3e-16 && b->kp.stepper_update_period < 1e300) {
        const double lo = std::min(update_period, b->kp.stepper_update_period), hi = std::max(update_period, b->kp.stepper_update_period);
        const double r = std::fmod(hi, lo);
        if (std::min(r, lo - r) > 1e-12)
            return fail(JB_ERR_INVALID_ARGUMENT, "In discrete mode, the update period of force profiles and the stepper update period must be multiple of each other.");
    }
    CU(cudaSetDevice(b->device));
    int slot = 0;
    int rc = ext_slot_for(b, joint, frame_translation, &slot);
    if (rc) return rc;
    const int j = b->kp.n_prof;
    b->kp.prof_slot[j] = slot;
    b->kp.prof_period[j] = update_period;
    b->kp.n_prof = j + 1;
    const size_t N = b->n_pad;
    CU(cudaMemsetAsync(b->d_prof_pending + static_cast<size_t>(j) * 6 * N, 0, sizeof(double) * 6 * N, b->stream));
    CU(cudaMemsetAsync(b->d_prof_latched + static_cast<size_t>(j) * 6 * N, 0, sizeof(double) * 6 * N, b->stream));
    const JbOptions o = b->kp.opt;
    apply_options(b, &o);
    if (slot_out) *slot_out = j;
    return JB_OK;
}

int jb_set_profile_force(JbBatch* b, int32_t slot, const double* wrench) {
    if (!b || !wrench) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (slot < 0 || slot >= b->kp.n_prof) return fail(JB_ERR_INVALID_ARGUMENT, "unknown profile force");
    CU(cudaSetDevice(b->device));
    const size_t N = b->n_pad;
    int rc = ensure_host_stage(b, sizeof(double) * 6 * N);
    if (rc) return rc;
    CU(cudaStreamSynchronize(b->stream));   // the staging buffer may still be in flight
    for (int c = 0; c < 6; ++c)
        for (size_t i = 0; i < N; ++i)
            b->h_stage[c * N + i] = wrench[std::min<size_t>(i, b->n_env - 1) * 6 + c];
    CU(cudaMemcpyAsync(b->d_prof_pending + static_cast<size_t>(slot) * 6 * N, b->h_stage, sizeof(double) * 6 * N, cudaMemcpyHostToDevice, b->stream));
    return JB_OK;
}

int jb_remove_all_forces(JbBatch* b) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (b->any_started) return fail(JB_ERR_BAD_CONTROL_FLOW, "Simulation already running. Please stop it before removing forces.");
    b->kp.n_imp = 0; b->kp.n_prof = 0; b->kp.n_eslot = 0;
    b->eframes.clear();
    b->smem_bytes = static_cast<size_t>(b->base_fields) * 32 * sizeof(double);
    const JbOptions o = b->kp.opt;
    apply_options(b, &o);
    return JB_OK;
}

int jb_set_command(JbBatch* b, const double* cmd) {
    if (!b || (!cmd && b->nmotors)) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->nmotors) return JB_OK;
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpyAsync(b->d_cmd, cmd, sizeof(double) * b->n_env * b->nmotors, cudaMemcpyHostToDevice, b->stream));
    return JB_OK;
}

int jb_set_command_device(JbBatch* b, const double* cmd_dev) {
    if (!b || (!cmd_dev && b->nmotors)) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->nmotors) return JB_OK;
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpyAsync(b->d_cmd, cmd_dev, sizeof(double) * b->n_env * b->nmotors, cudaMemcpyDeviceToDevice, b->stream));
    return JB_OK;
}

int jb_step(JbBatch* b, double step_dt) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->any_started) return fail(JB_ERR_BAD_CONTROL_FLOW, "No simulation running. Please start one before using step method.");
    if (step_dt > 2.220446049250313e-16 && step_dt < 1e-6) return fail(JB_ERR_INVALID_ARGUMENT, "Step size out of bounds.");
    CU(cudaSetDevice(b->device));
    return launch(b, MODE_STEP, step_dt);
}

int jb_compute_dynamics(JbBatch* b, const double* q, const double* v, const double* cmd, double* a, double* fext, double* u) {
    if (!b || !q || !v || !a) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpyAsync(b->d_qin, q, sizeof(double) * b->n_env * b->nq, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemcpyAsync(b->d_vin, v, sizeof(double) * b->n_env * b->nv, cudaMemcpyHostToDevice, b->stream));
    // the evaluation must leave the running envs alone: its command goes to a buffer of its own, and the persistent
    // constraint state (a joint outside its bounds in `q` would enable its constraint) is put back afterwards
    if (cmd && b->nmotors) {
        if (!b->d_cmd_dyn) { int rc0 = dev_alloc(b, &b->d_cmd_dyn, static_cast<size_t>(b->n_env) * b->nmotors); if (rc0) return rc0; }
        CU(cudaMemcpyAsync(b->d_cmd_dyn, cmd, sizeof(double) * b->n_env * b->nmotors, cudaMemcpyHostToDevice, b->stream));
    }
    const size_t cs_bytes = b->kp.cons_on ? sizeof(double) * static_cast<size_t>(b->kp.cs_total) * b->n_pad : 0;
    if (cs_bytes) {
        if (!b->d_cstate_save) { int rc0 = dev_alloc(b, &b->d_cstate_save, cs_bytes / sizeof(double)); if (rc0) return rc0; }
        CU(cudaMemcpyAsync(b->d_cstate_save, b->kp.cstate, cs_bytes, cudaMemcpyDeviceToDevice, b->stream));
    }
    int rc = launch(b, MODE_DYNAMICS, 0.0, nullptr, (cmd && b->nmotors) ? b->d_cmd_dyn : nullptr);
    if (rc) return rc;
    if (cs_bytes) CU(cudaMemcpyAsync(b->kp.cstate, b->d_cstate_save, cs_bytes, cudaMemcpyDeviceToDevice, b->stream));
    CU(cudaMemcpyAsync(a, b->d_aout, sizeof(double) * b->n_env * b->nv, cudaMemcpyDeviceToHost, b->stream));
    if (fext) CU(cudaMemcpyAsync(fext, b->d_fext, sizeof(double) * b->n_env * b->njoints * 6, cudaMemcpyDeviceToHost, b->stream));
    if (u) CU(cudaMemcpyAsync(u, b->d_u, sizeof(double) * b->n_env * b->nv, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

static int fetch_soa(JbBatch* b, const double* d_src, int width, double* host_dst) {
    const size_t total = static_cast<size_t>(b->n_env) * width;
    if (!total) return JB_OK;
    JB_LAUNCH(soa_to_aos_kernel, static_cast<unsigned>((total + 255) / 256), 256, 0, b->stream, d_src, b->d_stage, b->n_env, b->n_pad, width);
    CU(cudaGetLastError());
    ++b->launches;
    CU(cudaMemcpyAsync(host_dst, b->d_stage, total * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_get_state(JbBatch* b, double* t, double* q, double* v, double* a) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    int rc;
    if (t) { CU(cudaMemcpyAsync(t, b->d_sched + static_cast<size_t>(SCH_T) * b->n_pad, sizeof(double) * b->n_env, cudaMemcpyDeviceToHost, b->stream)); CU(cudaStreamSynchronize(b->stream)); }
    if (q && (rc = fetch_soa(b, b->d_q, b->nq, q))) return rc;
    if (v && (rc = fetch_soa(b, b->d_v, b->nv, v))) return rc;
    if (a && (rc = fetch_soa(b, b->d_a, b->nv, a))) return rc;
    return JB_OK;
}

static int store_soa(JbBatch* b, const double* host_src, int width, double* d_dst) {
    const size_t total = static_cast<size_t>(b->n_env) * width;
    if (!total) return JB_OK;
    CU(cudaMemcpyAsync(b->d_stage, host_src, total * sizeof(double), cudaMemcpyHostToDevice, b->stream));
    const size_t padded = static_cast<size_t>(b->n_pad) * width;
    JB_LAUNCH(aos_to_soa_kernel, static_cast<unsigned>((padded + 255) / 256), 256, 0, b->stream, b->d_stage, d_dst, b->n_env, b->n_pad, width);
    CU(cudaGetLastError());
    ++b->launches;
    CU(cudaStreamSynchronize(b->stream));   // d_stage and host_src are free again
    return JB_OK;
}

int jb_get_stepper_state(JbBatch* b, double* sched, double* command_held) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    int rc;
    if (sched && (rc = fetch_soa(b, b->d_sched, SCH_N, sched))) return rc;
    if (command_held && b->nmotors) {
        const double* src = (b->kp.pd_gains || b->kp.pdf) ? b->d_cmd_torque : b->d_cmd;
        CU(cudaMemcpyAsync(command_held, src, sizeof(double) * b->n_env * b->nmotors, cudaMemcpyDeviceToHost, b->stream));
        CU(cudaStreamSynchronize(b->stream));
    }
    return JB_OK;
}

int jb_set_stepper_state(JbBatch* b, const double* sched, const double* q, const double* v, const double* a,
                         const int64_t* iter, const int64_t* iter_failed, const double* command_held) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->any_started) return fail(JB_ERR_BAD_CONTROL_FLOW, "No simulation running. Please start one before restoring its state.");
    CU(cudaSetDevice(b->device));
    int rc;
    if (sched && (rc = store_soa(b, sched, SCH_N, b->d_sched))) return rc;
    if (q && (rc = store_soa(b, q, b->nq, b->d_q))) return rc;
    if (v && (rc = store_soa(b, v, b->nv, b->d_v))) return rc;
    if (a && (rc = store_soa(b, a, b->nv, b->d_a))) return rc;
    if (iter) CU(cudaMemcpyAsync(b->d_iters, iter, sizeof(int64_t) * b->n_env, cudaMemcpyHostToDevice, b->stream));
    if (iter_failed) CU(cudaMemcpyAsync(b->d_iters + b->n_pad, iter_failed, sizeof(int64_t) * b->n_env, cudaMemcpyHostToDevice, b->stream));
    if (command_held && b->nmotors) {
        double* dst = (b->kp.pd_gains || b->kp.pdf) ? b->d_cmd_torque : b->d_cmd;
        CU(cudaMemcpyAsync(dst, command_held, sizeof(double) * b->n_env * b->nmotors, cudaMemcpyHostToDevice, b->stream));
    }
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_get_efforts(JbBatch* b, double* u, double* u_motor, double* command, double* fext) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (u) CU(cudaMemcpyAsync(u, b->d_u, sizeof(double) * b->n_env * b->nv, cudaMemcpyDeviceToHost, b->stream));
    if (u_motor && b->nmotors) CU(cudaMemcpyAsync(u_motor, b->d_umotor, sizeof(double) * b->n_env * b->nmotors, cudaMemcpyDeviceToHost, b->stream));
    if (command && b->nmotors) CU(cudaMemcpyAsync(command, b->d_cmd, sizeof(double) * b->n_env * b->nmotors, cudaMemcpyDeviceToHost, b->stream));
    if (fext) CU(cudaMemcpyAsync(fext, b->d_fext, sizeof(double) * b->n_env * b->njoints * 6, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_get_sensors(JbBatch* b, double* out) {
    if (!b || !out) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (b->width) CU(cudaMemcpyAsync(out, b->d_sensors, sizeof(double) * b->n_env * b->width, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return check_peer_timeout(b);
}

int jb_sensor_layout(JbBatch* b, JbSensorLayout* out) {
    if (!b || !out) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    *out = b->kp.lay;
    return JB_OK;
}

int jb_get_extra_terms(JbBatch* b, double* energy, double* joint_a, double* joint_f) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    const size_t nj6 = static_cast<size_t>(b->n_env) * b->njoints * 6;
    if (energy) CU(cudaMemcpyAsync(energy, b->kp.extra_energy, sizeof(double) * 2 * b->n_env, cudaMemcpyDeviceToHost, b->stream));
    if (joint_a) CU(cudaMemcpyAsync(joint_a, b->kp.extra_a, sizeof(double) * nj6, cudaMemcpyDeviceToHost, b->stream));
    if (joint_f) CU(cudaMemcpyAsync(joint_f, b->kp.extra_f, sizeof(double) * nj6, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_get_centroidal(JbBatch* b, double* ycrb, double* com, double* vcom, double* hg, double* dhg) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    const size_t n = b->n_env, nj = b->njoints;
    if (ycrb) CU(cudaMemcpyAsync(ycrb, b->kp.extra_ycrb, sizeof(double) * n * nj * 10, cudaMemcpyDeviceToHost, b->stream));
    if (com) CU(cudaMemcpyAsync(com, b->kp.extra_com, sizeof(double) * n * nj * 3, cudaMemcpyDeviceToHost, b->stream));
    if (vcom) CU(cudaMemcpyAsync(vcom, b->kp.extra_vcom, sizeof(double) * n * nj * 3, cudaMemcpyDeviceToHost, b->stream));
    if (hg) CU(cudaMemcpy2DAsync(hg, 6 * sizeof(double), b->kp.extra_hg, 12 * sizeof(double), 6 * sizeof(double), n, cudaMemcpyDeviceToHost, b->stream));
    if (dhg) CU(cudaMemcpy2DAsync(dhg, 6 * sizeof(double), b->kp.extra_hg + 6, 12 * sizeof(double), 6 * sizeof(double), n, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_get_status(JbBatch* b, int32_t* status) {
    if (!b || !status) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    CU(cudaMemcpyAsync(status, b->d_status, sizeof(int32_t) * b->n_env, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_get_iters(JbBatch* b, int64_t* iter, int64_t* iter_failed) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (iter) CU(cudaMemcpyAsync(iter, b->d_iters, sizeof(int64_t) * b->n_env, cudaMemcpyDeviceToHost, b->stream));
    if (iter_failed) CU(cudaMemcpyAsync(iter_failed, b->d_iters + b->n_pad, sizeof(int64_t) * b->n_env, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
}

int jb_device_views(JbBatch* b, double** sensors_dev, double** qv_dev) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (sensors_dev) *sensors_dev = b->d_sensors;
    if (qv_dev) *qv_dev = b->d_qv;
    return JB_OK;
}

int jb_copy_sensors_device(JbBatch* b, double* dst_dev) {
    if (!b || !dst_dev) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (b->width) CU(cudaMemcpyAsync(dst_dev, b->d_sensors, sizeof(double) * b->n_env * b->width, cudaMemcpyDeviceToDevice, b->stream));
    return JB_OK;
}

// ---- observation exchange over peer memory ----------------------------------------------------------------
int jb_peer_obs_create(JbBatch* b, int32_t world, int32_t rank, uint8_t handle_out[64]) {
#ifdef JB_HOST_EMUL
    return fail(JB_ERR_NOT_IMPLEMENTED, "peer memory needs CUDA devices");
#else
    if (!b || !handle_out) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (world < 2 || world > 8 || rank < 0 || rank >= world) return fail(JB_ERR_INVALID_ARGUMENT, "world must be 2..8 and 0 <= rank < world");
    if (b->d_peer_buf) return fail(JB_ERR_BAD_CONTROL_FLOW, "peer buffer already created");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CU(cudaSetDevice(b->device));
    b->peer_world = world; b->peer_rank = rank;
    b->peer_obs_doubles = static_cast<size_t>(world) * b->n_env * std::max(b->width, 1);
    const size_t bytes = 2 * b->peer_obs_doubles * sizeof(double) + 2 * world * sizeof(long long);
    void* raw = nullptr;
    CU(cudaMalloc(&raw, bytes));          // a dedicated allocation: IPC handles map whole allocations
    CU(cudaMemset(raw, 0, bytes));
    b->allocs.push_back(raw);
    b->d_peer_buf = static_cast<char*>(raw);
    CU(cudaHostAlloc(reinterpret_cast<void**>(&b->h_peer_timeout), sizeof(int), cudaHostAllocMapped));
    *b->h_peer_timeout = 0;
    CU(cudaHostGetDevicePointer(reinterpret_cast<void**>(&b->d_peer_timeout), b->h_peer_timeout, 0));
    if (const char* e = std::getenv("JB_PEER_TIMEOUT_S")) b->peer_timeout_s = std::max(0.01, std::atof(e));
    {   // (queried once: the clock-rate attribute is a slow driver call)
        int khz = 1965000;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, b->device);
        b->peer_timeout_cycles = static_cast<long long>(b->peer_timeout_s * 1e3 * khz);
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, raw));
    std::memcpy(handle_out, &h, 64);
    CU(cudaStreamSynchronize(b->stream));
    return JB_OK;
#endif
}

int jb_peer_obs_connect(JbBatch* b, const uint8_t* handles) {
#ifdef JB_HOST_EMUL
    return fail(JB_ERR_NOT_IMPLEMENTED, "peer memory needs CUDA devices");
#else
    if (!b || !handles) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->d_peer_buf) return fail(JB_ERR_BAD_CONTROL_FLOW, "call jb_peer_obs_create first");
    if (!b->peer_opened.empty()) return fail(JB_ERR_BAD_CONTROL_FLOW, "already connected");
    CU(cudaSetDevice(b->device));
    for (int p = 0; p < b->peer_world; ++p) {
        if (p == b->peer_rank) { b->peer_base[p] = b->d_peer_buf; continue; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, handles + 64 * p, 64);
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return fail(JB_ERR_CUDA, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(p) + "): " + cudaGetErrorString(e));
        b->peer_opened.push_back(ptr);
        b->peer_base[p] = static_cast<char*>(ptr);
    }
    b->kp.peer_n = b->peer_world; b->kp.peer_rank = b->peer_rank;
    const size_t flag_off = 2 * b->peer_obs_doubles * sizeof(double);
    for (int p = 0; p < b->peer_world; ++p) {
        b->kp.peer_obs[p] = reinterpret_cast<double*>(b->peer_base[p]);
        b->kp.peer_flags[p] = reinterpret_cast<long long*>(b->peer_base[p] + flag_off);
    }
    unsigned int* d_counter = nullptr;
    int rc2 = dev_alloc(b, &d_counter, 1);
    if (rc2) return rc2;
    CU(cudaStreamSynchronize(b->stream));
    b->kp.peer_counter = d_counter;
    return JB_OK;
#endif
}

int jb_peer_obs_enable(JbBatch* b, int32_t on) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (b->peer_opened.empty()) return fail(JB_ERR_BAD_CONTROL_FLOW, "not connected (jb_peer_obs_connect)");
    b->peer_enabled = on != 0;
    return JB_OK;
}

int jb_peer_obs_wait(JbBatch* b) {
#ifdef JB_HOST_EMUL
    return fail(JB_ERR_NOT_IMPLEMENTED, "peer memory needs CUDA devices");
#else
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (b->peer_opened.empty() || !b->peer_enabled || b->step_id == 0) return fail(JB_ERR_BAD_CONTROL_FLOW, "no published step to wait for");
    CU(cudaSetDevice(b->device));
    const int parity = static_cast<int>(b->step_id & 1);
    volatile long long* mine = reinterpret_cast<volatile long long*>(b->d_peer_buf + 2 * b->peer_obs_doubles * sizeof(double));
    JB_LAUNCH(peer_wait_kernel, 1, 1, 0, b->stream, mine, b->peer_world, parity, b->step_id, b->peer_timeout_cycles, b->d_peer_timeout);
    CU(cudaGetLastError());
    ++b->launches;
    return JB_OK;
#endif
}

int jb_peer_obs_view(JbBatch* b, double** obs_dev) {
    if (!b || !obs_dev) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    if (!b->d_peer_buf) return fail(JB_ERR_BAD_CONTROL_FLOW, "call jb_peer_obs_create first");
    *obs_dev = reinterpret_cast<double*>(b->d_peer_buf) + static_cast<size_t>(b->step_id & 1) * b->peer_obs_doubles;
    return JB_OK;
}

int jb_get_stream(JbBatch* b, void** stream) {
    if (!b || !stream) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    *stream = b->stream;
    return JB_OK;
}

int64_t jb_launch_count(JbBatch* b) { return b ? b->launches : 0; }

int jb_state_ptrs(JbBatch* b, JbStateViews* host, JbStateViews* device) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    if (host && !b->h_mirror) {
        const size_t nt = b->n_env, nqv = static_cast<size_t>(b->n_env) * (b->nq + b->nv), na = static_cast<size_t>(b->n_env) * b->nv,
                     ns = static_cast<size_t>(b->n_env) * b->width;
        double* h = nullptr;
        CU(cudaMallocHost(reinterpret_cast<void**>(&h), sizeof(double) * (nt + nqv + na + ns + 4)));
        std::memset(h, 0, sizeof(double) * (nt + nqv + na + ns + 4));
        int rc = dev_alloc(b, &b->d_a_aos, std::max<size_t>(na, 1));
        if (rc) { cudaFreeHost(h); return rc; }
        b->h_mirror = h; b->hm_t = h; b->hm_qv = h + nt; b->hm_a = b->hm_qv + nqv; b->hm_sensors = b->hm_a + na;
        if (b->any_started) {
            // a running batch: fill the views with the current state right away
            CU(cudaMemcpyAsync(b->hm_t, b->d_sched + static_cast<size_t>(SCH_T) * b->n_pad, sizeof(double) * b->n_env, cudaMemcpyDeviceToHost, b->stream));
            CU(cudaMemcpyAsync(b->hm_qv, b->d_qv, sizeof(double) * nqv, cudaMemcpyDeviceToHost, b->stream));
            if (na && (rc = fetch_soa(b, b->d_a, b->nv, b->hm_a))) return rc;
            if (ns) CU(cudaMemcpyAsync(b->hm_sensors, b->d_sensors, sizeof(double) * ns, cudaMemcpyDeviceToHost, b->stream));
            CU(cudaStreamSynchronize(b->stream));
        }
    }
    if (host) {
        host->t = b->hm_t; host->qv = b->hm_qv; host->a = b->hm_a; host->sensors = b->hm_sensors;
        host->n_env = b->n_env; host->nq = b->nq; host->nv = b->nv; host->width = b->width;
    }
    if (device) {
        device->t = b->d_sched + static_cast<size_t>(SCH_T) * b->n_pad; device->qv = b->d_qv; device->a = b->d_a_aos; device->sensors = b->d_sensors;
        device->n_env = b->n_env; device->nq = b->nq; device->nv = b->nv; device->width = b->width;
    }
    return JB_OK;
}

#if defined(JB_PROFILE_CLOCKS) && !defined(JB_HOST_EMUL)
// development build only: read and clear the cycle counters of the full body (see jb_device.cuh)
int jb_debug_prof(JbBatch* b, double* out16) {
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    unsigned long long h[16];
    CU(cudaMemcpyFromSymbol(h, jb_prof, sizeof h));
    for (int i = 0; i < 16; ++i) out16[i] = static_cast<double>(h[i]);
    std::memset(h, 0, sizeof h);
    CU(cudaMemcpyToSymbol(jb_prof, h, sizeof h));
    return JB_OK;
}
#endif

int jb_synchronize(JbBatch* b) {
    if (!b) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    return check_peer_timeout(b);
}

// Host-side introspection of the lane planner (no device needed): used by the CPU test-suite.
int jb_plan_describe(const JbModelDesc* m, int32_t lanes, char* buf, int32_t len, int32_t* joint_lane) {
    if (!m || !buf) return fail(JB_ERR_INVALID_ARGUMENT, "null argument");
    try {
        Plan P = build_plan(*m, lanes, 0);
        std::snprintf(buf, len, "%s", P.describe().c_str());
        if (joint_lane) for (int j = 0; j < m->njoints; ++j) joint_lane[j] = P.joint_lane[j];
    } catch (const std::exception& ex) {
        return fail(JB_ERR_INVALID_ARGUMENT, ex.what());
    }
    return JB_OK;
}

}  // extern "C"
