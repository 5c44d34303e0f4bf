// hlynr_capi.cu -- host side of the C ABI declared in include/hlynr.h.
// Owns the SoA state planes, the ring planes and the statistics block of one GPU shard and launches the
// kernels of hlynr_device.cuh.  No torch types: callers pass raw device/host pointers and a stream.
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <thread>
#include <type_traits>
#include <vector>

#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "hlynr_device.cuh"
#include "hlynr_host.cuh"

using namespace hlynr;

static_assert(sizeof(HlynrDoneRecord) == 200, "HlynrDoneRecord is 50 words (mirrored by abi.done_record_numpy_dtype)");

static thread_local char g_err[512] = "";
extern "C" int hlynr_internal_fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}

// Staging memcpys between unpinned caller buffers and the pinned buffers.  A single thread copies ~5-10 GB/s, less than the
// PCIe link moves, so a few persistent helper threads pull 256 KiB blocks off an atomic counter, in address order.  start() is
// asynchronous: hlynr_step_host starts the staging of the WHOLE action array, then waits chunk by chunk (wait_prefix) only
// for the bytes the next host-to-device copy reads, helping with the copy while it waits.
class CopyPool {
  public:
    explicit CopyPool(int helpers) {
        for (int k = 0; k < helpers; ++k) th_.emplace_back([this] { worker(); });
    }
    ~CopyPool() {
        { std::lock_guard<std::mutex> l(m_); stop_ = true; ++gen_; }
        cv_.notify_all();
        for (auto& t : th_) t.join();
    }
    // asynchronous copy; exactly one job at a time: every start() is closed by finish()
    void start(void* dst, const void* src, size_t bytes) {
        const size_t nb = (bytes + kBlock - 1) / kBlock;
        if (flags_.size() < nb) flags_ = std::vector<std::atomic<uint8_t>>(nb);
        for (size_t k = 0; k < nb; ++k) flags_[k].store(0, std::memory_order_relaxed);
        waited_ = 0;
        woke_ = !th_.empty() && bytes >= kParallelMin;
        {
            std::lock_guard<std::mutex> l(m_);
            dst_ = (char*)dst; src_ = (const char*)src; bytes_ = bytes; nblocks_ = nb;
            next_.store(0);
            if (woke_) { busy_ = (int)th_.size(); ++gen_; }
        }
        if (woke_) cv_.notify_all();
    }
    // returns once [0, upto) of the job has been copied
    void wait_prefix(size_t upto) {
        const size_t need = upto >= bytes_ ? nblocks_ : upto / kBlock + (upto % kBlock ? 1 : 0);
        while (next_.load(std::memory_order_relaxed) < need) {
            const size_t b = next_.fetch_add(1);
            if (b >= nblocks_) break;
            copy_block(b);
        }
        for (; waited_ < need; ++waited_)
            while (!flags_[waited_].load(std::memory_order_acquire)) std::this_thread::yield();
    }
    void finish() {
        wait_prefix(bytes_);
        if (woke_) {  // the helpers must be parked again before the job description changes
            std::unique_lock<std::mutex> l(m_);
            done_.wait(l, [this] { return busy_ == 0; });
            woke_ = false;
        }
    }
    void copy(void* dst, const void* src, size_t bytes) {
        if (bytes < kParallelMin || th_.empty()) { memcpy(dst, src, bytes); return; }
        start(dst, src, bytes);
        finish();
    }

  private:
    static constexpr size_t kBlock = size_t(256) << 10;
    static constexpr size_t kParallelMin = size_t(1) << 20;
    // The destination is a pinned buffer the copy engine reads next (or a caller buffer nobody reads soon): streaming stores
    // keep it out of the CPU caches, so there is no read-for-ownership traffic and the DMA read is served from DRAM instead
    // of snooping dirty lines -- measured: a cached memcpy running next to the transfers slows the PCIe DMA itself.
    static void stream_copy(char* dst, const char* src, size_t bytes) {
#if defined(__x86_64__)
        if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
            const size_t vec = bytes / 64;
            for (size_t k = 0; k < vec; ++k) {
                const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 4 * k);
                const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 4 * k + 1);
                const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 4 * k + 2);
                const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 4 * k + 3);
                _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 4 * k, a);
                _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 4 * k + 1, b);
                _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 4 * k + 2, c);
                _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 4 * k + 3, d);
            }
            if (bytes % 64) memcpy(dst + vec * 64, src + vec * 64, bytes % 64);
            _mm_sfence();
            return;
        }
#endif
        memcpy(dst, src, bytes);
    }
    void copy_block(size_t b) {
        const size_t off = b * kBlock;
        stream_copy(dst_ + off, src_ + off, bytes_ - off < kBlock ? bytes_ - off : kBlock);
        flags_[b].store(1, std::memory_order_release);
    }
    void worker() {
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> l(m_);
                cv_.wait(l, [&] { return gen_ != seen; });
                seen = gen_;
                if (stop_) return;
            }
            for (;;) {
                const size_t b = next_.fetch_add(1);
                if (b >= nblocks_) break;
                copy_block(b);
            }
            { std::lock_guard<std::mutex> l(m_); --busy_; }
            done_.notify_one();
        }
    }
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    std::atomic<size_t> next_{0};
    std::vector<std::atomic<uint8_t>> flags_;
    char* dst_ = nullptr; const char* src_ = nullptr; size_t bytes_ = 0, nblocks_ = 0, waited_ = 0;
    int busy_ = 0; uint64_t gen_ = 0; bool stop_ = false, woke_ = false;
};

#define HLYNR_HOST_STREAMS 3
#define HLYNR_DONE_PREFIX 4096  // records fetched together with the count; the rest (rare) in a second copy

// The fields of HlynrInfoSoA (include/hlynr.h): X(name, element type, elements per env).
#define HLYNR_INFO_FIELDS(X)                                                                                                       \
    X(distance, float, 1) X(min_distance, float, 1) X(fuel_remaining, float, 1) X(fuel_used, float, 1) X(steps, int32_t, 1)        \
    X(flags, uint8_t, 1) X(interceptor_pos, float, 3) X(missile_pos, float, 3) X(episode_return, float, 1)                          \
    X(episode_length, int32_t, 1) X(missiles_intercepted, int32_t, 1) X(missiles_remaining, int32_t, 1)                             \
    X(missile_min_distances, float, HLYNR_MAX_VOLLEY) X(radar_quality, float, 1)
#define X(name, type, per_env) +1
static_assert(sizeof(HlynrInfoSoA) == (0 HLYNR_INFO_FIELDS(X)) * sizeof(void*), "every field of HlynrInfoSoA is in HLYNR_INFO_FIELDS");
#undef X

struct HostIO {  // pinned host + device staging for the *_host entry points
    PinnedPtr<float> h_actions, h_obs, h_reward;
    PinnedPtr<uint8_t> h_term, h_trunc, h_mask;
    DevPtr<float> d_actions, d_obs;
    DevPtr<uint8_t> d_mask;
#define X(name, type, per_env) DevPtr<type> info_##name;
    HLYNR_INFO_FIELDS(X)
#undef X
    HlynrInfoSoA d_info{};   // the info_* arrays
    DevPtr<HlynrDoneRecord> d_records;                // capacity n
    PinnedPtr<HlynrDoneRecord> h_records_ab[2];       // two host buffers: the records of a call survive the next call
    HlynrDoneRecord* h_records = nullptr;             // not owned: h_records_ab[call parity]
    PinnedPtr<uint8_t> h_done;                        // terminated | truncated, written by the kernel
    uint32_t calls = 0;
    DevPtr<int32_t> d_counter;
    PinnedPtr<int32_t> h_count;
    int32_t last_count = 0;
    StreamOwner streams[HLYNR_HOST_STREAMS];
    EventOwner ev_start, ev_done[HLYNR_HOST_STREAMS];
    std::unique_ptr<CopyPool> pool;
    bool ready = false, info_ready = false;
};

template <typename R> struct CurBlock {
    unsigned long long num_timesteps;
    KCurriculum<R> slot;
};

struct hlynr_sim {
    HlynrParams params;
    HlynrCurriculum cur;
    int64_t n = 0, n_pad = 0, env_offset = 0;
    int device = 0, precision = HLYNR_FP32;
    uint64_t seed = 0;
    uint64_t tick = 0;  // 64-bit: ring rows are tick % ring_len with lengths that are not powers of two, so the counter must never wrap
    int64_t launches = 0;
    double env_steps = 0.0;
    int specialise = 1;      // use the feature-specialised instantiations when the configuration matches one
    int sm_count = 148;  // ticks simulated since the statistics were last zeroed (n per launch tick)
    DevPtr<char> state_mem;
    StatePlanes<float> pf;
    StatePlanes<double> pd;
    DevPtr<double> stats;          // [HLYNR_STAT_SLOTS + 1][HLYNR_STATS_WORDS]; last row = reduced block
    DevPtr<HlynrEnvState> xchg;    // device staging for export/import
    int64_t xchg_cap = 0;
    HostIO hio;
    int host_info = 1, host_chunks = 0, host_threads = 0;
    int host_chunk_growth = 12;   // geometric chunk schedule of the host path, x1.5 per chunk (measured best on B200: 2.43 -> 2.35 ms at 2^20 envs, 26-D)
    int compact = 0;   // compact plane layout (fp32 build, cfg4 feature set): the counters ride in r6.w / f1.w and the i0 plane is unused
    int pdl = 1;   // step kernels are launched with programmatic stream serialization (option "pdl"; -1.5 us per launch on B200)
    int obs_dim = HLYNR_OBS_DIM;  // row pitch of every observation array of the API: 26, or 17 (option "obs_dim")
    int prefetch_waves = 1;  // CTAs per SM the step kernel looks ahead when it prefetches upcoming planes into L2 (0 = off)
    HlynrDoneRecord* done_records = nullptr;  // not owned: the caller's compact done list (hlynr_set_done_list)
    int32_t* done_counter = nullptr;          // not owned: its counter
    int32_t done_cap = 0;
    uint8_t* io_done = nullptr;   // not owned: set by hlynr_step_host for the duration of the call
    uint8_t* host_done = nullptr; // not owned: caller's page-locked `dones` buffer (hlynr_host_done_buffer), NULL = the handle's own
    // attached curriculum schedule (hlynr_attach_curriculum): a CurBlock<R>, sized for R = double, allocated on first attach
    DevPtr<CurBlock<double>> cur_block;
    bool cur_attached = false;
    HlynrCurriculumSchedule sched;
    int64_t cur_increment = 0;
};

// Calls f with the state planes of the handle's precision, s->pf or s->pd: the one place the precision picks the instantiations.
// f is a generic lambda; real_of<decltype(planes)> names its R.
template <class F> static auto with_planes(hlynr_sim* s, F&& f) {
    if (s->precision == HLYNR_FP32) return f(s->pf);
    return f(s->pd);
}
template <class P> struct PlanesReal;
template <class R> struct PlanesReal<StatePlanes<R>> { using type = R; };
template <class P> using real_of = typename PlanesReal<std::decay_t<P>>::type;
// with_planes plus the handle's plane layout as std::integral_constant<int, C>, C = s->compact (0 wide, 1 compact, 2 DR-compact;
// the compact layouts exist in the fp32 build only): the instantiations of the snapshot kernels.
template <class F> static void with_layout(hlynr_sim* s, F&& f) {
    if (s->precision != HLYNR_FP32) f(s->pd, std::integral_constant<int, 0>{});
    else if (s->compact == 1) f(s->pf, std::integral_constant<int, 1>{});
    else if (s->compact == 2) f(s->pf, std::integral_constant<int, 2>{});
    else f(s->pf, std::integral_constant<int, 0>{});
}

// ------------------------------------------------------------------------------------------------
// parameter conversion
// ------------------------------------------------------------------------------------------------
template <typename R> static KParams<R> make_kparams(const HlynrParams& p) {
    KParams<R> k;
    memset(&k, 0, sizeof(k));
    const R dt_r = (R)p.dt, tau_r = (R)p.thrust_tau;
    k.dt = dt_r; k.dt_d = p.dt; k.tau = tau_r;
    k.rc_dt = (R)(1.0 / (double)dt_r);               // RN(1/dt) for the Markstein constant division
    k.dt_over_tau = (R)((double)dt_r / (double)tau_r);
    k.isa_expo = (R)(9.80665 / (287.05 * 0.0065));   // physics_models.py:99
    k.gas_R = (R)287.05; k.gamma_R = (R)(1.4 * 287.05);
    k.sub_mach = (R)p.sub_mach; k.sup_mach = (R)p.sup_mach; k.sup_minus_sub = (R)(p.sup_mach - p.sub_mach);
    k.peak_minus1 = (R)(p.peak_mult - 1.0);
    k.cd_base = (R)0.3; k.cd_sup = (R)(0.3 * p.sup_mult); k.sup_mult_d = p.sup_mult;
    k.missile_ratio = (R)((0.3 * 1.5) / 0.3);        // environment.py:1090,1095
    k.rho_weak = (R)1.225; k.cs_weak = (R)343.0; k.half_rho_weak = (R)(0.5 * 1.225); k.nhcr_weak = (R)(-0.5 * 0.3 * 1.225);
    k.blh = (R)p.blh; k.rc_blh = (R)(1.0 / p.blh); k.pf_top = (R)pow(p.blh / 10.0, 0.143);
    k.ti_low = (R)(p.turb_intensity * 2.0); k.ti_high = (R)(p.turb_intensity * 0.3); k.turb = (R)p.turb_intensity;
    k.lp = (R)(1.0 - exp(-p.dt / 0.1));
    k.gust_scale_d = p.gust_scale; k.wind_var = (R)p.wind_variability;
    k.kill_radius = (R)p.kill_radius; k.target_x = (R)p.target[0]; k.target_y = (R)p.target[1];
    for (int i = 0; i < 3; ++i) {
        k.base_wind[i] = (R)p.base_wind[i]; k.gpos[i] = (float)p.ground_pos[i]; k.target_d[i] = p.target[i];
        k.m_pos_lo[i] = p.m_pos_lo[i]; k.m_pos_hi[i] = p.m_pos_hi[i]; k.i_pos_lo[i] = p.i_pos_lo[i]; k.i_pos_hi[i] = p.i_pos_hi[i];
        k.i_vel_lo[i] = p.i_vel_lo[i]; k.i_vel_hi[i] = p.i_vel_hi[i];
    }
    k.radar_range = (float)p.radar_range; k.rc_radar_range = (float)(1.0 / p.radar_range);
    k.radar_quality = (float)p.radar_quality; k.radar_quality_d = p.radar_quality;
    k.rc_max_velocity_f = (float)(1.0 / p.max_velocity); k.rc_max_range_f = (float)(1.0 / p.max_range);
    k.max_velocity_f = (float)p.max_velocity; k.max_range_f = (float)p.max_range;
    k.g_max_range = (float)p.g_max_range; k.rc_g_max_range = (float)(1.0 / p.g_max_range);
    // elevation gates asin(s) < min_el / > max_el (core.py:402-406) as thresholds on s itself
    k.g_sin_min_el = (float)sin(p.g_min_el); k.g_sin_max_el = (float)sin(p.g_max_el);
    k.g_base_q = (float)p.g_base_quality; k.max_link = (float)p.max_datalink_range; k.rc_max_link = (float)(1.0 / p.max_datalink_range);
    k.pkt_loss = (float)p.datalink_packet_loss;
    k.dtf = (float)p.dt;
    const double q = 25.0;  // process_noise 5.0 squared (core.py:331-335)
    k.q_pp = (float)(q * pow(p.dt, 4) / 4); k.q_pv = (float)(q * pow(p.dt, 3) / 2); k.q_vv = (float)(q * p.dt * p.dt);
    k.sigma_r = (R)p.g_sigma_r; k.sigma_v = (R)p.g_sigma_v;
    k.rc_max_range_w = (R)(1.0 / p.max_range); k.rc_max_velocity_w = (R)(1.0 / p.max_velocity);
    k.fus_035q = (float)(0.35 * p.radar_quality);
    k.m_speed_lo = p.m_speed_lo; k.m_speed_hi = p.m_speed_hi; k.m_radius_lo = p.m_radius_lo; k.m_radius_hi = p.m_radius_hi;
    k.m_az_lo = p.m_az_lo; k.m_az_hi = p.m_az_hi; k.m_el_lo = p.m_el_lo; k.m_el_hi = p.m_el_hi;
    k.i_speed_lo = p.i_speed_lo; k.i_speed_hi = p.i_speed_hi;
    for (int i = 0; i < HLYNR_N_DR; ++i) k.dr_var[i] = p.dr_variation[i];
    k.max_steps = p.max_steps; k.isa = p.isa_enabled; k.mach = p.mach_enabled; k.enh_wind = p.enh_wind_enabled;
    k.thrust_dyn = p.thrust_dyn_enabled; k.dr = p.dr_enabled; k.validate = p.validate_enabled; k.evasion = p.evasion_enabled;
    k.onboard_delay = p.onboard_delay; k.ground = p.ground_enabled; k.ground_delay = p.ground_enabled ? p.ground_delay : 0;
    k.spherical = p.m_spawn_spherical; k.toward_missile = p.i_vel_toward_missile; k.obs_mode = p.obs_mode;
    k.precision_mode = p.precision_mode; k.fuze = p.fuze_enabled; k.volley_k = p.volley_size;
    k.onb_ring_len = p.onboard_delay > 0 ? (p.dr_enabled ? HLYNR_MAX_ONBOARD_DELAY + 1 : p.onboard_delay + 1) : 0;
    k.gnd_ring_len = k.ground_delay > 0 ? k.ground_delay + 1 : 0;
    return k;
}
template <typename R> static KCurriculum<R> make_kcur(const HlynrCurriculum& c) {
    KCurriculum<R> k;
    k.intercept_radius = (R)c.intercept_radius;
    // beam gate acos(clip(c)) > np.radians(width / 2) (core.py:547-553)  <=>  c < cos(radians(width / 2))
    const double hb = (c.beam_width_deg / 2.0) * (M_PI / 180.0);
    k.cos_half_beam = hb >= M_PI ? -2.0f : (float)cos(hb);
    k.onboard_rel = (float)c.onboard_reliability; k.ground_rel = (float)c.ground_reliability;
    return k;
}
// ---- the curriculum schedule on the device --------------------------------------------------------------------------------
// config.Curriculum in double, operation by operation: the explicit _rn intrinsics keep nvcc from contracting a*(1-t) + b*t into
// an FMA, which would round once where Python rounds twice.  Counts are exact in double below 2^53, as in Python.
__device__ double ramp_dev(double c, double start, double end, double a, double b) {   // Curriculum._ramp
    if (c < start) return a;
    if (c >= end) return b;
    const double t = __ddiv_rn(__dsub_rn(c, start), __dsub_rn(end, start));
    return __dadd_rn(__dmul_rn(a, __dsub_rn(1.0, t)), __dmul_rn(b, t));
}
template <typename R> __device__ KCurriculum<R> kcur_at(const HlynrCurriculumSchedule& s, unsigned long long count) {
    const double c = (double)count;
    double radius = s.final_radius, beam = s.beam_initial, onb = s.onboard_initial, gnd = s.ground_initial;
    if (s.enabled) {   // Curriculum.intercept_radius
        double progress = __ddiv_rn(c, s.curriculum_steps);
        if (!(progress < 1.0)) progress = 1.0;   // Python min(1.0, x)
        radius = __dadd_rn(__dmul_rn(s.initial_radius, __dsub_rn(1.0, progress)), __dmul_rn(s.final_radius, progress));
    }
    if (s.radar_enabled) {   // Curriculum.set_training_step_count
        beam = ramp_dev(c, s.beam_start, s.beam_end, s.beam_initial, s.beam_final);
        onb = ramp_dev(c, s.onboard_start, s.onboard_end, s.onboard_initial, s.onboard_final);
        gnd = ramp_dev(c, s.ground_start, s.ground_end, s.ground_initial, s.ground_final);
    }
    KCurriculum<R> k;   // make_kcur
    k.intercept_radius = (R)radius;
    const double hb = __dmul_rn(__ddiv_rn(beam, 2.0), M_PI / 180.0);
    k.cos_half_beam = hb >= M_PI ? -2.0f : (float)cos(hb);
    k.onboard_rel = (float)onb; k.ground_rel = (float)gnd;
    return k;
}
// Launched by hlynr_step before the step kernel (increment = the run's env count) and by hlynr_reset before the reset kernel
// (increment 0), always WITHOUT programmatic serialization: it starts only once the previous kernel of the stream, which may be a
// step kernel still reading the slot, has completed.  It lets the next launch be scheduled at once; that launch reads the slot
// only after its griddepcontrol.wait, i.e. after this kernel has completed and its stores are visible (DESIGN section 15).
template <typename R> __global__ void curriculum_tick_kernel(CurBlock<R>* b, const HlynrCurriculumSchedule s, unsigned long long increment) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const unsigned long long c = b->num_timesteps;
#ifdef HLYNR_CURRICULUM_TICK_DELAY_NS
    // test hook, off in every ordinary build (tools/build_variant.py <tag> -DHLYNR_CURRICULUM_TICK_DELAY_NS=20000): holds the stores back
    // so that a step kernel reading the slot before its griddepcontrol.wait would see the previous tick's values (DESIGN section 15)
    for (int k = 0; k < HLYNR_CURRICULUM_TICK_DELAY_NS / 1000; ++k) __nanosleep(1000);
#endif
    b->slot = kcur_at<R>(s, c);
    b->num_timesteps = c + increment;
}
template <typename R> __global__ void curriculum_probe_kernel(const HlynrCurriculumSchedule s, unsigned long long count, double* out) {
    const KCurriculum<R> k = kcur_at<R>(s, count);
    out[0] = (double)k.intercept_radius; out[1] = (double)k.cos_half_beam; out[2] = (double)k.onboard_rel; out[3] = (double)k.ground_rel;
}
__global__ void set_timesteps_kernel(unsigned long long* count, unsigned long long value) { *count = value; }

static RoundKeys make_round_keys(uint64_t seed) {
    RoundKeys rk;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) { rk.k[2 * r] = k0; rk.k[2 * r + 1] = k1; k0 += HLYNR_PHILOX_W0; k1 += HLYNR_PHILOX_W1; }
    return rk;
}

// ------------------------------------------------------------------------------------------------
// small utility kernels
// ------------------------------------------------------------------------------------------------
template <typename R> __global__ void init_kernel(StatePlanes<R> s, int64_t n_pad, float peak, int compact) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    Vec4<R> z{R(0), R(0), R(0), R(0)};
    for (int k = 0; k < 6; ++k) s.r[k][i] = z;
    s.r[6][i] = Vec4<R>{R(0), R(0), R(0), R(288.15)};  // SEA_LEVEL_TEMPERATURE, physics_models.py:22
    s.f[0][i] = make_float4(1.f, 0.f, 0.f, 0.f);
    s.f[1][i] = make_float4(0.f, 0.f, 0.f, 0.3f);        // wind, base Cd
    s.f[2][i] = make_float4(0.f, 0.f, 1000.f, 1000.f);   // Kalman P_pv, P_vp, P_vv, P_pp
    s.f[3][i] = make_float4(peak, 0.f, 0.f, 0.f);
    s.i0[i] = make_int4(0, 0, 0, -1);  // episode -1: the first reset starts episode 0
    if (compact == 2) s.i0[i] = make_int4(0, __float_as_int(peak), 0, -1);   // DR-compact: the drag peak rides in i0.y
    if (compact == 1) {   // the same counters in the compact layout (hlynr_device.cuh load_env): steps = worsen = 0, episode = -1, flags = 0
        s.r[6][i] = Vec4<R>{R(0), R(0), R(0), bits_word(0, R(0))};
        s.f[1][i] = make_float4(0.f, 0.f, 0.f, __int_as_float(0x1ffffff));
    }
}

// [SLOTS+1][WORDS]: last row = sum of the slots; word 12 (ticks simulated) is known on the host
__global__ void stats_reduce_kernel(double* stats, double env_steps) {
    int k = threadIdx.x;
    if (k >= HLYNR_STATS_WORDS) return;
    double s = 0.0;
    for (int j = 0; j < HLYNR_STAT_SLOTS; ++j) s += stats[j * HLYNR_STATS_WORDS + k];
    stats[HLYNR_STAT_SLOTS * HLYNR_STATS_WORDS + k] = (k == 12) ? env_steps : s;
}

template <typename R> __global__ void export_kernel(KernelArgs<R> A, int64_t first, int64_t count, HlynrEnvState* out) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    Env<R> e;
    // the optional planes are always allocated and initialised, so read them unconditionally here
    KernelArgs<R> B = A;
    B.P.thrust_dyn = 1; B.P.dr = 1;
    load_env(B, first + j, e);
    HlynrEnvState s;
    memset(&s, 0, sizeof(s));
    s.ipos[0] = e.ipx; s.ipos[1] = e.ipy; s.ipos[2] = e.ipz; s.ivel[0] = e.ivx; s.ivel[1] = e.ivy; s.ivel[2] = e.ivz;
    s.quat[0] = e.qw; s.quat[1] = e.qx; s.quat[2] = e.qy; s.quat[3] = e.qz; s.fuel = e.fuel; s.fuel_used = e.fuel_used;
    s.mpos[0] = e.mpx; s.mpos[1] = e.mpy; s.mpos[2] = e.mpz; s.mvel[0] = e.mvx; s.mvel[1] = e.mvy; s.mvel[2] = e.mvz;
    s.wind[0] = e.wx; s.wind[1] = e.wy; s.wind[2] = e.wz; s.thrust[0] = e.thx; s.thrust[1] = e.thy; s.thrust[2] = e.thz;
    s.prev_d = e.prev_d; s.last_d = e.last_d; s.min_d = e.min_d; s.episode_return = e.ep_ret;
    s.kf_x[0] = e.kpx; s.kf_x[1] = e.kpy; s.kf_x[2] = e.kpz; s.kf_x[3] = e.kvx; s.kf_x[4] = e.kvy; s.kf_x[5] = e.kvz;
    s.kf_P[0] = e.Ppp; s.kf_P[1] = e.Ppv; s.kf_P[2] = e.Pvp; s.kf_P[3] = e.Pvv;
    s.T0 = e.T0; s.base_cd = e.base_cd; s.peak = e.peak;
    s.steps = e.steps; s.worsen_count = e.worsen; s.crossed = (e.flags & FLAG_CROSSED) ? 1 : 0;
    s.kf_init = (e.flags & FLAG_KF_INIT) ? 1 : 0; s.onboard_delay = A.P.onboard_delay > 0 ? FLAG_ODELAY(e.flags) : 0; s.episode = e.episode;
    for (int m = 0; m < A.P.volley_k; ++m) {
        const Vec4<R> a = A.st.vm[(int64_t)(2 * m) * A.ring_stride + first + j], b = A.st.vm[(int64_t)(2 * m + 1) * A.ring_stride + first + j];
        s.vpos[3 * m] = a.x; s.vpos[3 * m + 1] = a.y; s.vpos[3 * m + 2] = a.z; s.vmin[m] = a.w;
        s.vvel[3 * m] = b.x; s.vvel[3 * m + 1] = b.y; s.vvel[3 * m + 2] = b.z; s.vactive[m] = b.w != R(0) ? 1 : 0;
    }
    s.vcur = A.P.volley_k > 0 ? FLAG_VCUR(e.flags) : 0; s.vcount = A.P.volley_k > 0 ? FLAG_VCOUNT(e.flags) : 0;
    s.kf_f64 = (e.flags & FLAG_KF_F64) ? 1 : 0;
    out[j] = s;
}
template <typename R> __global__ void import_kernel(KernelArgs<R> A, int64_t first, int64_t count, const HlynrEnvState* in) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const HlynrEnvState s = in[j];
    Env<R> e;
    e.ipx = (R)s.ipos[0]; e.ipy = (R)s.ipos[1]; e.ipz = (R)s.ipos[2]; e.ivx = (R)s.ivel[0]; e.ivy = (R)s.ivel[1]; e.ivz = (R)s.ivel[2];
    e.qw = (float)s.quat[0]; e.qx = (float)s.quat[1]; e.qy = (float)s.quat[2]; e.qz = (float)s.quat[3];
    e.fuel = (R)s.fuel; e.fuel_used = (R)s.fuel_used;
    e.mpx = (R)s.mpos[0]; e.mpy = (R)s.mpos[1]; e.mpz = (R)s.mpos[2]; e.mvx = (R)s.mvel[0]; e.mvy = (R)s.mvel[1]; e.mvz = (R)s.mvel[2];
    e.wx = (float)s.wind[0]; e.wy = (float)s.wind[1]; e.wz = (float)s.wind[2];
    e.thx = (R)s.thrust[0]; e.thy = (R)s.thrust[1]; e.thz = (R)s.thrust[2];
    e.prev_d = (R)s.prev_d; e.last_d = (R)s.last_d; e.min_d = (R)s.min_d; e.ep_ret = (R)s.episode_return;
    e.kpx = (R)s.kf_x[0]; e.kpy = (R)s.kf_x[1]; e.kpz = (R)s.kf_x[2]; e.kvx = (R)s.kf_x[3]; e.kvy = (R)s.kf_x[4]; e.kvz = (R)s.kf_x[5];
    e.Ppp = (float)s.kf_P[0]; e.Ppv = (float)s.kf_P[1]; e.Pvp = (float)s.kf_P[2]; e.Pvv = (float)s.kf_P[3];
    e.T0 = (R)s.T0; e.base_cd = (float)s.base_cd; e.peak = (float)s.peak;
    e.steps = s.steps; e.worsen = s.worsen_count;
    e.flags = (s.crossed ? FLAG_CROSSED : 0) | (s.kf_init ? FLAG_KF_INIT : 0) | (s.kf_f64 ? FLAG_KF_F64 : 0) | ((s.onboard_delay & 0xf) << 8) | ((s.vcur & 0x7) << 12) |
              ((s.vcount & 0xf) << 16);
    for (int m = 0; m < A.P.volley_k; ++m) {
        A.st.vm[(int64_t)(2 * m) * A.ring_stride + first + j] = Vec4<R>{(R)s.vpos[3 * m], (R)s.vpos[3 * m + 1], (R)s.vpos[3 * m + 2], (R)s.vmin[m]};
        A.st.vm[(int64_t)(2 * m + 1) * A.ring_stride + first + j] = Vec4<R>{(R)s.vvel[3 * m], (R)s.vvel[3 * m + 1], (R)s.vvel[3 * m + 2], s.vactive[m] ? R(1) : R(0)};
    }
    e.episode = s.episode;
    KernelArgs<R> B = A;
    B.P.thrust_dyn = 1; B.P.dr = 1;
    store_env(B, first + j, e);
}

// ---- snapshots (include/hlynr.h): the canonical image <-> the state planes ----------------------------------------------------
// Columns of the image (the section list of hlynr.h), n envs each.
template <typename R> struct SnapImage {
    R* real;
    int32_t* ints;
    R* onb;
    R* gnd;
    int64_t n;
};
// pack: column <- state; unpack: state <- column.  Every value round-trips exactly (float state is widened to R).
template <bool kPack, typename T, typename U> __device__ __forceinline__ void snap_move(T& v, U* col) {
    if constexpr (kPack) *col = (U)v; else v = (T)*col;
}
// The one list of the image's columns, walked in both directions.  The per-env planes go through load_env / store_env, which know
// where each field sits in the handle's layout (Compact = KernelArgs::compact: 0 wide, 1 compact, 2 DR-compact); the volley and
// ring planes are addressed as the step, export and import kernels address them.
template <bool kPack, typename R, int Compact> __device__ void snapshot_env(const KernelArgs<R>& A, const SnapImage<R>& S, int64_t i) {
    KernelArgs<R> B = A;
    B.P.thrust_dyn = 1; B.P.dr = 1;   // the optional planes are always allocated and initialised: move them unconditionally
    B.compact = Compact;
    const int64_t n = S.n, stride = A.ring_stride;
    Env<R> e;
    if constexpr (kPack) load_env(B, i, e); else e.flags = 0;
    R* rc = S.real + i;
    auto mr = [&](auto& v) { snap_move<kPack>(v, rc); rc += n; };
    mr(e.ipx); mr(e.ipy); mr(e.ipz); mr(e.fuel); mr(e.ivx); mr(e.ivy); mr(e.ivz); mr(e.fuel_used);
    mr(e.mpx); mr(e.mpy); mr(e.mpz); mr(e.prev_d); mr(e.mvx); mr(e.mvy); mr(e.mvz); mr(e.last_d);
    mr(e.kpx); mr(e.kpy); mr(e.kpz); mr(e.min_d); mr(e.kvx); mr(e.kvy); mr(e.kvz); mr(e.ep_ret);
    mr(e.thx); mr(e.thy); mr(e.thz); mr(e.T0); mr(e.qw); mr(e.qx); mr(e.qy); mr(e.qz);
    mr(e.wx); mr(e.wy); mr(e.wz); mr(e.Ppp); mr(e.Ppv); mr(e.Pvp); mr(e.Pvv); mr(e.base_cd); mr(e.peak);
    int32_t* ic = S.ints + i;
    auto mi = [&](int& v) { snap_move<kPack>(v, ic); ic += n; };
    int crossed = e.flags & FLAG_CROSSED ? 1 : 0, kf_init = e.flags & FLAG_KF_INIT ? 1 : 0, kf_f64 = e.flags & FLAG_KF_F64 ? 1 : 0;
    int odelay = FLAG_ODELAY(e.flags), vcur = FLAG_VCUR(e.flags), vcount = FLAG_VCOUNT(e.flags);
    mi(e.steps); mi(e.worsen); mi(e.episode); mi(crossed); mi(kf_init); mi(kf_f64); mi(odelay); mi(vcur); mi(vcount);
    for (int m = 0; m < A.P.volley_k; ++m) {
        Vec4<R>* pa = A.st.vm + (int64_t)(2 * m) * stride + i;
        Vec4<R>* pb = A.st.vm + (int64_t)(2 * m + 1) * stride + i;
        Vec4<R> a{R(0), R(0), R(0), R(0)}, b = a;
        if constexpr (kPack) { a = *pa; b = *pb; }
        int act = b.w != R(0) ? 1 : 0;
        mr(a.x); mr(a.y); mr(a.z); mr(a.w); mr(b.x); mr(b.y); mr(b.z); mi(act);
        if constexpr (!kPack) { b.w = act ? R(1) : R(0); *pa = a; *pb = b; }
    }
    const int ol = A.P.onb_ring_len, gl = A.P.gnd_ring_len;
    R* oc = S.onb + i;
    for (int j = 0; j < ol; ++j) {   // age j = the sample written j ticks before the snapshot; A.o_row = the last tick's row
        const int row = A.o_row - j < 0 ? A.o_row - j + ol : A.o_row - j;
        float4* p = A.st.oring + (int64_t)row * stride + i;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if constexpr (kPack) v = *p;
        snap_move<kPack>(v.x, oc); snap_move<kPack>(v.y, oc + n); snap_move<kPack>(v.z, oc + 2 * n); snap_move<kPack>(v.w, oc + 3 * n);
        if constexpr (!kPack) *p = v;
        oc += 4 * n;
    }
    R* gc = S.gnd + i;
    for (int j = 0; j < gl; ++j) {
        const int row = A.g_row - j < 0 ? A.g_row - j + gl : A.g_row - j;
        Vec4<R>* p = A.st.gring + (int64_t)row * 2 * stride + i;
        for (int h = 0; h < 2; ++h) {
            Vec4<R> v{R(0), R(0), R(0), R(0)};
            if constexpr (kPack) v = p[h * stride];
            snap_move<kPack>(v.x, gc); snap_move<kPack>(v.y, gc + n); snap_move<kPack>(v.z, gc + 2 * n); snap_move<kPack>(v.w, gc + 3 * n);
            if constexpr (!kPack) p[h * stride] = v;
            gc += 4 * n;
        }
    }
    if constexpr (!kPack) {
        e.flags = (crossed ? FLAG_CROSSED : 0) | (kf_init ? FLAG_KF_INIT : 0) | (kf_f64 ? FLAG_KF_F64 : 0) | ((odelay & 0xf) << 8) |
                  ((vcur & 0x7) << 12) | ((vcount & 0xf) << 16);
        store_env(B, i, e);
    }
}
template <typename R, int Compact> __global__ void snapshot_pack_kernel(const KernelArgs<R> A, const SnapImage<R> S) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < S.n; i += (int64_t)gridDim.x * blockDim.x)
        snapshot_env<true, R, Compact>(A, S, i);
}
template <typename R, int Compact> __global__ void snapshot_unpack_kernel(const KernelArgs<R> A, const SnapImage<R> S) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < S.n; i += (int64_t)gridDim.x * blockDim.x)
        snapshot_env<false, R, Compact>(A, S, i);
}

__global__ void debug_draw_kernel(const __grid_constant__ RoundKeys rk, int64_t env, uint32_t episode, uint32_t step,
                                  uint32_t blk, uint32_t* raw, float* uni, float* nrm) {
    RngKey k;
    k.rk = &rk;
    k.c0 = (uint32_t)((uint64_t)env & 0xffffffffu);
    k.c3hi = (uint32_t)((uint64_t)env >> 32) << 16;
    uint4 r = draw_raw(k, episode, step, blk);
    raw[0] = r.x; raw[1] = r.y; raw[2] = r.z; raw[3] = r.w;
    uni[0] = u01(r.x); uni[1] = u01(r.y); uni[2] = u01(r.z); uni[3] = u01(r.w);
    box_muller(r.x, r.y, &nrm[0], &nrm[1]);
    box_muller(r.z, r.w, &nrm[2], &nrm[3]);
}

// ------------------------------------------------------------------------------------------------
// allocation
// ------------------------------------------------------------------------------------------------
template <typename R> static size_t carve(StatePlanes<R>& s, char* base, int64_t n_pad, int gl, int ol, int vk) {
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += (bytes + 255) & ~size_t(255); return p; };
    for (int k = 0; k < 7; ++k) s.r[k] = (Vec4<R>*)take(sizeof(Vec4<R>) * n_pad);
    for (int k = 0; k < 4; ++k) s.f[k] = (float4*)take(sizeof(float4) * n_pad);
    s.i0 = (int4*)take(sizeof(int4) * n_pad);
    s.vm = (Vec4<R>*)take(sizeof(Vec4<R>) * n_pad * 2 * (vk > 0 ? vk : 1));
    s.gring = (Vec4<R>*)take(sizeof(Vec4<R>) * n_pad * 2 * (gl > 0 ? gl : 1));
    s.oring = (float4*)take(sizeof(float4) * n_pad * (ol > 0 ? ol : 1));
    return off;
}

template <typename R> static void set_tick(KernelArgs<R>& A, uint64_t tick) {
    A.tick = (uint32_t)tick;
    A.g_row = A.P.gnd_ring_len > 0 ? (int32_t)(tick % (uint64_t)A.P.gnd_ring_len) : 0;
    A.o_row = A.P.onb_ring_len > 0 ? (int32_t)(tick % (uint64_t)A.P.onb_ring_len) : 0;
    // the rows an API-mode tick reads (prefetched in the kernel prologue); they are valid row addresses even while a ring still fills
    A.pf_o = nullptr; A.pf_g = nullptr;
    if (A.P.onb_ring_len > 0 && !A.P.dr) {
        int rrow = A.o_row - A.P.onboard_delay;
        if (rrow < 0) rrow += A.P.onb_ring_len;
        A.pf_o = A.st.oring + (int64_t)rrow * A.ring_stride;
    }
    if (A.P.gnd_ring_len > 0) {
        const int rrow = A.g_row + 1 == A.P.gnd_ring_len ? 0 : A.g_row + 1;
        A.pf_g = A.st.gring + (int64_t)rrow * 2 * A.ring_stride;
    }
}
template <typename R> static KernelArgs<R> base_args(hlynr_sim* s, const StatePlanes<R>& planes) {
    KernelArgs<R> A;
    memset(&A, 0, sizeof(A));
    A.P = make_kparams<R>(s->params);
    A.C = make_kcur<R>(s->cur);
    A.st = planes;
    A.n = s->n; A.first = 0; A.lim = s->n;
    A.io.done_records = s->done_records; A.io.done_counter = s->done_counter; A.io.done_cap = s->done_cap;
    A.io.done = s->io_done;
    A.ring_stride = s->n_pad;
    A.env_offset = s->env_offset;
    A.rk = make_round_keys(s->seed);
    set_tick(A, s->tick);
    A.io.stats = s->stats.get();
    A.k_steps = 1;
    A.prefetch_ahead = s->sm_count * s->prefetch_waves * HLYNR_BLOCK;
    A.obs_dim = s->obs_dim;
    A.compact = s->compact;
    A.cur_dev = s->cur_attached ? &((CurBlock<R>*)s->cur_block.get())->slot : nullptr;
    return A;
}
// Before a step (increment = the attached increment) or a reset (0): the slot the next launch reads, and the count advanced.
static int curriculum_tick(hlynr_sim* s, int64_t increment, cudaStream_t st) {
    if (!s->cur_attached) return 0;
    with_planes(s, [&](auto& planes) {
        using R = real_of<decltype(planes)>;
        curriculum_tick_kernel<R><<<1, 1, 0, st>>>((CurBlock<R>*)s->cur_block.get(), s->sched, (unsigned long long)increment);
    });
    CK(cudaGetLastError());
    s->launches += 1;
    return 0;
}
static inline int grid_for(int64_t n, int block) { return (int)((n + block - 1) / block); }

// Feature set of a resolved configuration; a specialised instantiation exists for FT_V2ON and FT_V2OFF.
static int feature_set(const HlynrParams& p) {
    if (p.obs_mode != HLYNR_OBS_WORLD || p.volley_size > 0) return FT_GENERIC_MODES;
    if (p.precision_mode || p.fuze_enabled) return FT_GENERIC;
    int f = p.dr_enabled ? FT_DR : 0;
    if (p.isa_enabled) f |= FT_ISA;
    if (p.mach_enabled) f |= FT_MACH;
    if (p.enh_wind_enabled) f |= FT_ENHW;
    if (p.thrust_dyn_enabled) f |= FT_THRUST;
    if (p.onboard_delay > 0) f |= FT_ONBD;
    if (p.ground_enabled) f |= FT_GROUND;
    if (p.ground_enabled && p.ground_delay > 0) f |= FT_GDELAY;
    if (p.evasion_enabled) f |= FT_EVADE;
    return (f == FT_V2ON || f == FT_V2OFF || f == FT_V2ON_DR) ? f : FT_GENERIC;
}
// Both builds dispatch to the feature-specialised instantiation of the three BASELINE configurations when it matches.
// One launch of an instantiation.  pdl: programmatic dependent launch -- the grid may be scheduled while the previous kernel
// of the stream is still draining; the kernel itself waits (griddepcontrol.wait, its first instruction that matters) until
// that kernel has completed and its writes are visible, so only launch latency and the tail of the previous grid overlap.
template <typename R, bool kRollout, int F, bool kCur> static void launch_inst(const KernelArgs<R>& A, int grid, cudaStream_t st, bool pdl) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(HLYNR_STEP_BLOCK); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    {   // measurement aid (tools/occupancy_sweep.sh): HLYNR_OCC_PAD_BYTES of unused dynamic shared memory per CTA lower the
        // resident CTAs per SM, which gives the sensitivity of the launch time to the number of resident warps
        static const int pad = getenv("HLYNR_OCC_PAD_BYTES") ? atoi(getenv("HLYNR_OCC_PAD_BYTES")) : 0;
        if (pad > 0) {
            cudaFuncSetAttribute(step_kernel<R, kRollout, F, kCur>, cudaFuncAttributeMaxDynamicSharedMemorySize, pad);
            cfg.dynamicSmemBytes = (size_t)pad;
        }
    }
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1u : 0u;
    cudaLaunchKernelEx(&cfg, step_kernel<R, kRollout, F, kCur>, A);
}
template <typename R, bool kRollout, bool kCur> static void launch_feature(const KernelArgs<R>& A, int f, int grid, cudaStream_t st, bool pdl) {
    if (f == FT_V2ON) launch_inst<R, kRollout, FT_V2ON, kCur>(A, grid, st, pdl);
    else if (f == FT_V2OFF) launch_inst<R, kRollout, FT_V2OFF, kCur>(A, grid, st, pdl);
    else if (f == FT_V2ON_DR) launch_inst<R, kRollout, FT_V2ON_DR, kCur>(A, grid, st, pdl);
    else if (f == FT_GENERIC_MODES) launch_inst<R, kRollout, FT_GENERIC_MODES, kCur>(A, grid, st, pdl);
    else launch_inst<R, kRollout, FT_GENERIC, kCur>(A, grid, st, pdl);
}
// Both builds dispatch to the feature-specialised instantiation of the three BASELINE configurations when it matches, and API-mode
// ticks to the instantiation that reads the curriculum slot while a schedule is attached (hlynr_rollout refuses one).
template <typename R, bool kRollout> static void launch_step(const hlynr_sim* s, const KernelArgs<R>& A, cudaStream_t st, bool specialise) {
    const int grid = grid_for(A.lim - A.first, HLYNR_STEP_BLOCK);
    const bool pdl = s->pdl != 0;
    int f = feature_set(s->params);
    if (!specialise && f >= 0) f = FT_GENERIC;
    if constexpr (!kRollout) {
        if (A.cur_dev) { launch_feature<R, false, true>(A, f, grid, st, pdl); return; }
    }
    launch_feature<R, kRollout, false>(A, f, grid, st, pdl);
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* hlynr_last_error(void) { return g_err; }
int hlynr_abi_version(void) { return HLYNR_ABI_VERSION; }
size_t hlynr_params_size(void) { return sizeof(HlynrParams); }
size_t hlynr_env_state_size(void) { return sizeof(HlynrEnvState); }
size_t hlynr_curriculum_schedule_size(void) { return sizeof(HlynrCurriculumSchedule); }

void hlynr_destroy(hlynr_t* s) {
    if (!s) return;
    DeviceGuard g(s->device);
    delete s;
}

int hlynr_create(const HlynrParams* p, int64_t n_envs, int device, uint64_t seed, int64_t env_id_offset, int precision,
                 hlynr_t** out) {
    if (!p || !out) return fail("hlynr_create: null argument");
    if (p->abi_version != HLYNR_ABI_VERSION) return fail("hlynr_create: params.abi_version %d != %d", p->abi_version, HLYNR_ABI_VERSION);
    if (n_envs <= 0) return fail("hlynr_create: n_envs must be positive");
    if (precision != HLYNR_FP32 && precision != HLYNR_FP64) return fail("hlynr_create: precision must be 32 or 64");
    if (p->obs_mode != HLYNR_OBS_WORLD && p->obs_mode != HLYNR_OBS_BODY && p->obs_mode != HLYNR_OBS_LOS)
        return fail("hlynr_create: unknown observation_mode %d", p->obs_mode);
    if (p->volley_size < 0 || p->volley_size > HLYNR_MAX_VOLLEY) return fail("hlynr_create: volley_size must be in [0, %d]", HLYNR_MAX_VOLLEY);
    if (p->onboard_delay < 0 || p->onboard_delay > HLYNR_MAX_ONBOARD_DELAY) return fail("hlynr_create: onboard_delay out of range");
    if (p->ground_delay < 0 || p->ground_delay > HLYNR_MAX_GROUND_DELAY) return fail("hlynr_create: ground_delay out of range");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail("hlynr_create: device %d not available (%d devices)", device, ndev);
    DeviceGuard g(device);
    if (!g.ok) return fail("hlynr_create: cannot select device %d", device);
    std::unique_ptr<hlynr_sim> s(new (std::nothrow) hlynr_sim());
    if (!s) return fail("hlynr_create: out of host memory");
    s->params = *p;
    s->cur = HlynrCurriculum{200.0, 60.0, 1.0, 1.0};
    s->n = n_envs; s->n_pad = (n_envs + 127) & ~int64_t(127);  // whole 128-env tiles
    s->device = device; s->precision = precision; s->seed = seed; s->env_offset = env_id_offset;
    KParams<float> kp = make_kparams<float>(*p);
    const int gl = kp.gnd_ring_len, ol = kp.onb_ring_len;
    const size_t state_bytes = with_planes(s.get(), [&](auto& planes) { return carve(planes, nullptr, s->n_pad, gl, ol, p->volley_size); });
    const cudaError_t e = alloc(s->state_mem, state_bytes);
    if (e != cudaSuccess) return fail("hlynr_create: cudaMalloc(%zu bytes) failed: %s", state_bytes, cudaGetErrorString(e));
    CK(alloc(s->stats, (HLYNR_STAT_SLOTS + 1) * HLYNR_STATS_WORDS));
    CK(cudaMemset(s->state_mem.get(), 0, state_bytes));
    CK(cudaMemset(s->stats.get(), 0, sizeof(double) * (HLYNR_STAT_SLOTS + 1) * HLYNR_STATS_WORDS));
    CK(cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, device));
    const int blk = 256;
    with_planes(s.get(), [&](auto& planes) {
        using R = real_of<decltype(planes)>;
        carve(planes, s->state_mem.get(), s->n_pad, gl, ol, p->volley_size);
        // compact plane layout (fp32 build only; hlynr_device.cuh load_env): fixed for the life of the handle, whichever kernel
        // instantiation runs
        s->compact = 0;
        if (std::is_same<R, float>::value && p->max_steps < 65536 && !getenv("HLYNR_NO_COMPACT"))
            s->compact = feature_set(*p) == FT_V2ON ? 1 : (feature_set(*p) == FT_V2ON_DR ? 2 : 0);
        init_kernel<R><<<grid_for(s->n_pad, blk), blk>>>(planes, s->n_pad, (float)p->peak_mult, s->compact);
    });
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    s->launches += 1;
    *out = s.release();
    return 0;
}

int hlynr_num_envs(const hlynr_t* s, int64_t* out) { if (!s || !out) return fail("null argument"); *out = s->n; return 0; }
int hlynr_set_curriculum(hlynr_t* s, const HlynrCurriculum* c) {
    if (!s || !c) return fail("null argument");
    if (s->cur_attached)
        return fail("hlynr_set_curriculum: a curriculum schedule is attached and the device computes the curriculum from its counter: "
                    "set the count with hlynr_set_timesteps, or hlynr_detach_curriculum first");
    s->cur = *c;
    return 0;
}
int hlynr_get_curriculum(const hlynr_t* s, HlynrCurriculum* c) { if (!s || !c) return fail("null argument"); *c = s->cur; return 0; }
int hlynr_seed(hlynr_t* s, uint64_t seed) { if (!s) return fail("null handle"); s->seed = seed; return 0; }
static int make_pool(hlynr_sim* s);
int hlynr_set_option(hlynr_t* s, const char* name, int64_t value) {
    if (!s || !name) return fail("null argument");
    if (strcmp(name, "specialise") == 0) { s->specialise = value != 0; return 0; }
    if (strcmp(name, "host_info") == 0) { s->host_info = value != 0; return 0; }
    if (strcmp(name, "prefetch_waves") == 0) {
        if (value < 0 || value > 64) return fail("prefetch_waves must be in [0, 64]");
        s->prefetch_waves = (int)value;
        return 0;
    }
    if (strcmp(name, "obs_dim") == 0) {
        if (value != HLYNR_OBS_DIM && value != 17) return fail("obs_dim must be 26 (the reference's vector) or 17 (its leading radar channels obs[0:17])");
        s->obs_dim = (int)value;
        return 0;
    }
    if (strcmp(name, "host_chunks") == 0) {
        if (value < 0 || value > 64) return fail("host_chunks must be in [0, 64]");
        s->host_chunks = (int)value;
        return 0;
    }
    if (strcmp(name, "pdl") == 0) { s->pdl = value != 0; return 0; }
    if (strcmp(name, "host_chunk_growth") == 0) {
        if (value < 0 || value > 64) return fail("host_chunk_growth must be in [0, 64] (eighths: 16 = chunks double, 0 = uniform chunks)");
        s->host_chunk_growth = (int)value;
        return 0;
    }
    if (strcmp(name, "host_threads") == 0) {
        if (value < 0 || value > 64) return fail("host_threads must be in [0, 64]");
        s->host_threads = (int)value;
        return s->hio.ready ? make_pool(s) : 0;
    }
    return fail("hlynr_set_option: unknown option '%s'", name);
}
static int64_t gcd64(int64_t a, int64_t b) { while (b) { int64_t t = a % b; a = b; b = t; } return a; }
int hlynr_ring_period(const hlynr_t* s, int* out) {
    if (!s || !out) return fail("null argument");
    const KParams<float> k = make_kparams<float>(s->params);
    const int64_t a = k.onb_ring_len > 0 ? k.onb_ring_len : 1, b = k.gnd_ring_len > 0 ? k.gnd_ring_len : 1;
    *out = (int)(a / gcd64(a, b) * b);
    return 0;
}
int hlynr_note_replayed_ticks(hlynr_t* s, int64_t ticks, int64_t launches) {
    if (!s) return fail("hlynr_note_replayed_ticks: null handle");
    // negative values undo the host-side bookkeeping of calls that were only RECORDED into a graph (not executed)
    s->tick = (uint64_t)((int64_t)s->tick + ticks); s->env_steps += (double)s->n * (double)ticks; s->launches += launches;
    return 0;
}
int hlynr_tick_count(const hlynr_t* s, int64_t* out) { if (!s || !out) return fail("null argument"); *out = (int64_t)s->tick; return 0; }
int hlynr_launch_count(const hlynr_t* s, int64_t* out) { if (!s || !out) return fail("null argument"); *out = s->launches; return 0; }

int hlynr_reset(hlynr_t* s, const uint8_t* mask_dev, float* obs_dev, void* stream) {
    if (!s) return fail("hlynr_reset: null handle");
    DeviceGuard g(s->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (curriculum_tick(s, 0, st)) return 1;   // the reference's reset uses the last pushed count and does not advance it
    with_planes(s, [&](auto& planes) {
        using R = real_of<decltype(planes)>;
        KernelArgs<R> A = base_args(s, planes);
        A.io.reset_mask = mask_dev; A.io.obs = obs_dev;
        // the instantiation that reads the curriculum slot while a schedule is attached
        const auto kernel = A.cur_dev ? reset_kernel<R, true> : reset_kernel<R, false>;
        kernel<<<grid_for(s->n, HLYNR_BLOCK), HLYNR_BLOCK, 0, st>>>(A);
    });
    CK(cudaGetLastError());
    s->launches += 1;
    return 0;
}

// One tick of the envs [first, lim) (multiples of 128 except lim == n); the caller has advanced s->tick.  The
// pointers are the [N]-sized arrays (indexed by the local env id), not chunk-relative ones.
static int step_range(hlynr_sim* s, int64_t first, int64_t lim, const float* actions_dev, float* obs_dev, float* reward_dev,
                      uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev, const HlynrInfoSoA* info,
                      int auto_reset, cudaStream_t st) {
    with_planes(s, [&](auto& planes) {
        using R = real_of<decltype(planes)>;
        KernelArgs<R> A = base_args(s, planes);
        A.first = first; A.lim = lim;
        A.io.actions = actions_dev; A.io.obs = obs_dev; A.io.reward = reward_dev; A.io.terminated = terminated_dev;
        A.io.truncated = truncated_dev; A.io.terminal_obs = terminal_obs_dev; A.auto_reset = auto_reset;
        if (info) { A.io.info = *info; A.has_info = 1; }
        launch_step<R, false>(s, A, st, s->specialise != 0);
    });
    CK(cudaGetLastError());
    s->launches += 1;
    s->env_steps += (double)(lim - first);
    return 0;
}

int hlynr_step(hlynr_t* s, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* terminated_dev,
               uint8_t* truncated_dev, float* terminal_obs_dev, const HlynrInfoSoA* info, int auto_reset, void* stream) {
    if (!s) return fail("hlynr_step: null handle");
    if (!actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev) return fail("hlynr_step: null output/input pointer");
    DeviceGuard g(s->device);
    if (curriculum_tick(s, s->cur_increment, (cudaStream_t)stream)) return 1;
    s->tick += 1;
    return step_range(s, 0, s->n, actions_dev, obs_dev, reward_dev, terminated_dev, truncated_dev, terminal_obs_dev, info,
                      auto_reset, (cudaStream_t)stream);
}

// The schedules hlynr_attach_curriculum (and hlynr_snapshot_load, which re-attaches one) accept.
static int check_schedule(const HlynrCurriculumSchedule* c, int64_t increment, const char* who) {
    const double f[] = {c->initial_radius, c->final_radius, c->curriculum_steps, c->beam_initial, c->beam_final, c->beam_start,
                        c->beam_end, c->onboard_initial, c->onboard_final, c->onboard_start, c->onboard_end, c->ground_initial,
                        c->ground_final, c->ground_start, c->ground_end};
    for (double v : f)
        if (!std::isfinite(v)) return fail("%s: every field of the schedule must be finite", who);
    if (c->enabled && !(c->curriculum_steps > 0.0)) return fail("%s: curriculum_steps must be positive while the curriculum is enabled", who);
    if (increment < 0) return fail("%s: increment must not be negative", who);
    return 0;
}
int hlynr_attach_curriculum(hlynr_t* s, const HlynrCurriculumSchedule* c, uint64_t num_timesteps, int64_t increment) {
    if (!s || !c) return fail("hlynr_attach_curriculum: null argument");
    if (check_schedule(c, increment, "hlynr_attach_curriculum")) return 1;
    DeviceGuard g(s->device);
    if (!s->cur_block) CK(alloc(s->cur_block, 1));
    CK(cudaDeviceSynchronize());   // no launch of an earlier attachment still reads or writes the block
    const unsigned long long v = num_timesteps;
    CK(cudaMemcpy(s->cur_block.get(), &v, sizeof(v), cudaMemcpyHostToDevice));
    s->sched = *c; s->cur_increment = increment; s->cur_attached = true;
    return 0;
}
int hlynr_detach_curriculum(hlynr_t* s) {
    if (!s) return fail("hlynr_detach_curriculum: null handle");
    s->cur_attached = false;
    return 0;
}
int hlynr_set_timesteps(hlynr_t* s, uint64_t num_timesteps, void* stream) {
    if (!s) return fail("hlynr_set_timesteps: null handle");
    if (!s->cur_attached) return fail("hlynr_set_timesteps: no curriculum schedule is attached (hlynr_attach_curriculum)");
    DeviceGuard g(s->device);
    set_timesteps_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((unsigned long long*)s->cur_block.get(), (unsigned long long)num_timesteps);
    CK(cudaGetLastError());
    s->launches += 1;
    return 0;
}
int hlynr_get_timesteps(hlynr_t* s, uint64_t* out, void* stream) {
    if (!s || !out) return fail("hlynr_get_timesteps: null argument");
    if (!s->cur_attached) return fail("hlynr_get_timesteps: no curriculum schedule is attached (hlynr_attach_curriculum)");
    DeviceGuard g(s->device);
    const cudaStream_t st = (cudaStream_t)stream;
    CK(cudaStreamSynchronize(st));
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, s->cur_block.get(), sizeof(v), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *out = (uint64_t)v;
    return 0;
}
int hlynr_debug_curriculum_at(hlynr_t* s, uint64_t count, double out[4]) {
    if (!s || !out) return fail("hlynr_debug_curriculum_at: null argument");
    if (!s->cur_attached) return fail("hlynr_debug_curriculum_at: no curriculum schedule is attached (hlynr_attach_curriculum)");
    DeviceGuard g(s->device);
    DevPtr<double> buf;
    CK(alloc(buf, 4));
    with_planes(s, [&](auto& planes) { curriculum_probe_kernel<real_of<decltype(planes)>><<<1, 1>>>(s->sched, (unsigned long long)count, buf.get()); });
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, buf.get(), 4 * sizeof(double), cudaMemcpyDeviceToHost));
    s->launches += 1;
    return 0;
}

int hlynr_set_done_list(hlynr_t* s, HlynrDoneRecord* records_dev, int32_t* counter_dev, int32_t capacity) {
    if (!s) return fail("hlynr_set_done_list: null handle");
    if (records_dev && (!counter_dev || capacity <= 0)) return fail("hlynr_set_done_list: counter_dev and a positive capacity are required");
    s->done_records = records_dev; s->done_counter = records_dev ? counter_dev : nullptr; s->done_cap = records_dev ? capacity : 0;
    return 0;
}

int hlynr_rollout(hlynr_t* s, int k_steps, const float* actions_dev, float* obs_dev, float* reward_sum_dev,
                  int32_t* done_count_dev, void* stream) {
    if (!s) return fail("hlynr_rollout: null handle");
    if (k_steps <= 0) return fail("hlynr_rollout: k_steps must be positive");
    if (s->cur_attached)
        return fail("hlynr_rollout: not available while a curriculum schedule is attached (the fused ticks would each need their own "
                    "curriculum slot): step with hlynr_step, or hlynr_detach_curriculum first");
    DeviceGuard g(s->device);
    cudaStream_t st = (cudaStream_t)stream;
    with_planes(s, [&](auto& planes) {
        using R = real_of<decltype(planes)>;
        KernelArgs<R> A = base_args(s, planes);
        set_tick(A, s->tick + 1); A.k_steps = k_steps; A.auto_reset = 1;
        A.io.actions = actions_dev; A.io.obs = obs_dev; A.io.reward_sum = reward_sum_dev; A.io.done_count = done_count_dev;
        launch_step<R, true>(s, A, st, s->specialise != 0);
    });
    CK(cudaGetLastError());
    s->tick += (uint64_t)k_steps;
    s->launches += 1;
    s->env_steps += (double)s->n * k_steps;
    return 0;
}

int hlynr_stats_device_ptr(hlynr_t* s, double** out) {
    if (!s || !out) return fail("null argument");
    *out = s->stats.get() + HLYNR_STAT_SLOTS * HLYNR_STATS_WORDS;
    return 0;
}

// Folds the per-block slots into the reduced row (device side; call before an NCCL all-reduce on it).
int hlynr_stats_reduce(hlynr_t* s, void* stream) {
    if (!s) return fail("null handle");
    DeviceGuard g(s->device);
    stats_reduce_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(s->stats.get(), s->env_steps);
    CK(cudaGetLastError());
    s->launches += 1;
    return 0;
}

int hlynr_get_stats(hlynr_t* s, HlynrStats* host_out, int zero_after, void* stream) {
    if (!s || !host_out) return fail("null argument");
    DeviceGuard g(s->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (hlynr_stats_reduce(s, stream)) return 1;
    CK(cudaMemcpyAsync(host_out, s->stats.get() + HLYNR_STAT_SLOTS * HLYNR_STATS_WORDS, sizeof(double) * HLYNR_STATS_WORDS,
                       cudaMemcpyDeviceToHost, st));
    if (zero_after) {
        CK(cudaMemsetAsync(s->stats.get(), 0, sizeof(double) * (HLYNR_STAT_SLOTS + 1) * HLYNR_STATS_WORDS, st));
        s->env_steps = 0.0;
    }
    CK(cudaStreamSynchronize(st));
    return 0;
}

static int ensure_xchg(hlynr_sim* s, int64_t count) {
    if (s->xchg_cap >= count) return 0;
    s->xchg_cap = 0;
    CK(alloc(s->xchg, count));
    s->xchg_cap = count;
    return 0;
}

int hlynr_export_state(hlynr_t* s, int64_t first, int64_t count, HlynrEnvState* host_out) {
    if (!s || !host_out) return fail("null argument");
    if (first < 0 || count < 0 || first + count > s->n) return fail("hlynr_export_state: range out of bounds");
    if (count == 0) return 0;
    DeviceGuard g(s->device);
    CK(cudaDeviceSynchronize());
    if (ensure_xchg(s, count)) return 1;
    with_planes(s, [&](auto& planes) {
        export_kernel<real_of<decltype(planes)>><<<grid_for(count, 128), 128>>>(base_args(s, planes), first, count, s->xchg.get());
    });
    CK(cudaGetLastError());
    CK(cudaMemcpy(host_out, s->xchg.get(), sizeof(HlynrEnvState) * count, cudaMemcpyDeviceToHost));
    s->launches += 1;
    return 0;
}

int hlynr_import_state(hlynr_t* s, int64_t first, int64_t count, const HlynrEnvState* host_in) {
    if (!s || !host_in) return fail("null argument");
    if (first < 0 || count < 0 || first + count > s->n) return fail("hlynr_import_state: range out of bounds");
    if (count == 0) return 0;
    DeviceGuard g(s->device);
    CK(cudaDeviceSynchronize());
    if (ensure_xchg(s, count)) return 1;
    CK(cudaMemcpy(s->xchg.get(), host_in, sizeof(HlynrEnvState) * count, cudaMemcpyHostToDevice));
    with_planes(s, [&](auto& planes) {
        import_kernel<real_of<decltype(planes)>><<<grid_for(count, 128), 128>>>(base_args(s, planes), first, count, s->xchg.get());
    });
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    s->launches += 1;
    return 0;
}

int hlynr_debug_draws(hlynr_t* s, int64_t env_global_id, uint32_t episode, uint32_t step, uint32_t block, uint32_t raw_out[4],
                      float uniform_out[4], float normal_out[4]) {
    if (!s) return fail("null handle");
    DeviceGuard g(s->device);
    DevPtr<char> buf;
    CK(alloc(buf, 48));
    debug_draw_kernel<<<1, 1>>>(make_round_keys(s->seed), env_global_id, episode, step, block,
                                (uint32_t*)buf.get(), (float*)(buf.get() + 16), (float*)(buf.get() + 32));
    char host[48];
    CK(cudaMemcpy(host, buf.get(), 48, cudaMemcpyDeviceToHost));
    memcpy(raw_out, host, 16); memcpy(uniform_out, host + 16, 16); memcpy(normal_out, host + 32, 16);
    s->launches += 1;
    return 0;
}

}  // extern "C"

// ---- snapshots ---------------------------------------------------------------------------------------------------------------
static_assert(HLYNR_STAT_ROWS == HLYNR_STAT_SLOTS + 1, "the image's statistics section is the whole statistics block");
static_assert(sizeof(HlynrSnapshotInfo) == 952, "HlynrSnapshotInfo is mirrored by abi.HlynrSnapshotInfo");
// every field of HlynrParams, compared one by one so that a refused load names the field
#define HLYNR_PARAMS_FIELDS(X) \
    X(abi_version) X(max_steps) X(dt) X(max_range) X(max_velocity) X(target) X(m_spawn_spherical) X(i_vel_toward_missile) \
    X(m_pos_lo) X(m_pos_hi) X(m_speed_lo) X(m_speed_hi) X(m_radius_lo) X(m_radius_hi) X(m_az_lo) X(m_az_hi) X(m_el_lo) \
    X(m_el_hi) X(i_pos_lo) X(i_pos_hi) X(i_vel_lo) X(i_vel_hi) X(i_speed_lo) X(i_speed_hi) X(base_wind) X(wind_variability) \
    X(isa_enabled) X(mach_enabled) X(enh_wind_enabled) X(thrust_dyn_enabled) X(dr_enabled) X(validate_enabled) \
    X(evasion_enabled) X(onboard_delay) X(sub_mach) X(sup_mach) X(peak_mult) X(sup_mult) X(blh) X(turb_intensity) \
    X(gust_scale) X(thrust_tau) X(dr_variation) X(radar_range) X(radar_quality) X(ground_enabled) X(ground_delay) \
    X(ground_pos) X(g_max_range) X(g_min_el) X(g_max_el) X(g_sigma_r) X(g_sigma_v) X(g_base_quality) X(max_datalink_range) \
    X(datalink_packet_loss) X(obs_mode) X(precision_mode) X(fuze_enabled) X(volley_size) X(kill_radius)

// The descriptor of the handle's current state, with the byte offsets of the image's sections (256-byte aligned).
static void snapshot_describe(const hlynr_sim* s, HlynrSnapshotInfo* info) {
    memset(info, 0, sizeof(*info));
    const KParams<float> k = make_kparams<float>(s->params);
    info->format_version = HLYNR_SNAPSHOT_VERSION; info->abi_version = HLYNR_ABI_VERSION;
    info->precision = s->precision; info->obs_dim = s->obs_dim;
    info->n_envs = s->n; info->env_id_offset = s->env_offset; info->seed = s->seed;
    info->volley_k = s->params.volley_size; info->onboard_ring_len = k.onb_ring_len; info->ground_ring_len = k.gnd_ring_len;
    info->curriculum_attached = s->cur_attached ? 1 : 0;
    info->tick = s->tick; info->env_steps = s->env_steps;
    info->params = s->params; info->curriculum = s->cur;
    if (s->cur_attached) { info->schedule = s->sched; info->curriculum_increment = s->cur_increment; }
    const size_t rs = s->precision == HLYNR_FP32 ? sizeof(float) : sizeof(double), n = (size_t)s->n, K = (size_t)s->params.volley_size;
    const size_t bytes[HLYNR_SNAP_SECTIONS] = {(HLYNR_SNAP_REAL_COLS + 7 * K) * n * rs, (HLYNR_SNAP_INT_COLS + K) * n * sizeof(int32_t),
                                               (size_t)k.onb_ring_len * 4 * n * rs, (size_t)k.gnd_ring_len * 8 * n * rs,
                                               sizeof(double) * HLYNR_STAT_ROWS * HLYNR_STATS_WORDS, sizeof(uint64_t)};
    size_t off = 0;
    for (int j = 0; j < HLYNR_SNAP_SECTIONS; ++j) { info->section_offset[j] = off; off += (bytes[j] + 255) & ~size_t(255); }
    info->device_bytes = off;
}
template <typename R> static SnapImage<R> snap_image(const HlynrSnapshotInfo& info, char* base) {
    SnapImage<R> S;
    S.real = (R*)(base + info.section_offset[HLYNR_SNAP_REAL]); S.ints = (int32_t*)(base + info.section_offset[HLYNR_SNAP_INT]);
    S.onb = (R*)(base + info.section_offset[HLYNR_SNAP_ONBOARD]); S.gnd = (R*)(base + info.section_offset[HLYNR_SNAP_GROUND]);
    S.n = info.n_envs;
    return S;
}
// Launches the pack or unpack kernel of the handle's precision and layout; the ring rows of the last executed tick come from the
// handle's tick (set_tick), so load restores the tick first.
static int snapshot_kernels(hlynr_sim* s, const HlynrSnapshotInfo& info, char* base, bool pack, cudaStream_t st) {
    const int grid = (int)std::min<int64_t>(grid_for(s->n, 256), (int64_t)s->sm_count * 8);
    with_layout(s, [&](auto& planes, auto compact) {
        using R = real_of<decltype(planes)>;
        constexpr int C = decltype(compact)::value;
        const KernelArgs<R> A = base_args(s, planes);
        const SnapImage<R> S = snap_image<R>(info, base);
        if (pack) snapshot_pack_kernel<R, C><<<grid, 256, 0, st>>>(A, S);
        else snapshot_unpack_kernel<R, C><<<grid, 256, 0, st>>>(A, S);
    });
    CK(cudaGetLastError());
    s->launches += 1;
    return 0;
}

extern "C" {

size_t hlynr_snapshot_info_size(void) { return sizeof(HlynrSnapshotInfo); }

int hlynr_snapshot_layout(const hlynr_t* s, HlynrSnapshotInfo* info, size_t* device_bytes) {
    if (!s || !info || !device_bytes) return fail("hlynr_snapshot_layout: null argument");
    snapshot_describe(s, info);
    *device_bytes = (size_t)info->device_bytes;
    return 0;
}

int hlynr_snapshot_save(hlynr_t* s, void* dev_out, HlynrSnapshotInfo* info, void* stream) {
    if (!s || !dev_out || !info) return fail("hlynr_snapshot_save: null argument");
    DeviceGuard g(s->device);
    const cudaStream_t st = (cudaStream_t)stream;
    if (refuse_capture(st, "hlynr_snapshot_save")) return 1;
    snapshot_describe(s, info);
    char* base = (char*)dev_out;
    if (snapshot_kernels(s, *info, base, true, st)) return 1;
    CK(cudaMemcpyAsync(base + info->section_offset[HLYNR_SNAP_STATS], s->stats.get(), sizeof(double) * HLYNR_STAT_ROWS * HLYNR_STATS_WORDS,
                       cudaMemcpyDeviceToDevice, st));
    if (s->cur_attached)   // CurBlock::num_timesteps is the block's first member
        CK(cudaMemcpyAsync(base + info->section_offset[HLYNR_SNAP_CURRICULUM], s->cur_block.get(), sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    else
        CK(cudaMemsetAsync(base + info->section_offset[HLYNR_SNAP_CURRICULUM], 0, sizeof(uint64_t), st));
    return 0;
}

int hlynr_snapshot_load(hlynr_t* s, const HlynrSnapshotInfo* info, const void* dev_in, void* stream) {
    if (!s || !info || !dev_in) return fail("hlynr_snapshot_load: null argument");
    HlynrSnapshotInfo mine;
    snapshot_describe(s, &mine);
    const HlynrSnapshotInfo& in = *info;
#define HLYNR_SNAP_REFUSE(cond, what, ...) if (cond) return fail("hlynr_snapshot_load: the snapshot's " what " differs from the handle's: " __VA_ARGS__)
    HLYNR_SNAP_REFUSE(in.format_version != mine.format_version, "format version", "%d, expected %d", in.format_version, mine.format_version);
    HLYNR_SNAP_REFUSE(in.abi_version != mine.abi_version, "ABI version", "%d, expected %d", in.abi_version, mine.abi_version);
    HLYNR_SNAP_REFUSE(in.precision != mine.precision, "precision", "fp%d into an fp%d handle", in.precision, mine.precision);
    HLYNR_SNAP_REFUSE(in.n_envs != mine.n_envs, "n_envs", "%lld, the handle has %lld", (long long)in.n_envs, (long long)mine.n_envs);
    HLYNR_SNAP_REFUSE(in.env_id_offset != mine.env_id_offset, "env_id_offset", "%lld, the handle has %lld", (long long)in.env_id_offset,
                      (long long)mine.env_id_offset);
    HLYNR_SNAP_REFUSE(in.obs_dim != mine.obs_dim, "obs_dim", "%d, the handle has %d", in.obs_dim, mine.obs_dim);
    HLYNR_SNAP_REFUSE(in.volley_k != mine.volley_k, "volley size K", "%d, the handle has %d", in.volley_k, mine.volley_k);
    HLYNR_SNAP_REFUSE(in.onboard_ring_len != mine.onboard_ring_len, "onboard ring length", "%d, the handle has %d", in.onboard_ring_len,
                      mine.onboard_ring_len);
    HLYNR_SNAP_REFUSE(in.ground_ring_len != mine.ground_ring_len, "ground ring length", "%d, the handle has %d", in.ground_ring_len,
                      mine.ground_ring_len);
#define X(f) HLYNR_SNAP_REFUSE(memcmp(&in.params.f, &mine.params.f, sizeof(in.params.f)) != 0, "configuration", "field HlynrParams." #f);
    HLYNR_PARAMS_FIELDS(X)
#undef X
    for (int j = 0; j < HLYNR_SNAP_SECTIONS; ++j)
        HLYNR_SNAP_REFUSE(in.section_offset[j] != mine.section_offset[j], "image layout", "offset of section %d", j);
    HLYNR_SNAP_REFUSE(in.device_bytes != mine.device_bytes, "image size", "%llu bytes, expected %llu", (unsigned long long)in.device_bytes,
                      (unsigned long long)mine.device_bytes);
#undef HLYNR_SNAP_REFUSE
    if (in.curriculum_attached && check_schedule(&in.schedule, in.curriculum_increment, "hlynr_snapshot_load")) return 1;
    DeviceGuard g(s->device);
    const cudaStream_t st = (cudaStream_t)stream;
    if (refuse_capture(st, "hlynr_snapshot_load")) return 1;
    if (in.curriculum_attached && !s->cur_block) CK(alloc(s->cur_block, 1));
    // the host state first: the unpack kernel's ring rows follow the restored tick
    s->tick = in.tick; s->env_steps = in.env_steps; s->seed = in.seed; s->cur = in.curriculum;
    s->cur_attached = in.curriculum_attached != 0;
    if (s->cur_attached) { s->sched = in.schedule; s->cur_increment = in.curriculum_increment; }
    char* base = (char*)dev_in;
    if (snapshot_kernels(s, in, base, false, st)) return 1;
    CK(cudaMemcpyAsync(s->stats.get(), base + in.section_offset[HLYNR_SNAP_STATS], sizeof(double) * HLYNR_STAT_ROWS * HLYNR_STATS_WORDS,
                       cudaMemcpyDeviceToDevice, st));
    if (s->cur_attached)
        CK(cudaMemcpyAsync(s->cur_block.get(), base + in.section_offset[HLYNR_SNAP_CURRICULUM], sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    return 0;
}

}  // extern "C"

extern "C" {

// ---- host-buffer entry points ----------------------------------------------------------------
static int make_pool(hlynr_sim* s) {
    HostIO& h = s->hio;
    h.pool.reset();
    int helpers = s->host_threads > 0 ? s->host_threads - 1 : 3;
    const int hw = (int)std::thread::hardware_concurrency();
    if (hw > 0 && helpers > hw - 1) helpers = hw - 1;
    if ((size_t)s->n * 26 * sizeof(float) < (size_t(4) << 20)) helpers = 0;  // small shards never reach the pool's threshold
    h.pool.reset(new (std::nothrow) CopyPool(helpers));
    if (!h.pool) return fail("out of host memory");
    return 0;
}
// Page-locked host memory (cudaMallocHost / cudaHostAlloc / cudaHostRegister, e.g. a torch pin_memory() tensor) can be the
// source or target of the DMA -- and, under unified addressing, of the kernel's own stores -- without a staging copy.
static bool is_pinned_host(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}
// The address the DEVICE uses for a page-locked host buffer the kernel stores into (identical to the host address wherever
// cudaDevAttrCanUseHostPointerForRegisteredMem holds, which is every platform this library targets, but asked for anyway);
// nullptr if the buffer is not device-accessible.
static void* device_view(void* host_ptr) {
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, host_ptr, 0) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return d;
}
static int ensure_hostio(hlynr_sim* s) {
    HostIO& h = s->hio;
    if (h.ready) return 0;
    const size_t n = (size_t)s->n;
    CK(alloc(h.h_actions, n * 6));
    CK(alloc(h.h_obs, n * 26));
    CK(alloc(h.h_reward, n));
    CK(alloc(h.h_term, n)); CK(alloc(h.h_trunc, n)); CK(alloc(h.h_mask, n));
    CK(alloc(h.h_records_ab[0], n));
    CK(alloc(h.h_records_ab[1], n));
    h.h_records = h.h_records_ab[0].get();
    CK(alloc(h.h_done, n));
    CK(alloc(h.h_count, 1));
    CK(alloc(h.d_actions, n * 6));
    CK(alloc(h.d_obs, n * 26));
    CK(alloc(h.d_mask, n));
    CK(alloc(h.d_records, n));
    CK(alloc(h.d_counter, 1));
    CK(cudaMemset(h.d_counter.get(), 0, sizeof(int32_t)));
    for (int k = 0; k < HLYNR_HOST_STREAMS; ++k) {
        CK(stream_create(h.streams[k]));
        CK(event_create(h.ev_done[k]));
    }
    CK(event_create(h.ev_start));
    if (make_pool(s)) return 1;
    h.ready = true;
    return 0;
}
// Orders the handle's own streams after the work already queued on the legacy default stream (where torch's
// current stream normally is), so that a tensor-API call followed by a *_host call on the same handle is safe.
// Work queued on other caller streams must be synchronised by the caller.
static int host_streams_begin(hlynr_sim* s) {
    HostIO& h = s->hio;
    CK(cudaEventRecord(h.ev_start.get(), cudaStreamLegacy));
    for (int k = 0; k < HLYNR_HOST_STREAMS; ++k) CK(cudaStreamWaitEvent(h.streams[k].get(), h.ev_start.get(), 0));
    return 0;
}
static int ensure_host_info(hlynr_sim* s) {
    HostIO& h = s->hio;
    if (h.info_ready) return 0;
    const size_t n = (size_t)s->n;
#define X(name, type, per_env) CK(alloc(h.info_##name, n * (per_env))); h.d_info.name = h.info_##name.get();
    HLYNR_INFO_FIELDS(X)
#undef X
    h.info_ready = true;
    return 0;
}

int hlynr_reset_host(hlynr_t* s, const uint8_t* mask_host, float* obs_host) {
    if (!s || !obs_host) return fail("hlynr_reset_host: null argument");
    DeviceGuard g(s->device);
    if (ensure_hostio(s)) return 1;
    HostIO& h = s->hio;
    cudaStream_t st = h.streams[0].get();
    const size_t n = (size_t)s->n, ob = (size_t)s->obs_dim * sizeof(float);
    if (host_streams_begin(s)) return 1;
    if (mask_host) {
        memcpy(h.h_mask.get(), mask_host, n);
        CK(cudaMemcpyAsync(h.d_mask.get(), h.h_mask.get(), n, cudaMemcpyHostToDevice, st));
        // rows of envs that are not reset keep the caller's content
        if (obs_host != h.h_obs.get()) h.pool->copy(h.h_obs.get(), obs_host, n * ob);
        CK(cudaMemcpyAsync(h.d_obs.get(), h.h_obs.get(), n * ob, cudaMemcpyHostToDevice, st));
    }
    if (hlynr_reset(s, mask_host ? h.d_mask.get() : nullptr, h.d_obs.get(), st)) return 1;
    CK(cudaMemcpyAsync(h.h_obs.get(), h.d_obs.get(), n * ob, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (obs_host != h.h_obs.get()) h.pool->copy(obs_host, h.h_obs.get(), n * ob);
    return 0;
}

// step through host buffers.  The shard is cut into chunks of whole 128-env tiles; chunk c runs
//   H2D(actions) -> step kernel -> D2H(obs, reward, terminated, truncated)
// on stream c % 3, so the upload of one chunk, the kernel of another and the download of a third overlap (PCIe is
// full duplex; the download, 110 B per env, is what bounds the call).  Finished episodes come back as a compact
// record list (count + first records in one small copy), never as [N]-sized arrays.
int hlynr_step_host(hlynr_t* s, const float* actions_host, float* obs_host, float* reward_host, uint8_t* terminated_host,
                    uint8_t* truncated_host, float* terminal_obs_host, int auto_reset) {
    if (!s || !actions_host || !obs_host || !reward_host || !terminated_host || !truncated_host) return fail("hlynr_step_host: null argument");
    if (s->cur_attached)
        return fail("hlynr_step_host: not available while a curriculum schedule is attached: the host path takes its curriculum from "
                    "hlynr_set_curriculum, which the host-side training callback drives; hlynr_detach_curriculum first");
    DeviceGuard g(s->device);
    if (ensure_hostio(s)) return 1;
    if (s->host_info && ensure_host_info(s)) return 1;
    HostIO& h = s->hio;
    const int64_t n = s->n, od = s->obs_dim;
    // chunk boundaries (whole 128-env tiles).  Uniform: host_chunks equal chunks.  Geometric (option "host_chunk_growth" > 0, the
    // default for large shards): a small first chunk so the download starts early, then chunks that grow by the factor growth/8
    // up to a cap -- the download of the chunks already in flight (75-111 B per env) always outlasts the upload + kernel of the
    // next, larger one (24 B per env), so the copy engine never idles and there are fewer per-copy gaps.
    int64_t bounds[65];
    int64_t chunks = 0;
    bounds[0] = 0;
    if (s->host_chunks > 0 || s->host_chunk_growth <= 0 || n < (int64_t(1) << 17)) {
        chunks = s->host_chunks > 0 ? s->host_chunks : (n >= (int64_t(1) << 19) ? 16 : (n >= (int64_t(1) << 17) ? 8 : (n >= (int64_t(1) << 15) ? 4 : 1)));
        const int64_t per = ((n + chunks - 1) / chunks + 127) & ~int64_t(127);
        chunks = (n + per - 1) / per;
        for (int64_t c = 1; c <= chunks; ++c) bounds[c] = c * per < n ? c * per : n;
    } else {
        int64_t sz = 16384;
        const int64_t cap = (int64_t(1) << 17) + (int64_t(1) << 16);   // 196608 envs: ~20 MB of observations per copy
        while (bounds[chunks] < n && chunks < 63) {
            const int64_t next = bounds[chunks] + sz;
            bounds[chunks + 1] = (next >= n || n - next < sz / 2) ? n : next;
            ++chunks;
            sz = (sz * s->host_chunk_growth / 8 + 127) & ~int64_t(127);
            if (sz > cap) sz = cap;
        }
        bounds[chunks] = n;
    }
    // the handle's own done list for this call (a caller-attached list is restored afterwards)
    HlynrDoneRecord* keep_r = s->done_records; int32_t* keep_c = s->done_counter; const int32_t keep_cap = s->done_cap;
    s->done_records = h.d_records.get(); s->done_counter = h.d_counter.get(); s->done_cap = (int32_t)(n < INT32_MAX ? n : INT32_MAX);
    s->io_done = s->host_done ? s->host_done : h.h_done.get();
    // caller buffers that are page-locked are used in place; pageable ones go through the handle's pinned staging buffers
    const bool stage = !(actions_host == h.h_actions.get() || is_pinned_host(actions_host));
    const float* act_src = stage ? h.h_actions.get() : actions_host;
    const bool out_direct = (obs_host == h.h_obs.get() || is_pinned_host(obs_host)) && (reward_host == h.h_reward.get() || is_pinned_host(reward_host)) &&
                            (terminated_host == h.h_term.get() || is_pinned_host(terminated_host)) &&
                            (truncated_host == h.h_trunc.get() || is_pinned_host(truncated_host));
    float* obs_dst = out_direct ? obs_host : h.h_obs.get();
    float* reward_dst = out_direct ? reward_host : h.h_reward.get();
    uint8_t* term_dst = out_direct ? terminated_host : h.h_term.get();
    uint8_t* trunc_dst = out_direct ? truncated_host : h.h_trunc.get();
    struct Restore { hlynr_sim* s; HlynrDoneRecord* r; int32_t* c; int32_t cap;
                     ~Restore() { s->done_records = r; s->done_counter = c; s->done_cap = cap; s->io_done = nullptr; } }
        restore{s, keep_r, keep_c, keep_cap};
    // reward / terminated / truncated / dones are stored by the kernel: it needs their device-side addresses
    float* reward_k = (float*)device_view(reward_dst);
    uint8_t *term_k = (uint8_t*)device_view(term_dst), *trunc_k = (uint8_t*)device_view(trunc_dst);
    s->io_done = (uint8_t*)device_view(s->io_done);
    if (!reward_k || !term_k || !trunc_k || !s->io_done) return fail("hlynr_step_host: a page-locked output buffer is not device-accessible");
    static const bool trace = getenv("HLYNR_HOST_TRACE") != nullptr;   // debugging aid: host-side timeline on stderr
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    double t_staged[64] = {0}, t_issued = 0, t_synced = 0;
    if (host_streams_begin(s)) return 1;
    CK(cudaMemsetAsync(h.d_counter.get(), 0, sizeof(int32_t), h.streams[0].get()));
    CK(cudaEventRecord(h.ev_start.get(), h.streams[0].get()));
    for (int k = 1; k < HLYNR_HOST_STREAMS; ++k) CK(cudaStreamWaitEvent(h.streams[k].get(), h.ev_start.get(), 0));
    s->tick += 1;
    const HlynrInfoSoA* info = s->host_info ? &h.d_info : nullptr;
    struct StageGuard { CopyPool* p; ~StageGuard() { if (p) p->finish(); } } stage_guard{stage ? h.pool.get() : nullptr};
    if (stage) h.pool->start(h.h_actions.get(), actions_host, (size_t)n * 24);
    for (int64_t c = 0; c < chunks; ++c) {
        const int64_t first = bounds[c], lim = bounds[c + 1], cnt = lim - first;
        cudaStream_t st = h.streams[c % HLYNR_HOST_STREAMS].get();
        if (stage) h.pool->wait_prefix((size_t)lim * 24);
        if (trace && c < 64) t_staged[c] = since();
        CK(cudaMemcpyAsync(h.d_actions.get() + first * 6, act_src + first * 6, (size_t)cnt * 24, cudaMemcpyHostToDevice, st));
        // reward / terminated / truncated (6 B per env) are written by the kernel STRAIGHT into the pinned host buffers
        // (cudaMallocHost memory is device-accessible under unified addressing; coalesced posted PCIe writes, +26 us per
        // 2^20 envs): three small copy-engine transfers per chunk, each with its own fixed latency, disappear and only the
        // observation (104 B per env) rides the copy engine
        if (step_range(s, first, lim, h.d_actions.get(), h.d_obs.get(), reward_k, term_k, trunc_k, nullptr, info, auto_reset, st)) return 1;
        CK(cudaMemcpyAsync(obs_dst + first * od, h.d_obs.get() + first * od, (size_t)(cnt * od) * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    // done list: after every chunk's kernel; count + the first records in one go on stream 0
    for (int k = 1; k < HLYNR_HOST_STREAMS; ++k) {
        CK(cudaEventRecord(h.ev_done[k].get(), h.streams[k].get()));
        CK(cudaStreamWaitEvent(h.streams[0].get(), h.ev_done[k].get(), 0));
    }
    const size_t prefix = (size_t)(n < HLYNR_DONE_PREFIX ? n : HLYNR_DONE_PREFIX);
    h.h_records = h.h_records_ab[(h.calls++) & 1u].get();
    CK(cudaMemcpyAsync(h.h_count.get(), h.d_counter.get(), sizeof(int32_t), cudaMemcpyDeviceToHost, h.streams[0].get()));
    CK(cudaMemcpyAsync(h.h_records, h.d_records.get(), prefix * sizeof(HlynrDoneRecord), cudaMemcpyDeviceToHost, h.streams[0].get()));
    if (trace) t_issued = since();
    for (int k = HLYNR_HOST_STREAMS - 1; k >= 0; --k) CK(cudaStreamSynchronize(h.streams[k].get()));
    if (trace) {
        t_synced = since();
        fprintf(stderr, "hlynr_step_host: staged");
        for (int64_t c = 0; c < chunks && c < 64; ++c) fprintf(stderr, " %.2f", t_staged[c]);
        fprintf(stderr, " | issued %.2f | synced %.2f ms\n", t_issued, t_synced);
    }
    if (obs_host != obs_dst) h.pool->copy(obs_host, obs_dst, (size_t)(n * od) * sizeof(float));
    if (reward_host != reward_dst) h.pool->copy(reward_host, reward_dst, (size_t)n * 4);
    if (terminated_host != term_dst) h.pool->copy(terminated_host, term_dst, (size_t)n);
    if (truncated_host != trunc_dst) h.pool->copy(truncated_host, trunc_dst, (size_t)n);
    int32_t count = *h.h_count;
    if (count > s->done_cap) count = s->done_cap;
    if ((size_t)count > prefix) {
        CK(cudaMemcpyAsync(h.h_records + prefix, h.d_records.get() + prefix, ((size_t)count - prefix) * sizeof(HlynrDoneRecord),
                           cudaMemcpyDeviceToHost, h.streams[0].get()));
        CK(cudaStreamSynchronize(h.streams[0].get()));
    }
    h.last_count = count;
    if (terminal_obs_host)  // only rows of finished envs are written (info['terminal_observation'])
        for (int32_t k = 0; k < count; ++k)
            memcpy(terminal_obs_host + (size_t)h.h_records[k].env * od, h.h_records[k].terminal_obs, (size_t)od * sizeof(float));
    return 0;
}

int hlynr_done_records_host(hlynr_t* s, const HlynrDoneRecord** records, int32_t* count) {
    if (!s || !records || !count) return fail("hlynr_done_records_host: null argument");
    if (!s->hio.ready) return fail("hlynr_done_records_host: no hlynr_step_host call yet");
    *records = s->hio.h_records; *count = s->hio.last_count;
    return 0;
}

int hlynr_info_host(hlynr_t* s, HlynrInfoSoA* o) {
    if (!s || !o) return fail("hlynr_info_host: null argument");
    if (!s->hio.ready || !s->hio.info_ready) return fail("hlynr_info_host: no hlynr_step_host call with option host_info = 1 yet");
    DeviceGuard g(s->device);
    const HlynrInfoSoA& d = s->hio.d_info;
    const size_t n = (size_t)s->n;
    cudaStream_t st = s->hio.streams[0].get();
#define X(name, type, per_env) if (o->name) CK(cudaMemcpyAsync(o->name, d.name, n * (per_env) * sizeof(type), cudaMemcpyDeviceToHost, st));
    HLYNR_INFO_FIELDS(X)
#undef X
    CK(cudaStreamSynchronize(st));
    return 0;
}

// terminated | truncated of the last hlynr_step_host call, written by the kernel itself into pinned host memory.
int hlynr_pinned_done(hlynr_t* s, uint8_t** done) {
    if (!s || !done) return fail("hlynr_pinned_done: null argument");
    DeviceGuard g(s->device);
    if (ensure_hostio(s)) return 1;
    *done = s->hio.h_done.get();
    return 0;
}

int hlynr_host_done_buffer(hlynr_t* s, uint8_t* done_pinned) {
    if (!s) return fail("hlynr_host_done_buffer: null handle");
    DeviceGuard g(s->device);
    if (done_pinned && !is_pinned_host(done_pinned))
        return fail("hlynr_host_done_buffer: the buffer must be page-locked host memory (the kernel writes it directly)");
    s->host_done = done_pinned;
    return 0;
}

// Pinned host buffers owned by the handle (numpy callers wrap them to avoid the staging memcpy).
int hlynr_pinned_buffers(hlynr_t* s, float** actions, float** obs, float** reward, uint8_t** terminated, uint8_t** truncated) {
    if (!s) return fail("null handle");
    DeviceGuard g(s->device);
    if (ensure_hostio(s)) return 1;
    if (actions) *actions = s->hio.h_actions.get();
    if (obs) *obs = s->hio.h_obs.get();
    if (reward) *reward = s->hio.h_reward.get();
    if (terminated) *terminated = s->hio.h_term.get();
    if (truncated) *truncated = s->hio.h_trunc.get();
    return 0;
}

}  // extern "C"
