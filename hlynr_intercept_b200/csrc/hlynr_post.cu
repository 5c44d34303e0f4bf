// hlynr_post.cu -- on-device VecFrameStack + VecNormalize (C ABI: include/hlynr_post.h, SURVEY 8f rank 1).
//
// Semantics restated from stable-baselines3 2.x (oracle/sb3_post.py cites the source files):
//   stacked[e] = concat(frame[t-k+1], ..., frame[t]); a finished env's stack is zeroed before its reset observation
//   is inserted; info['terminal_observation'] = concat(previous_stack[F:], terminal_obs[0:F]);
//   obs_rms.update(stacked batch) (batch mean/var merged into the running float64 moments), then
//   out = clip((stacked - mean) / sqrt(var + eps), -clip, clip) as float32; terminal observations likewise.
//
// HBM traffic per env-step (n_stack = 4): 104 B column-sum read of the new frame + 416 B ring read + 416 B output
// write (+ 9 B age/done flags, 16 B returns) -- the explicit roll/copy of SB3 (another 832 B) never happens, and the
// step kernel writes its observation straight into the ring slot.
//
// The frame width F is 26 (the full observation) or 17 (the leading radar channels obs[0:17], HlynrSim(obs_dim=17)); every
// kernel that touches the ring is a template on F, so the 26-wide code is what it was before F became a parameter.
#include <cmath>
#include <cstring>
#include <new>
#include <type_traits>

#include <cuda_runtime.h>

#include "../../include/hlynr_post.h"
#include "hlynr_host.cuh"

namespace {

constexpr int OD = HLYNR_OBS_DIM;  // 26: the widest frame, and the row capacity of the per-lag arrays of PostStats
constexpr int KMAX = HLYNR_POST_MAX_STACK;
constexpr int DMAX = OD * KMAX;

// device statistics block (doubles); a 17-wide frame uses the first 17 entries of every [KMAX][OD] row
struct PostStats {
    double S[KMAX][OD], Q[KMAX][OD];        // per-lag column sums / sums of squares of the current stacked batch (lag 0 = newest)
    double col[OD], colq[OD];               // scratch: sums over the new frame
    double corr[KMAX][OD], corrq[KMAX][OD]; // scratch: frames of the envs that finished in this step (subtracted)
    double ret_sum, ret_sq;                 // scratch: sums over the discounted returns
    double mean[DMAX], var[DMAX], count;    // obs_rms (feature f = j*F + c, j = 0 oldest)
    double ret_mean, ret_var, ret_count;    // ret_rms
    double chk_S[KMAX][OD], chk_Q[KMAX][OD];  // check_sums scratch
    double inv_std[DMAX];                   // 1 / sqrt(var + eps): the normalise kernels compute in float64 like SB3 (obs f32 - mean f64)
};

__device__ __forceinline__ int ring_slot(int newest, int lag, int k) { int s = newest - lag; return s < 0 ? s + k : s; }

// ---- sums over the new frame: thread-constant channel, 16 envs per 16*F-thread block iteration, coalesced ----
// Every reduction of this file is two-stage and atomic-free: blocks write partial sums to partials[block][word], one
// block per word then folds them in a fixed order, so the statistics (and with them the normalised observations) are
// bit-reproducible from run to run.
template <int F>   // word offsets of a partial row for frame width F: [col F | colq F | ret | retq | corr (k-1)*F | corrq (k-1)*F]
struct PW { static constexpr int COL = 0, COLQ = F, RET = 2 * F, RETQ = 2 * F + 1, CORR = 2 * F + 2; };
constexpr int PART_WORDS = PW<OD>::CORR + 2 * (KMAX - 1) * OD;   // sized for the widest frame

template <int F>
__global__ void __launch_bounds__(16 * F) colsum_kernel(const float* __restrict__ frame, int64_t n, double* __restrict__ partials) {
    __shared__ double sh[16 * F];
    const int t = threadIdx.x, c = t % F, r = t / F;
    double s = 0.0, q = 0.0;
    for (int64_t e = (int64_t)blockIdx.x * 16 + r; e < n; e += (int64_t)gridDim.x * 16) {
        const double v = (double)frame[e * F + c];
        s += v; q += v * v;
    }
    sh[t] = s;
    __syncthreads();
    double* mine = partials + (size_t)blockIdx.x * PART_WORDS;
    if (r == 0) { double a = 0.0; for (int i = 0; i < 16; ++i) a += sh[i * F + c]; mine[PW<F>::COL + c] = a; }
    __syncthreads();
    sh[t] = q;
    __syncthreads();
    if (r == 0) { double a = 0.0; for (int i = 0; i < 16; ++i) a += sh[i * F + c]; mine[PW<F>::COLQ + c] = a; }
}

// second stage: block w folds word w of the partial rows (fixed order) into its PostStats field
template <int F>
__global__ void __launch_bounds__(256) fold_kernel(const double* __restrict__ partials, int nb_col, int nb_ret, int nb_corr, int per,
                                                   PostStats* st) {
    __shared__ double sh[256];
    const int w = blockIdx.x;
    const int nblocks = w < 2 * F ? nb_col : (w < PW<F>::CORR ? nb_ret : nb_corr);
    double a = 0.0;
    for (int b = threadIdx.x; b < nblocks; b += 256) a += partials[(size_t)b * PART_WORDS + w];
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    if (w < F) st->col[w] = sh[0];
    else if (w < 2 * F) st->colq[w - F] = sh[0];
    else if (w < PW<F>::CORR) (&st->ret_sum)[w - 2 * F] = sh[0];     // ret_sum, ret_sq
    else if (w - PW<F>::CORR < per) { const int f = w - PW<F>::CORR; st->corr[1 + f / F][f % F] = sh[0]; }
    else { const int f = w - PW<F>::CORR - per; st->corrq[1 + f / F][f % F] = sh[0]; }
}

// ---- VecNormalize._update_reward: returns = returns * gamma + reward; ret_rms sums; returns[done] = 0 ----
// Also the per-env part of VecFrameStack: age_new = done ? 0 : min(age_old + 1, k - 1) (how many older frames of the
// ring belong to the env's current episode).
template <int F>
__global__ void __launch_bounds__(256) returns_kernel(double* __restrict__ ret, const float* __restrict__ rew,
                                                      const uint8_t* __restrict__ term, const uint8_t* __restrict__ trunc, int64_t n,
                                                      double gamma, double* __restrict__ partials, int training,
                                                      const uint8_t* __restrict__ age_in, uint8_t* __restrict__ age_out, int k) {
    double s = 0.0, q = 0.0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        double r = ret[e];
        // SB3's `returns * gamma + rewards` rounds twice: _rn keeps nvcc from contracting it into one DFMA
        if (training) { r = __dadd_rn(__dmul_rn(r, gamma), (double)rew[e]); s += r; q += r * r; }
        const bool done = (term[e] | trunc[e]) != 0;
        ret[e] = done ? 0.0 : r;  // returns[dones] = 0 happens whether or not the statistics move
        const int a = (int)age_in[e] + 1;
        age_out[e] = (uint8_t)(done ? 0 : (a < k - 1 ? a : k - 1));
    }
    if (!training) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
    __shared__ double shs[8], shq[8];
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { shs[w] = s; shq[w] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += shs[i]; b += shq[i]; }
        partials[(size_t)blockIdx.x * PART_WORDS + PW<F>::RET] = a; partials[(size_t)blockIdx.x * PART_WORDS + PW<F>::RETQ] = b;
    }
}

// ---- frames of finished envs leave the stack: accumulate what has to be subtracted from the shifted sums ----
// thread = (record lane r, old lag d in [0, k-2], channel c); old lag d becomes lag d+1 for the envs that go on.
template <int F>
__global__ void __launch_bounds__(512) done_corr_kernel(const HlynrDoneRecord* __restrict__ recs, const int32_t* __restrict__ counter,
                                                        int32_t cap, const float* __restrict__ frames, int64_t plane,
                                                        const uint8_t* __restrict__ age_old, int k, int newest_old,
                                                        double* __restrict__ partials) {
    const int per = (k - 1) * F;                  // threads per record
    const int lanes = blockDim.x / per;           // records per block iteration
    const int t = threadIdx.x;
    if (t >= lanes * per) return;
    const int r = t / per, f = t % per, d = f / F, c = f % F;
    int32_t count = *counter;
    if (count > cap) count = cap;
    double s = 0.0, q = 0.0;
    const float* src = frames + (int64_t)ring_slot(newest_old, d, k) * plane;
    for (int32_t i = blockIdx.x * lanes + r; i < count; i += gridDim.x * lanes) {
        const int32_t e = recs[i].env;
        if (d <= (int)age_old[e]) { const double v = (double)src[(int64_t)e * F + c]; s += v; q += v * v; }
    }
    // fold the record lanes of this block, then one partial row per block: [corr (k-1)*F | corrq (k-1)*F]
    __shared__ double sh[512];
    sh[t] = s;
    __syncthreads();
    double* mine = partials + (size_t)blockIdx.x * PART_WORDS + PW<F>::CORR;
    if (r == 0) { double a = 0.0; for (int i = 0; i < lanes; ++i) a += sh[i * per + f]; mine[f] = a; }
    __syncthreads();
    sh[t] = q;
    __syncthreads();
    if (r == 0) { double a = 0.0; for (int i = 0; i < lanes; ++i) a += sh[i * per + f]; mine[per + f] = a; }
}

// ---- shift the per-lag sums, merge the batch moments into obs_rms / ret_rms (RunningMeanStd.update_from_moments) ----
// The merge rounds every product and sum on its own in numpy's order (_rn: no contraction into DFMA), so batch moments that
// are exact (e.g. dyadic frames) give obs_rms bit for bit as numpy does.
__device__ __forceinline__ void rms_merge(double& mean, double& var, double count, double bm, double bv, double n) {
    const double delta = bm - mean, tot = count + n;
    const double m2 = __dadd_rn(__dadd_rn(__dmul_rn(var, count), __dmul_rn(bv, n)), __dmul_rn(__dmul_rn(__dmul_rn(delta, delta), count), n) / tot);
    mean = __dadd_rn(mean, __dmul_rn(delta, n) / tot);
    var = m2 / tot;
}

template <int F>
__global__ void merge_kernel(PostStats* st, int k, double n, int shift, int training, int reset_all, int with_returns, double eps) {
    const int f = threadIdx.x, D = k * F;
    if (shift && f < F) {  // the per-lag sums follow the ring on every reset / step
        const int c = f;
        for (int d = k - 1; d >= 1; --d) {
            st->S[d][c] = reset_all ? 0.0 : st->S[d - 1][c] - st->corr[d][c];
            st->Q[d][c] = reset_all ? 0.0 : st->Q[d - 1][c] - st->corrq[d][c];
            st->corr[d][c] = 0.0; st->corrq[d][c] = 0.0;
        }
        st->S[0][c] = st->col[c]; st->Q[0][c] = st->colq[c];
        st->col[c] = 0.0; st->colq[c] = 0.0;
    }
    const double count = st->count;
    __syncthreads();
    if (f < D) {
        if (training) {
            const int j = f / F, c = f % F, d = k - 1 - j;
            const double bm = st->S[d][c] / n;
            double bv = __dsub_rn(st->Q[d][c] / n, __dmul_rn(bm, bm));
            if (bv < 0.0) bv = 0.0;
            rms_merge(st->mean[f], st->var[f], count, bm, bv, n);
        }
        st->inv_std[f] = 1.0 / sqrt(st->var[f] + eps);
    }
    __syncthreads();
    if (f == 0 && training) {
        st->count = count + n;
        if (with_returns) {
            const double bm = st->ret_sum / n;
            double bv = __dsub_rn(st->ret_sq / n, __dmul_rn(bm, bm));
            if (bv < 0.0) bv = 0.0;
            rms_merge(st->ret_mean, st->ret_var, st->ret_count, bm, bv, n);
            st->ret_count = st->ret_count + n;
        }
        st->ret_sum = 0.0; st->ret_sq = 0.0;
    }
}

// ---- stacked (+ normalised) observation of 26-wide frames: thread-constant feature PAIR (26 is even, so a float2 never
// straddles two ring slots and every load/store is 8-byte aligned), 8 envs in flight per thread, coalesced [N, 26k] output ----
#define NORM_UNROLL 8
__global__ void __launch_bounds__(512) normalize_kernel(const float* __restrict__ frames, int64_t plane, const uint8_t* __restrict__ age,
                                                        const PostStats* __restrict__ st, float* __restrict__ out, int64_t n, int k,
                                                        int newest, float clip, int raw) {
    const int D = k * OD, P = D / 2, lanes = blockDim.x / P, t = threadIdx.x;
    if (t >= lanes * P) return;
    const int r = t / P, p = t % P, f = 2 * p, j = f / OD, c = f % OD, lag = k - 1 - j;
    // SB3 evaluates (obs_f32 - mean_f64) / sqrt(var + eps) in float64 and rounds the result to float32.  Here the mean is
    // split into a float pair (hi + lo), so the cancellation obs - mean keeps ~48 bits; the product and the clip are float:
    // the result is within 3 float ulps of SB3's, without touching the FP64 pipe (3, not 2: obs - m_hi rounds in the operands'
    // binade, and the result can land one binade lower, where that rounding error is 2 ulps).
    const float m0h = (float)st->mean[f], m0l = (float)(st->mean[f] - (double)m0h), i0 = (float)st->inv_std[f];
    const float m1h = (float)st->mean[f + 1], m1l = (float)(st->mean[f + 1] - (double)m1h), i1 = (float)st->inv_std[f + 1];
    const float* src = frames + (int64_t)ring_slot(newest, lag, k) * plane + c;
    const int64_t stride = (int64_t)gridDim.x * lanes;
    for (int64_t e0 = (int64_t)blockIdx.x * lanes + r; e0 < n; e0 += stride * NORM_UNROLL) {
        float2 v[NORM_UNROLL];
        int ag[NORM_UNROLL];
        bool ok[NORM_UNROLL];
#pragma unroll
        for (int u = 0; u < NORM_UNROLL; ++u) {  // frame and age loads are independent: all in flight together; a slot
            const int64_t e = e0 + u * stride;   // older than the env's episode holds stale but readable data
            ok[u] = e < n;
            v[u] = make_float2(0.f, 0.f);
            ag[u] = 0;
            if (ok[u]) { v[u] = __ldcs(reinterpret_cast<const float2*>(src + e * OD)); ag[u] = (int)__ldg(age + e); }
        }
#pragma unroll
        for (int u = 0; u < NORM_UNROLL; ++u) {
            if (!ok[u]) continue;
            float2 w = lag <= ag[u] ? v[u] : make_float2(0.f, 0.f);
            if (!raw) {
                w.x = fminf(fmaxf(((w.x - m0h) - m0l) * i0, -clip), clip);
                w.y = fminf(fmaxf(((w.y - m1h) - m1l) * i1, -clip), clip);
            }
            __stcs(reinterpret_cast<float2*>(out + (e0 + u * stride) * D + f), w);
        }
    }
}

// ---- the same for 17-wide frames: thread-constant single feature.  A feature pair would straddle two ring slots at every
// odd frame boundary, and an output row of odd width 17k starts only 4-byte aligned, so every access is one float; the
// block's `lanes` consecutive envs still read lanes * 17 contiguous floats per ring slot and write lanes * 17k contiguous
// floats, and NORM_UNROLL envs are in flight per thread.  Per element the same float operations as normalize_kernel. ----
template <int F>
__global__ void __launch_bounds__(512) normalize1_kernel(const float* __restrict__ frames, int64_t plane, const uint8_t* __restrict__ age,
                                                         const PostStats* __restrict__ st, float* __restrict__ out, int64_t n, int k,
                                                         int newest, float clip, int raw) {
    const int D = k * F, lanes = blockDim.x / D, t = threadIdx.x;
    if (t >= lanes * D) return;
    const int r = t / D, f = t % D, j = f / F, c = f % F, lag = k - 1 - j;
    const float mh = (float)st->mean[f], ml = (float)(st->mean[f] - (double)mh), inv = (float)st->inv_std[f];
    const float* src = frames + (int64_t)ring_slot(newest, lag, k) * plane + c;
    const int64_t stride = (int64_t)gridDim.x * lanes;
    for (int64_t e0 = (int64_t)blockIdx.x * lanes + r; e0 < n; e0 += stride * NORM_UNROLL) {
        float v[NORM_UNROLL];
        int ag[NORM_UNROLL];
        bool ok[NORM_UNROLL];
#pragma unroll
        for (int u = 0; u < NORM_UNROLL; ++u) {
            const int64_t e = e0 + u * stride;
            ok[u] = e < n;
            v[u] = 0.f;
            ag[u] = 0;
            if (ok[u]) { v[u] = __ldcs(src + e * F); ag[u] = (int)__ldg(age + e); }
        }
#pragma unroll
        for (int u = 0; u < NORM_UNROLL; ++u) {
            if (!ok[u]) continue;
            float w = lag <= ag[u] ? v[u] : 0.f;
            if (!raw) w = fminf(fmaxf(((w - mh) - ml) * inv, -clip), clip);
            __stcs(out + (e0 + u * stride) * D + f, w);
        }
    }
}

// ---- info['terminal_observation'] of finished envs: concat(previous_stack[F:], terminal_obs[0:F]), normalised ----
template <int F>
__global__ void __launch_bounds__(512) terminal_kernel(const HlynrDoneRecord* __restrict__ recs, const int32_t* __restrict__ counter, int32_t cap,
                                                       const float* __restrict__ frames, int64_t plane, const uint8_t* __restrict__ age_old,
                                                       const PostStats* __restrict__ st, float* __restrict__ out, int k, int newest_old,
                                                       float clip) {
    const int D = k * F, lanes = blockDim.x / D, t = threadIdx.x;
    if (t >= lanes * D) return;
    const int r = t / D, f = t % D, j = f / F, c = f % F;
    const double mean = st->mean[f], inv = st->inv_std[f];
    int32_t count = *counter;
    if (count > cap) count = cap;
    for (int32_t i = blockIdx.x * lanes + r; i < count; i += gridDim.x * lanes) {
        float v;
        if (j == k - 1) v = recs[i].terminal_obs[c];
        else {
            const int32_t e = recs[i].env;
            const int lag_old = k - 2 - j;
            v = lag_old <= (int)age_old[e] ? frames[(int64_t)ring_slot(newest_old, lag_old, k) * plane + (int64_t)e * F + c] : 0.f;
        }
        out[(int64_t)i * D + f] = (float)fmin(fmax(((double)v - mean) * inv, -(double)clip), (double)clip);
    }
}

// ---- VecNormalize.normalize_obs on caller rows ----
__global__ void __launch_bounds__(512) normalize_rows_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t rows, int D,
                                                             const PostStats* __restrict__ st, float clip) {
    const int lanes = blockDim.x / D, t = threadIdx.x;
    if (t >= lanes * D) return;
    const int r = t / D, f = t % D;
    const double mean = st->mean[f], inv = st->inv_std[f];
    for (int64_t e = (int64_t)blockIdx.x * lanes + r; e < rows; e += (int64_t)gridDim.x * lanes)
        out[e * D + f] = (float)fmin(fmax(((double)in[e * D + f] - mean) * inv, -(double)clip), (double)clip);
}

// ---- test hook: per-lag sums recomputed from the ring ----
template <int F>
__global__ void __launch_bounds__(512) recompute_sums_kernel(const float* __restrict__ frames, int64_t plane, const uint8_t* __restrict__ age,
                                                             int64_t n, int k, int newest, PostStats* st) {
    const int D = k * F, lanes = blockDim.x / D, t = threadIdx.x;
    if (t >= lanes * D) return;
    const int r = t / D, f = t % D, d = f / F, c = f % F;  // here f enumerates (lag d, channel c)
    const float* src = frames + (int64_t)ring_slot(newest, d, k) * plane + c;
    double s = 0.0, q = 0.0;
    for (int64_t e = (int64_t)blockIdx.x * lanes + r; e < n; e += (int64_t)gridDim.x * lanes)
        if (d <= (int)age[e]) { const double v = (double)src[e * F]; s += v; q += v * v; }
    atomicAdd(&st->chk_S[d][c], s); atomicAdd(&st->chk_Q[d][c], q);
}

}  // namespace

struct hlynr_post {
    int64_t n = 0, plane = 0;   // plane = floats per ring slot (n * fw rounded up to 128-byte multiples)
    int device = 0, fw = OD, k = 1, D = OD;   // frame width (26 or 17), n_stack, fw * n_stack
    double clip = 10.0, eps = 1e-8, gamma = 0.99;
    DevPtr<float> frames;
    DevPtr<uint8_t> age[2];
    int age_cur = 0;
    DevPtr<double> returns;
    DevPtr<PostStats> st;
    DevPtr<double> partials;    // [max_blocks][PART_WORDS] first-stage sums
    uint32_t t = 0;             // frames written so far; target slot = t % k, newest = (t - 1) % k
    bool sums_valid = false;    // the per-lag sums S/Q describe the current ring (maintained by every reset/step that can)
    int sm_count = 148;
    int64_t launches = 0;
};

// Calls f(std::integral_constant<int, F>{}) for the handle's frame width F, 26 or 17: the one place the width picks the
// instantiations of the ring kernels.
template <class Fn> static auto with_width(const hlynr_post* p, Fn&& f) {
    if (p->fw == OD) return f(std::integral_constant<int, OD>{});
    return f(std::integral_constant<int, 17>{});
}

static int blocks_for(const hlynr_post* p, int64_t items, int per_block) {
    int64_t b = (items + per_block - 1) / per_block;
    const int64_t cap = (int64_t)p->sm_count * 8;
    if (b > cap) b = cap;
    return b < 1 ? 1 : (int)b;
}

template <int F>
static int launch_normalize_t(hlynr_post* p, float* out, int raw, cudaStream_t st) {
    const int newest = (int)((p->t - 1) % (uint32_t)p->k);
    if constexpr (F % 2 == 0) {
        const int P = p->D / 2;
        const int lanes = 512 / P > 0 ? 512 / P : 1;
        normalize_kernel<<<blocks_for(p, (p->n + NORM_UNROLL - 1) / NORM_UNROLL, lanes), lanes * P, 0, st>>>(
            p->frames.get(), p->plane, p->age[p->age_cur].get(), p->st.get(), out, p->n, p->k, newest, (float)p->clip, raw);
    } else {
        const int lanes = 512 / p->D;
        normalize1_kernel<F><<<blocks_for(p, (p->n + NORM_UNROLL - 1) / NORM_UNROLL, lanes), lanes * p->D, 0, st>>>(
            p->frames.get(), p->plane, p->age[p->age_cur].get(), p->st.get(), out, p->n, p->k, newest, (float)p->clip, raw);
    }
    CK(cudaGetLastError());
    p->launches += 1;
    return 0;
}

static int launch_normalize(hlynr_post* p, float* out, int raw, cudaStream_t st) {
    return with_width(p, [&](auto F) { return launch_normalize_t<F>(p, out, raw, st); });
}

template <int F>
static int reset_t(hlynr_post* p, float* out_dev, int training, cudaStream_t st) {
    const float* frame = p->frames.get() + (int64_t)(p->t % (uint32_t)p->k) * p->plane;
    p->t += 1;
    CK(cudaMemsetAsync(p->returns.get(), 0, sizeof(double) * p->n, st));  // VecNormalize.reset: returns = zeros
    const int nb_col = blocks_for(p, p->n, 16);
    colsum_kernel<F><<<nb_col, 16 * F, 0, st>>>(frame, p->n, p->partials.get());
    fold_kernel<F><<<2 * F, 256, 0, st>>>(p->partials.get(), nb_col, 0, 0, 0, p->st.get());
    merge_kernel<F><<<1, 256, 0, st>>>(p->st.get(), p->k, (double)p->n, 1, training, 1, 0, p->eps);
    CK(cudaGetLastError());
    p->launches += 3;
    p->sums_valid = true;
    CK(cudaMemsetAsync(p->age[p->age_cur].get(), 0, p->n, st));  // VecFrameStack.reset: only the newest frame is valid
    return launch_normalize_t<F>(p, out_dev, 0, st);
}

template <int F>
static int step_t(hlynr_post* p, const float* reward_dev, const uint8_t* terminated_dev, const uint8_t* truncated_dev,
                  const HlynrDoneRecord* records_dev, const int32_t* counter_dev, int32_t capacity, float* out_dev,
                  float* terminal_out_dev, int training, bool can_maintain, cudaStream_t st) {
    const int newest_old = (int)((p->t - 1) % (uint32_t)p->k);
    const float* frame = p->frames.get() + (int64_t)(p->t % (uint32_t)p->k) * p->plane;
    const uint8_t* age_old = p->age[p->age_cur].get();
    p->t += 1;
    const int nb_ret = blocks_for(p, p->n, 256);
    returns_kernel<F><<<nb_ret, 256, 0, st>>>(p->returns.get(), reward_dev, terminated_dev, truncated_dev, p->n, p->gamma, p->partials.get(), training,
                                              age_old, p->age[p->age_cur ^ 1].get(), p->k);
    p->launches += 1;
    if (can_maintain && p->sums_valid) {  // the sums follow the ring on every step; obs_rms / ret_rms only move when training
        const int nb_col = blocks_for(p, p->n, 16);
        colsum_kernel<F><<<nb_col, 16 * F, 0, st>>>(frame, p->n, p->partials.get());
        p->launches += 1;
        const int per = (p->k - 1) * F;
        if (p->k > 1) {
            const int lanes = 512 / per;
            done_corr_kernel<F><<<64, lanes * per, 0, st>>>(records_dev, counter_dev, capacity, p->frames.get(), p->plane, age_old, p->k, newest_old,
                                                            p->partials.get());
            p->launches += 1;
        }
        fold_kernel<F><<<2 * F + 2 + 2 * per, 256, 0, st>>>(p->partials.get(), nb_col, training ? nb_ret : 0, 64, per, p->st.get());
        p->launches += 1;
        merge_kernel<F><<<1, 256, 0, st>>>(p->st.get(), p->k, (double)p->n, 1, training, 0, training, p->eps);
        p->launches += 1;
    } else {
        p->sums_valid = false;
    }
    if (terminal_out_dev) {
        const int lanes = 512 / p->D > 0 ? 512 / p->D : 1;
        terminal_kernel<F><<<64, lanes * p->D, 0, st>>>(records_dev, counter_dev, capacity, p->frames.get(), p->plane, age_old, p->st.get(), terminal_out_dev,
                                                        p->k, newest_old, (float)p->clip);
        p->launches += 1;
    }
    CK(cudaGetLastError());
    p->age_cur ^= 1;  // returns_kernel wrote the new ages; done_corr / terminal above used the old ones
    return launch_normalize_t<F>(p, out_dev, 0, st);
}

extern "C" {

int hlynr_post_create(int64_t n_envs, int device, int n_stack, double clip_obs, double epsilon, double gamma, hlynr_post_t** out) {
    return hlynr_post_create_frames(n_envs, device, OD, n_stack, clip_obs, epsilon, gamma, out);
}

int hlynr_post_create_frames(int64_t n_envs, int device, int frame_dim, int n_stack, double clip_obs, double epsilon, double gamma,
                             hlynr_post_t** out) {
    if (!out) return fail("hlynr_post_create: null argument");
    if (n_envs <= 0) return fail("hlynr_post_create: n_envs must be positive");
    if (frame_dim != OD && frame_dim != 17) return fail("hlynr_post_create: frame_dim must be 26 or 17, got %d", frame_dim);
    if (n_stack < 1 || n_stack > KMAX) return fail("hlynr_post_create: n_stack must be in [1, %d]", KMAX);
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail("hlynr_post_create: device %d not available", device);
    DeviceGuard g(device);
    std::unique_ptr<hlynr_post> p(new (std::nothrow) hlynr_post());
    if (!p) return fail("hlynr_post_create: out of host memory");
    p->n = n_envs; p->device = device; p->fw = frame_dim; p->k = n_stack; p->D = frame_dim * n_stack;
    p->clip = clip_obs; p->eps = epsilon; p->gamma = gamma;
    p->plane = ((n_envs * frame_dim + 31) / 32) * 32;  // every slot starts 128-byte aligned
    CK(cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, device));
    const size_t partial_words = PART_WORDS * ((size_t)p->sm_count * 8 + 64);
    CK(alloc(p->frames, p->plane * n_stack));
    CK(alloc(p->age[0], n_envs));
    CK(alloc(p->age[1], n_envs));
    CK(alloc(p->returns, n_envs));
    CK(alloc(p->st, 1));
    CK(alloc(p->partials, partial_words));
    CK(cudaMemset(p->partials.get(), 0, sizeof(double) * partial_words));
    CK(cudaMemset(p->frames.get(), 0, sizeof(float) * p->plane * n_stack));
    CK(cudaMemset(p->age[0].get(), 0, n_envs)); CK(cudaMemset(p->age[1].get(), 0, n_envs));
    CK(cudaMemset(p->returns.get(), 0, sizeof(double) * n_envs));
    std::unique_ptr<PostStats> h(new (std::nothrow) PostStats());   // value-initialised: all zeros
    if (!h) return fail("hlynr_post_create: out of host memory");
    for (int f = 0; f < DMAX; ++f) { h->var[f] = 1.0; h->inv_std[f] = 1.0 / sqrt(1.0 + epsilon); }
    h->count = 1e-4; h->ret_var = 1.0; h->ret_count = 1e-4;  // RunningMeanStd(epsilon=1e-4)
    CK(cudaMemcpy(p->st.get(), h.get(), sizeof(*h), cudaMemcpyHostToDevice));
    *out = p.release();
    return 0;
}

void hlynr_post_destroy(hlynr_post_t* p) {
    if (!p) return;
    DeviceGuard g(p->device);
    delete p;
}

int hlynr_post_obs_dim(const hlynr_post_t* p, int* out) { if (!p || !out) return fail("null argument"); *out = p->D; return 0; }
int hlynr_post_launch_count(const hlynr_post_t* p, int64_t* out) { if (!p || !out) return fail("null argument"); *out = p->launches; return 0; }

int hlynr_post_note_replayed_steps(hlynr_post_t* p, int64_t steps, int64_t launches) {
    if (!p) return fail("hlynr_post_note_replayed_steps: null handle");
    p->t = (uint32_t)((int64_t)p->t + steps); p->launches += launches;  // negative: undo the bookkeeping of recorded-only calls
    return 0;
}

int hlynr_post_obs_target(hlynr_post_t* p, float** obs_dev) {
    if (!p || !obs_dev) return fail("hlynr_post_obs_target: null argument");
    *obs_dev = p->frames.get() + (int64_t)(p->t % (uint32_t)p->k) * p->plane;
    return 0;
}

int hlynr_post_reset(hlynr_post_t* p, float* out_dev, int training, void* stream) {
    if (!p || !out_dev) return fail("hlynr_post_reset: null argument");
    DeviceGuard g(p->device);
    cudaStream_t st = (cudaStream_t)stream;
    return with_width(p, [&](auto F) { return reset_t<F>(p, out_dev, training, st); });
}

int hlynr_post_step(hlynr_post_t* p, const float* reward_dev, const uint8_t* terminated_dev, const uint8_t* truncated_dev,
                    const HlynrDoneRecord* records_dev, const int32_t* counter_dev, int32_t capacity, float* out_dev,
                    float* terminal_out_dev, int training, void* stream) {
    if (!p || !reward_dev || !terminated_dev || !truncated_dev || !out_dev) return fail("hlynr_post_step: null argument");
    if (p->t == 0) return fail("hlynr_post_step: call hlynr_post_reset first");
    const bool can_maintain = p->k == 1 || (records_dev && counter_dev);
    if (training && !can_maintain) return fail("hlynr_post_step: training with n_stack > 1 needs the done list of the step");
    if (training && !p->sums_valid)
        return fail("hlynr_post_step: the column sums are stale (earlier steps ran without a done list); call hlynr_post_check_sums(resync=1) first");
    if (terminal_out_dev && (!records_dev || !counter_dev)) return fail("hlynr_post_step: terminal_out_dev needs the done list of the step");
    DeviceGuard g(p->device);
    cudaStream_t st = (cudaStream_t)stream;
    return with_width(p, [&](auto F) {
        return step_t<F>(p, reward_dev, terminated_dev, truncated_dev, records_dev, counter_dev, capacity, out_dev, terminal_out_dev,
                         training, can_maintain, st);
    });
}

int hlynr_post_original(hlynr_post_t* p, float* out_dev, void* stream) {
    if (!p || !out_dev) return fail("hlynr_post_original: null argument");
    if (p->t == 0) return fail("hlynr_post_original: no observation yet");
    DeviceGuard g(p->device);
    return launch_normalize(p, out_dev, 1, (cudaStream_t)stream);
}

int hlynr_post_normalize(hlynr_post_t* p, const float* stacked_dev, int64_t rows, float* out_dev, void* stream) {
    if (!p || !stacked_dev || !out_dev) return fail("hlynr_post_normalize: null argument");
    if (rows <= 0) return 0;
    DeviceGuard g(p->device);
    const int lanes = 512 / p->D > 0 ? 512 / p->D : 1;
    normalize_rows_kernel<<<blocks_for(p, rows, lanes), lanes * p->D, 0, (cudaStream_t)stream>>>(stacked_dev, out_dev, rows, p->D, p->st.get(), (float)p->clip);
    CK(cudaGetLastError());
    p->launches += 1;
    return 0;
}

int hlynr_post_get_stats(hlynr_post_t* p, double* mean, double* var, double* count, double* ret_mean, double* ret_var,
                         double* ret_count, void* stream) {
    if (!p) return fail("hlynr_post_get_stats: null handle");
    DeviceGuard g(p->device);
    std::unique_ptr<PostStats> h(new (std::nothrow) PostStats());
    if (!h) return fail("out of host memory");
    CK(cudaMemcpyAsync(h.get(), p->st.get(), sizeof(*h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    if (mean) memcpy(mean, h->mean, sizeof(double) * p->D);
    if (var) memcpy(var, h->var, sizeof(double) * p->D);
    if (count) *count = h->count;
    if (ret_mean) *ret_mean = h->ret_mean;
    if (ret_var) *ret_var = h->ret_var;
    if (ret_count) *ret_count = h->ret_count;
    return 0;
}

int hlynr_post_set_stats(hlynr_post_t* p, const double* mean, const double* var, double count, double ret_mean, double ret_var,
                         double ret_count, void* stream) {
    if (!p || !mean || !var) return fail("hlynr_post_set_stats: null argument");
    DeviceGuard g(p->device);
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaMemcpyAsync(p->st->mean, mean, sizeof(double) * p->D, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(p->st->var, var, sizeof(double) * p->D, cudaMemcpyHostToDevice, st));
    const double tail[4] = {count, ret_mean, ret_var, ret_count};
    CK(cudaMemcpyAsync(&p->st->count, &tail[0], sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(&p->st->ret_mean, &tail[1], sizeof(double) * 3, cudaMemcpyHostToDevice, st));
    with_width(p, [&](auto F) { merge_kernel<F><<<1, 256, 0, st>>>(p->st.get(), p->k, (double)p->n, 0, 0, 0, 0, p->eps); });  // refresh inv_std
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));  // `tail` is a stack array
    p->launches += 1;
    return 0;
}

static_assert(sizeof(HlynrPostSnapshotInfo) == 104, "HlynrPostSnapshotInfo is mirrored by abi.HlynrPostSnapshotInfo");
size_t hlynr_post_snapshot_info_size(void) { return sizeof(HlynrPostSnapshotInfo); }

static void post_snapshot_describe(const hlynr_post* p, HlynrPostSnapshotInfo* info) {
    memset(info, 0, sizeof(*info));
    info->format_version = HLYNR_POST_SNAPSHOT_VERSION;
    info->frame_dim = p->fw; info->n_stack = p->k; info->sums_valid = p->sums_valid ? 1 : 0;
    info->n_envs = p->n; info->t = p->t;
    info->clip_obs = p->clip; info->epsilon = p->eps; info->gamma = p->gamma;
    info->stats_bytes = sizeof(PostStats);
    const size_t n = (size_t)p->n;
    const size_t bytes[HLYNR_POST_SNAP_SECTIONS] = {sizeof(float) * n * p->fw * p->k, n, sizeof(double) * n, sizeof(PostStats)};
    size_t off = 0;
    for (int j = 0; j < HLYNR_POST_SNAP_SECTIONS; ++j) { info->section_offset[j] = off; off += (bytes[j] + 255) & ~size_t(255); }
    info->device_bytes = off;
}
// Copies the frame ring between the handle (slot t % k is written next) and the image (oldest frame first), in either direction.
static int post_snapshot_copy(hlynr_post* p, const HlynrPostSnapshotInfo& info, char* base, bool save, cudaStream_t st) {
    const size_t slot = sizeof(float) * (size_t)p->n * p->fw;
    const int newest = (int)((p->t - 1) % (uint32_t)p->k);
    for (int j = 0; j < p->k; ++j) {
        float* ring = p->frames.get() + (int64_t)((newest - (p->k - 1 - j) + p->k) % p->k) * p->plane;
        char* img = base + info.section_offset[HLYNR_POST_SNAP_FRAMES] + (size_t)j * slot;
        CK(cudaMemcpyAsync(save ? (void*)img : (void*)ring, save ? (const void*)ring : (const void*)img, slot, cudaMemcpyDeviceToDevice, st));
    }
    uint8_t* age = p->age[p->age_cur].get();
    char* img_age = base + info.section_offset[HLYNR_POST_SNAP_AGE];
    char* img_ret = base + info.section_offset[HLYNR_POST_SNAP_RETURNS];
    char* img_st = base + info.section_offset[HLYNR_POST_SNAP_STATS];
    if (save) {
        CK(cudaMemcpyAsync(img_age, age, (size_t)p->n, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(img_ret, p->returns.get(), sizeof(double) * p->n, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(img_st, p->st.get(), sizeof(PostStats), cudaMemcpyDeviceToDevice, st));
    } else {
        CK(cudaMemcpyAsync(age, img_age, (size_t)p->n, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(p->returns.get(), img_ret, sizeof(double) * p->n, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(p->st.get(), img_st, sizeof(PostStats), cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

int hlynr_post_snapshot_layout(const hlynr_post_t* p, HlynrPostSnapshotInfo* info, size_t* device_bytes) {
    if (!p || !info || !device_bytes) return fail("hlynr_post_snapshot_layout: null argument");
    post_snapshot_describe(p, info);
    *device_bytes = (size_t)info->device_bytes;
    return 0;
}

int hlynr_post_snapshot_save(hlynr_post_t* p, void* dev_out, HlynrPostSnapshotInfo* info, void* stream) {
    if (!p || !dev_out || !info) return fail("hlynr_post_snapshot_save: null argument");
    DeviceGuard g(p->device);
    const cudaStream_t st = (cudaStream_t)stream;
    if (refuse_capture(st, "hlynr_post_snapshot_save")) return 1;
    post_snapshot_describe(p, info);
    return post_snapshot_copy(p, *info, (char*)dev_out, true, st);
}

int hlynr_post_snapshot_load(hlynr_post_t* p, const HlynrPostSnapshotInfo* info, const void* dev_in, void* stream) {
    if (!p || !info || !dev_in) return fail("hlynr_post_snapshot_load: null argument");
    HlynrPostSnapshotInfo mine;
    post_snapshot_describe(p, &mine);
    const HlynrPostSnapshotInfo& in = *info;
#define HLYNR_POST_REFUSE(cond, what, ...) \
    if (cond) return fail("hlynr_post_snapshot_load: the snapshot's " what " differs from the pipeline's: " __VA_ARGS__)
    HLYNR_POST_REFUSE(in.format_version != mine.format_version, "format version", "%d, expected %d", in.format_version, mine.format_version);
    HLYNR_POST_REFUSE(in.n_envs != mine.n_envs, "n_envs", "%lld, the pipeline has %lld", (long long)in.n_envs, (long long)mine.n_envs);
    HLYNR_POST_REFUSE(in.frame_dim != mine.frame_dim, "frame width", "%d, the pipeline has %d", in.frame_dim, mine.frame_dim);
    HLYNR_POST_REFUSE(in.n_stack != mine.n_stack, "n_stack", "%d, the pipeline has %d", in.n_stack, mine.n_stack);
    HLYNR_POST_REFUSE(memcmp(&in.clip_obs, &mine.clip_obs, sizeof(double)) != 0, "clip_obs", "%g, the pipeline has %g", in.clip_obs, mine.clip_obs);
    HLYNR_POST_REFUSE(memcmp(&in.epsilon, &mine.epsilon, sizeof(double)) != 0, "epsilon", "%g, the pipeline has %g", in.epsilon, mine.epsilon);
    HLYNR_POST_REFUSE(memcmp(&in.gamma, &mine.gamma, sizeof(double)) != 0, "gamma", "%g, the pipeline has %g", in.gamma, mine.gamma);
    HLYNR_POST_REFUSE(in.stats_bytes != mine.stats_bytes, "statistics block", "%llu bytes, expected %llu", (unsigned long long)in.stats_bytes,
                      (unsigned long long)mine.stats_bytes);
    for (int j = 0; j < HLYNR_POST_SNAP_SECTIONS; ++j)
        HLYNR_POST_REFUSE(in.section_offset[j] != mine.section_offset[j], "image layout", "offset of section %d", j);
    HLYNR_POST_REFUSE(in.device_bytes != mine.device_bytes, "image size", "%llu bytes, expected %llu", (unsigned long long)in.device_bytes,
                      (unsigned long long)mine.device_bytes);
#undef HLYNR_POST_REFUSE
    DeviceGuard g(p->device);
    const cudaStream_t st = (cudaStream_t)stream;
    if (refuse_capture(st, "hlynr_post_snapshot_load")) return 1;
    p->t = (uint32_t)in.t; p->sums_valid = in.sums_valid != 0;   // the ring slots follow the restored t
    return post_snapshot_copy(p, in, (char*)dev_in, false, st);
}

int hlynr_post_check_sums(hlynr_post_t* p, int resync, double* max_abs_diff, void* stream) {
    if (!p || !max_abs_diff) return fail("hlynr_post_check_sums: null argument");
    if (p->t == 0) return fail("hlynr_post_check_sums: no observation yet");
    DeviceGuard g(p->device);
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaMemsetAsync(p->st->chk_S, 0, sizeof(double) * KMAX * OD * 2, st));
    const int lanes = 512 / p->D > 0 ? 512 / p->D : 1;
    const int newest = (int)((p->t - 1) % (uint32_t)p->k);
    with_width(p, [&](auto F) {
        recompute_sums_kernel<F><<<blocks_for(p, p->n, lanes), lanes * p->D, 0, st>>>(p->frames.get(), p->plane, p->age[p->age_cur].get(), p->n, p->k,
                                                                                     newest, p->st.get());
    });
    CK(cudaGetLastError());
    p->launches += 1;
    std::unique_ptr<PostStats> h(new (std::nothrow) PostStats());
    if (!h) return fail("out of host memory");
    CK(cudaMemcpyAsync(h.get(), p->st.get(), sizeof(*h), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    double m = 0.0;
    for (int d = 0; d < p->k; ++d)
        for (int c = 0; c < p->fw; ++c) {
            m = fmax(m, fabs(h->S[d][c] - h->chk_S[d][c]));
            m = fmax(m, fabs(h->Q[d][c] - h->chk_Q[d][c]));
        }
    *max_abs_diff = m;
    if (resync) {
        CK(cudaMemcpyAsync(p->st->S, p->st->chk_S, sizeof(double) * KMAX * OD, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(p->st->Q, p->st->chk_Q, sizeof(double) * KMAX * OD, cudaMemcpyDeviceToDevice, st));
        p->sums_valid = true;
    }
    return 0;
}

}  // extern "C"
