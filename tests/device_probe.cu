// device_probe.cu -- test-only launchers for the arithmetic helpers of the step kernel (csrc/hlynr_device.cuh), so that
// tests/test_device_math.py can run each helper on the device, element by element, against a float64 or exact reference.
// Not part of the library (hlynr_intercept_b200/build.py does not compile it): the test builds it into a temporary directory.
//
// Every launcher takes device pointers, an element count and a cudaStream_t (as void*), launches one grid-stride kernel
// and returns the cudaError_t of the launch.  Arrays of vectors are element-major: a[3 * i + k] is component k of element i.
#include "../hlynr_intercept_b200/csrc/hlynr_device.cuh"

using namespace hlynr;

#define EACH(n) for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)
static unsigned blocks(int64_t n) { return (unsigned)(n <= 0 ? 1 : (n + 255) / 256 < 8192 ? (n + 255) / 256 : 8192); }
#define GRID(n) blocks(n), 256, 0, (cudaStream_t)stream
#define LAUNCHED return (int)cudaGetLastError()

// ---- divisions, reciprocals, square roots -------------------------------------------------------------------------------
__global__ void k_cdiv_f(const float* x, float c, float rc, float* y, int64_t n) { EACH(n) y[i] = cdiv(x[i], c, rc); }
__global__ void k_cdiv_d(const double* x, double c, double rc, double* y, int64_t n) { EACH(n) y[i] = cdiv(x[i], c, rc); }
__global__ void k_drcp(const double* b, double* y, int64_t n) { EACH(n) y[i] = drcp(b[i]); }
__global__ void k_nrcp_d(const double* b, double* y, int64_t n) { EACH(n) y[i] = nrcp(b[i]); }
__global__ void k_dvd_d(const double* a, const double* b, double* y, int64_t n) { EACH(n) y[i] = dvd(a[i], b[i]); }
__global__ void k_sqr_d(const double* a, double* y, int64_t n) { EACH(n) y[i] = sqr(a[i]); }

extern "C" int probe_cdiv_f(const float* x, float c, float rc, float* y, int64_t n, void* stream) {
    k_cdiv_f<<<GRID(n)>>>(x, c, rc, y, n); LAUNCHED;
}
extern "C" int probe_cdiv_d(const double* x, double c, double rc, double* y, int64_t n, void* stream) {
    k_cdiv_d<<<GRID(n)>>>(x, c, rc, y, n); LAUNCHED;
}
extern "C" int probe_drcp(const double* b, double* y, int64_t n, void* stream) { k_drcp<<<GRID(n)>>>(b, y, n); LAUNCHED; }
extern "C" int probe_nrcp_d(const double* b, double* y, int64_t n, void* stream) { k_nrcp_d<<<GRID(n)>>>(b, y, n); LAUNCHED; }
extern "C" int probe_dvd_d(const double* a, const double* b, double* y, int64_t n, void* stream) {
    k_dvd_d<<<GRID(n)>>>(a, b, y, n); LAUNCHED;
}
extern "C" int probe_sqr_d(const double* a, double* y, int64_t n, void* stream) { k_sqr_d<<<GRID(n)>>>(a, y, n); LAUNCHED; }

// ---- dot products -------------------------------------------------------------------------------------------------------
template <typename T> __global__ void k_dot3(const T* a, const T* b, T* y, int64_t n) {
    EACH(n) y[i] = dot3(a[3 * i], a[3 * i + 1], a[3 * i + 2], b[3 * i], b[3 * i + 1], b[3 * i + 2]);
}
__global__ void k_dot2_f(const float* a, const float* b, float* y, int64_t n) { EACH(n) y[i] = dot2(a[2 * i], a[2 * i + 1], b[2 * i], b[2 * i + 1]); }

extern "C" int probe_dot3_f(const float* a, const float* b, float* y, int64_t n, void* stream) { k_dot3<<<GRID(n)>>>(a, b, y, n); LAUNCHED; }
extern "C" int probe_dot3_d(const double* a, const double* b, double* y, int64_t n, void* stream) { k_dot3<<<GRID(n)>>>(a, b, y, n); LAUNCHED; }
extern "C" int probe_dot2_f(const float* a, const float* b, float* y, int64_t n, void* stream) { k_dot2_f<<<GRID(n)>>>(a, b, y, n); LAUNCHED; }

// ---- angles -------------------------------------------------------------------------------------------------------------
__global__ void k_atan2(const float* y, const float* x, float* r, int64_t n) { EACH(n) r[i] = fast_atan2(y[i], x[i]); }
__global__ void k_asin(const float* x, float* r, int64_t n) { EACH(n) r[i] = fast_asin(x[i]); }
__global__ void k_euler(const float* q, float* r, int64_t n) {   // q = (w, x, y, z), r = (roll, pitch, yaw) / pi
    EACH(n) euler_over_pi(q[4 * i], q[4 * i + 1], q[4 * i + 2], q[4 * i + 3], &r[3 * i], &r[3 * i + 1], &r[3 * i + 2]);
}

extern "C" int probe_fast_atan2(const float* y, const float* x, float* r, int64_t n, void* stream) { k_atan2<<<GRID(n)>>>(y, x, r, n); LAUNCHED; }
extern "C" int probe_fast_asin(const float* x, float* r, int64_t n, void* stream) { k_asin<<<GRID(n)>>>(x, r, n); LAUNCHED; }
extern "C" int probe_euler_over_pi(const float* q, float* r, int64_t n, void* stream) { k_euler<<<GRID(n)>>>(q, r, n); LAUNCHED; }

// ---- normal draws -------------------------------------------------------------------------------------------------------
__global__ void k_fast_pair(const uint32_t* xa, const uint32_t* xb, float* z0, float* z1, int64_t n) { EACH(n) fast_pair(xa[i], xb[i], &z0[i], &z1[i]); }
__global__ void k_box_muller(const uint32_t* xa, const uint32_t* xb, float* z0, float* z1, int64_t n) { EACH(n) box_muller(xa[i], xb[i], &z0[i], &z1[i]); }

extern "C" int probe_fast_pair(const uint32_t* xa, const uint32_t* xb, float* z0, float* z1, int64_t n, void* stream) {
    k_fast_pair<<<GRID(n)>>>(xa, xb, z0, z1, n); LAUNCHED;
}
extern "C" int probe_box_muller(const uint32_t* xa, const uint32_t* xb, float* z0, float* z1, int64_t n, void* stream) {
    k_box_muller<<<GRID(n)>>>(xa, xb, z0, z1, n); LAUNCHED;
}

// ---- quaternion integration: q (float32, in place) <- quat_step(q, w, dt); w and dt in the build's type R ---------------
template <typename R> __global__ void k_quat_step(float* q, const R* w, R dt, int64_t n) {
    EACH(n) {
        Env<R> e = {};   // quat_step reads and writes the quaternion only
        e.qw = q[4 * i]; e.qx = q[4 * i + 1]; e.qy = q[4 * i + 2]; e.qz = q[4 * i + 3];
        quat_step(e, w[3 * i], w[3 * i + 1], w[3 * i + 2], dt);
        q[4 * i] = e.qw; q[4 * i + 1] = e.qx; q[4 * i + 2] = e.qy; q[4 * i + 3] = e.qz;
    }
}
extern "C" int probe_quat_step_f(float* q, const float* w, float dt, int64_t n, void* stream) { k_quat_step<<<GRID(n)>>>(q, w, dt, n); LAUNCHED; }
extern "C" int probe_quat_step_d(float* q, const double* w, double dt, int64_t n, void* stream) { k_quat_step<<<GRID(n)>>>(q, w, dt, n); LAUNCHED; }

// ---- ISA atmosphere ----------------------------------------------------------------------------------------------------
template <typename R> __global__ void k_isa(KParams<R> P, const R* T0, const R* alt, R* rho, R* cs, int64_t n) {
    EACH(n) isa_props(P, T0[i], alt[i], &rho[i], &cs[i]);
}
template <typename R> static int isa(const R* T0, const R* alt, R* rho, R* cs, int64_t n, void* stream) {
    KParams<R> P;   // isa_props reads these three fields, filled as make_kparams does (csrc/hlynr_capi.cu:255-256)
    memset(&P, 0, sizeof(P));
    P.isa_expo = (R)(9.80665 / (287.05 * 0.0065));
    P.gas_R = (R)287.05; P.gamma_R = (R)(1.4 * 287.05);
    k_isa<<<GRID(n)>>>(P, T0, alt, rho, cs, n); LAUNCHED;
}
extern "C" int probe_isa_props_f(const float* T0, const float* alt, float* rho, float* cs, int64_t n, void* stream) {
    return isa(T0, alt, rho, cs, n, stream);
}
extern "C" int probe_isa_props_d(const double* T0, const double* alt, double* rho, double* cs, int64_t n, void* stream) {
    return isa(T0, alt, rho, cs, n, stream);
}

// ---- validation guards -------------------------------------------------------------------------------------------------
template <typename R> __global__ void k_any_nonfinite(const R* a, uint8_t* y, int64_t n) { EACH(n) y[i] = any_nonfinite(a[3 * i], a[3 * i + 1], a[3 * i + 2]); }
template <typename R> __global__ void k_nan_guard(const R* a, R lim, R* y, int64_t n) { EACH(n) y[i] = nan_guard(a[i], lim); }

extern "C" int probe_any_nonfinite_f(const float* a, uint8_t* y, int64_t n, void* stream) { k_any_nonfinite<<<GRID(n)>>>(a, y, n); LAUNCHED; }
extern "C" int probe_any_nonfinite_d(const double* a, uint8_t* y, int64_t n, void* stream) { k_any_nonfinite<<<GRID(n)>>>(a, y, n); LAUNCHED; }
extern "C" int probe_nan_guard_f(const float* a, float lim, float* y, int64_t n, void* stream) { k_nan_guard<<<GRID(n)>>>(a, lim, y, n); LAUNCHED; }
extern "C" int probe_nan_guard_d(const double* a, double lim, double* y, int64_t n, void* stream) { k_nan_guard<<<GRID(n)>>>(a, lim, y, n); LAUNCHED; }
