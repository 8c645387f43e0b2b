// numerics_probe.cu -- test-only elementwise / per-warp wrappers of the search's numeric primitives.
// It includes the engine's own headers, so what tests/test_numerics_gpu.py measures is the code the
// kernels run.  Host entry points take host arrays, copy them in, run one kernel and copy the result
// out; they return 0 or the CUDA error code.
#include "gmz_internal.h"
#include "gmz_tree.cuh"
#include "gmz_play.cuh"

__global__ void k_exp_nonpos(const double *x, double *y, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = exp_nonpos(x[i]);
}
// d as the certified select passes it: a float64 difference rounded to float32 (gmz_tree.cuh select_interior)
__global__ void k_exp_approx(const double *d, float *y, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = exp_approx((float)d[i]);
}
__global__ void k_rcp(const double *x, float *ra, double *rn, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { ra[i] = rcp_approx((float)x[i]); rn[i] = rcp_newton(x[i]); }
}
// n = 32 * warps; every lane writes what it got back
__global__ void k_warp_sum_fx(const float *v, float *y, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i - (i & 31) >= n) return;
    y[i] = warp_sum_fx(v[i]);
}
__global__ void k_warp_sum_f64(const double *v, double *y, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i - (i & 31) >= n) return;
    y[i] = warp_sum_f64(v[i]);
}
__global__ void k_warp_ext(const double *v, double *mx, double *mn, unsigned long long *mk, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i - (i & 31) >= n) return;
    mx[i] = warp_max_f64(v[i]);
    mn[i] = warp_min_f64(v[i]);
    mk[i] = warp_max_key(f64_key(v[i]));
}
__global__ void k_keys(const double *x, unsigned long long *k, double *back, const float *xf, unsigned *kf, float *backf, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    k[i] = f64_key(x[i]); back[i] = f64_unkey(k[i]);
    kf[i] = f32_key(xf[i]); backf[i] = f32_unkey(kf[i]);
}

namespace {
struct Dev {
    void *p = nullptr;
    cudaError_t err = cudaSuccess;
    Dev(size_t bytes, const void *host = nullptr)
    {
        err = cudaMalloc(&p, bytes ? bytes : 1);
        if (err == cudaSuccess && host) err = cudaMemcpy(p, host, bytes, cudaMemcpyHostToDevice);
    }
    ~Dev() { if (p) cudaFree(p); }
    template <class T> T *as() const { return static_cast<T *>(p); }
};
int finish(cudaError_t e) { return e != cudaSuccess ? (int)e : (int)cudaDeviceSynchronize(); }
int copy_out(void *host, const Dev &d, size_t bytes)
{
    return (int)cudaMemcpy(host, d.p, bytes, cudaMemcpyDeviceToHost);
}
unsigned blocks(int n) { return (unsigned)((n + 255) / 256); }
}  // namespace

#define PROBE_CHECK(x) do { const int rc_ = (int)(x); if (rc_) return rc_; } while (0)

extern "C" double probe_cert_eps() { return kCertEps; }

extern "C" int probe_exp_nonpos(const double *x, double *y, int n)
{
    Dev dx(n * sizeof(double), x), dy(n * sizeof(double));
    PROBE_CHECK(dx.err); PROBE_CHECK(dy.err);
    k_exp_nonpos<<<blocks(n), 256>>>(dx.as<double>(), dy.as<double>(), n);
    PROBE_CHECK(finish(cudaGetLastError()));
    return copy_out(y, dy, n * sizeof(double));
}

extern "C" int probe_exp_approx(const double *d, float *y, int n)
{
    Dev dd(n * sizeof(double), d), dy(n * sizeof(float));
    PROBE_CHECK(dd.err); PROBE_CHECK(dy.err);
    k_exp_approx<<<blocks(n), 256>>>(dd.as<double>(), dy.as<float>(), n);
    PROBE_CHECK(finish(cudaGetLastError()));
    return copy_out(y, dy, n * sizeof(float));
}

extern "C" int probe_rcp(const double *x, float *ra, double *rn, int n)
{
    Dev dx(n * sizeof(double), x), da(n * sizeof(float)), dn(n * sizeof(double));
    PROBE_CHECK(dx.err); PROBE_CHECK(da.err); PROBE_CHECK(dn.err);
    k_rcp<<<blocks(n), 256>>>(dx.as<double>(), da.as<float>(), dn.as<double>(), n);
    PROBE_CHECK(finish(cudaGetLastError()));
    PROBE_CHECK(copy_out(ra, da, n * sizeof(float)));
    return copy_out(rn, dn, n * sizeof(double));
}

// n must be a multiple of 32 (one warp per 32 consecutive values)
extern "C" int probe_warp_sum_fx(const float *v, float *y, int n)
{
    if (n % 32) return -1;
    Dev dv(n * sizeof(float), v), dy(n * sizeof(float));
    PROBE_CHECK(dv.err); PROBE_CHECK(dy.err);
    k_warp_sum_fx<<<blocks(n), 256>>>(dv.as<float>(), dy.as<float>(), n);
    PROBE_CHECK(finish(cudaGetLastError()));
    return copy_out(y, dy, n * sizeof(float));
}

extern "C" int probe_warp_sum_f64(const double *v, double *y, int n)
{
    if (n % 32) return -1;
    Dev dv(n * sizeof(double), v), dy(n * sizeof(double));
    PROBE_CHECK(dv.err); PROBE_CHECK(dy.err);
    k_warp_sum_f64<<<blocks(n), 256>>>(dv.as<double>(), dy.as<double>(), n);
    PROBE_CHECK(finish(cudaGetLastError()));
    return copy_out(y, dy, n * sizeof(double));
}

extern "C" int probe_warp_ext(const double *v, double *mx, double *mn, unsigned long long *mk, int n)
{
    if (n % 32) return -1;
    Dev dv(n * sizeof(double), v), dx(n * sizeof(double)), dn(n * sizeof(double)), dk(n * sizeof(unsigned long long));
    PROBE_CHECK(dv.err); PROBE_CHECK(dx.err); PROBE_CHECK(dn.err); PROBE_CHECK(dk.err);
    k_warp_ext<<<blocks(n), 256>>>(dv.as<double>(), dx.as<double>(), dn.as<double>(), dk.as<unsigned long long>(), n);
    PROBE_CHECK(finish(cudaGetLastError()));
    PROBE_CHECK(copy_out(mx, dx, n * sizeof(double)));
    PROBE_CHECK(copy_out(mn, dn, n * sizeof(double)));
    return copy_out(mk, dk, n * sizeof(unsigned long long));
}

extern "C" int probe_keys(const double *x, unsigned long long *k, double *back, const float *xf, unsigned *kf, float *backf, int n)
{
    Dev dx(n * sizeof(double), x), dk(n * sizeof(unsigned long long)), db(n * sizeof(double));
    Dev dxf(n * sizeof(float), xf), dkf(n * sizeof(unsigned)), dbf(n * sizeof(float));
    PROBE_CHECK(dx.err); PROBE_CHECK(dk.err); PROBE_CHECK(db.err);
    PROBE_CHECK(dxf.err); PROBE_CHECK(dkf.err); PROBE_CHECK(dbf.err);
    k_keys<<<blocks(n), 256>>>(dx.as<double>(), dk.as<unsigned long long>(), db.as<double>(), dxf.as<float>(),
                               dkf.as<unsigned>(), dbf.as<float>(), n);
    PROBE_CHECK(finish(cudaGetLastError()));
    PROBE_CHECK(copy_out(k, dk, n * sizeof(unsigned long long)));
    PROBE_CHECK(copy_out(back, db, n * sizeof(double)));
    PROBE_CHECK(copy_out(kf, dkf, n * sizeof(unsigned)));
    return copy_out(backf, dbf, n * sizeof(float));
}
