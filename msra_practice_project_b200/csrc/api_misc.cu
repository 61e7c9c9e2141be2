// Error reporting, version and argument checks shared by every entry point of libb2r.
#include <cmath>
#include "common.cuh"

namespace b2r {

char* err_buf() {
    static thread_local char buf[512] = {0};
    return buf;
}

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(err_buf(), 512, fmt, ap);
    va_end(ap);
    return code;
}

int check_mlp_input(const b2r_mlp_input* in) {
    B2R_CHECK_ARG(in != nullptr, "mlp input descriptor is NULL");
    int modes = (in->rays != nullptr) + (in->x != nullptr) + (in->grid_n > 0) + lattice_mode(in);
    B2R_CHECK_ARG(modes == 1, "exactly one of rays / x / grid_n / lattice_dims must be given (got %d)", modes);
    B2R_CHECK_ARG(in->n_rays >= 0, "n_rays < 0");
    if (in->rays) {
        B2R_CHECK_ARG(in->z != nullptr, "rays mode needs z");
        B2R_CHECK_ARG(in->n_samples >= 1, "rays mode needs n_samples >= 1");
    } else {
        B2R_CHECK_ARG(in->n_samples == 1, "x / grid mode needs n_samples == 1");
    }
    if (in->grid_n > 0) {
        B2R_CHECK_ARG(in->grid_n >= 2, "grid_n must be >= 2");
        long long n3 = (long long)in->grid_n * in->grid_n * in->grid_n;
        B2R_CHECK_ARG(in->grid_begin >= 0 && in->grid_begin + in->n_rays <= n3, "grid range outside the N^3 lattice");
    }
    if (lattice_mode(in)) {
        const int* d = in->lattice_dims;
        B2R_CHECK_ARG(d[0] >= 2 && d[1] >= 2 && d[2] >= 2, "lattice_dims: every axis needs n >= 2 (got %d x %d x %d)", d[0], d[1], d[2]);
        const long long pts = (long long)d[0] * d[1] * d[2];
        B2R_CHECK_ARG(pts <= INT32_MAX, "lattice of %lld points exceeds INT32_MAX", pts);
        B2R_CHECK_ARG(in->lattice_voxel > 0.f && std::isfinite(in->lattice_voxel), "lattice_voxel must be finite and > 0 (got %g)",
                      (double)in->lattice_voxel);
        B2R_CHECK_ARG(in->grid_begin >= 0 && in->grid_begin + in->n_rays <= pts, "lattice range [%lld, %lld) outside the %lld points",
                      in->grid_begin, in->grid_begin + in->n_rays, pts);
    }
    return 0;
}

}  // namespace b2r

extern "C" const char* b2r_last_error(void) { return b2r::err_buf(); }
extern "C" int b2r_version(void) { return B2R_VERSION; }

extern "C" int b2r_device_ok(void) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 0; }
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) { cudaGetLastError(); return 0; }
    return major == 10 ? 1 : 0;
}
