// Library-wide pieces of the C-ABI: error state, device capabilities, tuning options.
#include <stdarg.h>

#include "score_common.cuh"

namespace phm {

static thread_local char g_error[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int time_kernels = 0;

unsigned long long kernel_launches = 0;

// device attributes, cached per device ordinal (a process may drive several GPUs from several threads)
static constexpr int kMaxDevices = 64;
static int g_sm_count[kMaxDevices], g_smem_optin[kMaxDevices];

static int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return (dev >= 0 && dev < kMaxDevices) ? dev : 0;
}

int sm_count() {
    const int dev = current_device();
    if (g_sm_count[dev] == 0) {
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        g_sm_count[dev] = v > 0 ? v : 148;
    }
    return g_sm_count[dev];
}
int max_smem_optin() {
    const int dev = current_device();
    if (g_smem_optin[dev] == 0) {
        int v = 0;
        cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        g_smem_optin[dev] = v;
    }
    return g_smem_optin[dev];
}

extern int hist_stride_for_k4;
extern int hist_stride_for_k5;
extern int hist_warps_k6;
extern int hist_warps_k5;
extern int hist_tma;
extern int hist_canonical_swizzle;
extern int hist_plan;
extern int score_path;
extern int score_collect_stats;
extern int score_list_pass;
extern int score_force_fallback;
int kmer_hist_last_ms(float *ms);

}  // namespace phm

using namespace phm;

extern "C" int phm_version(void) { return PHM_VERSION; }

extern "C" const char *phm_last_error(void) { return g_error; }

extern "C" int phm_device_caps(phm_caps *out) {
    PHM_REQUIRE(out != nullptr, "out is null");
    int dev = 0;
    PHM_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    PHM_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    out->device = dev;
    out->sm_major = prop.major;
    out->sm_minor = prop.minor;
    out->sm_count = prop.multiProcessorCount;
    out->max_smem_optin = (int32_t)prop.sharedMemPerBlockOptin;
    out->hbm_bytes = (int64_t)prop.totalGlobalMem;
    if (prop.major != 10) {
        set_error("phamers_b200 is built for sm_100a only; device %d is sm_%d%d", dev, prop.major, prop.minor);
        return PHM_E_UNSUPPORTED;
    }
    return PHM_OK;
}

// Tuning knobs for experiments (bench.py --opt name=value).  Unknown names are an error.
extern "C" int phm_set_option(const char *name, int64_t value) {
    PHM_REQUIRE(name != nullptr, "name is null");
    if (!strcmp(name, "hist_stride_k4")) { PHM_REQUIRE(value == 1 || value == 2, "1 or 2"); hist_stride_for_k4 = (int)value; return PHM_OK; }
    if (!strcmp(name, "hist_stride_k5")) { PHM_REQUIRE(value >= 0 && value <= 2, "0 (automatic), 1 or 2"); hist_stride_for_k5 = (int)value; return PHM_OK; }
    if (!strcmp(name, "hist_canonical_swizzle")) { hist_canonical_swizzle = value != 0; return PHM_OK; }
    if (!strcmp(name, "hist_plan")) { hist_plan = value != 0; return PHM_OK; }
    if (!strcmp(name, "hist_tma")) { hist_tma = value != 0; return PHM_OK; }
    if (!strcmp(name, "hist_warps_k5")) { PHM_REQUIRE(value == 8 || value == 18, "8 or 18"); hist_warps_k5 = (int)value; return PHM_OK; }
    if (!strcmp(name, "hist_warps_k6")) { PHM_REQUIRE(value == 4 || value == 13, "4 or 13"); hist_warps_k6 = (int)value; return PHM_OK; }
    if (!strcmp(name, "score_path")) { PHM_REQUIRE(value >= 0 && value <= 2, "0 auto, 1 exact, 2 tensor cores"); score_path = (int)value; return PHM_OK; }
    if (!strcmp(name, "time_kernels")) { time_kernels = value != 0; return PHM_OK; }
    if (!strcmp(name, "score_force_fallback")) { score_force_fallback = value != 0; return PHM_OK; }
    if (!strcmp(name, "score_stats")) { score_collect_stats = value != 0; return PHM_OK; }
    if (!strcmp(name, "score_list_pass")) { score_list_pass = value != 0; return PHM_OK; }
    set_error("unknown option '%s'", name);
    return PHM_E_ARG;
}

extern "C" uint64_t phm_kernel_launches(void) { return (uint64_t)kernel_launches; }

// Device time of the most recent launch of a named hot kernel (bench.py's roofline numerator); synchronises on that launch.
extern "C" int phm_last_kernel_ms(const char *kernel, float *ms) {
    PHM_REQUIRE(kernel != nullptr && ms != nullptr, "null pointer");
    if (!strcmp(kernel, "score_tc_kernel")) return tc::score_tc_last_ms(ms);
    if (!strcmp(kernel, "score_decide_kernel")) return tc::score_decide_last_ms(ms);
    if (!strcmp(kernel, "kmer_hist_kernel")) return kmer_hist_last_ms(ms);
    set_error("no timing hook for kernel '%s'", kernel);
    return PHM_E_ARG;
}
