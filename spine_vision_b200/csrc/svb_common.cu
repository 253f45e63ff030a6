// svb_common.cu -- host utilities: error string, device check, TMA descriptor encoding.
#include "svb_common.cuh"

#include <atomic>
#include <cstring>
#include <mutex>

namespace svb {

std::string& last_error_ref() {
    static thread_local std::string err;
    return err;
}

int set_error(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error_ref() = buf;
    return code;
}

static std::atomic<long long> g_launches{0};
void count_launch(long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long long launches_total(bool reset) { return reset ? g_launches.exchange(0) : g_launches.load(); }

int check_device_sm100() {
    int dev = 0;
    SVB_CUDA_OK(cudaGetDevice(&dev));
    int major = 0, minor = 0;
    SVB_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    SVB_CUDA_OK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
    SVB_REQUIRE(major == 10 && minor == 0, SVB_ERR_UNSUPPORTED_DEVICE,
                "libspine_b200 is built for sm_100a (B200) only; device %d is sm_%d%d and there is no fallback",
                dev, major, minor);
    return SVB_OK;
}

long long launches_total(bool reset);
int num_sms() {
    static int cached = 0;
    if (cached) return cached;
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
    cached = n;
    return n;
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    });
    return fn;
}

int encode_tmap(CUtensorMap* map, CUtensorMapDataType dt, uint32_t rank, const void* base, const uint64_t* dims,
                const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz) {
    PFN_encodeTiled fn = get_encode_fn();
    SVB_REQUIRE(fn != nullptr, SVB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    cuuint64_t gdims[5];
    cuuint64_t gstr[5];
    cuuint32_t gbox[5];
    for (uint32_t i = 0; i < rank; ++i) {
        gdims[i] = dims[i];
        gbox[i] = box[i];
        if (i + 1 < rank) gstr[i] = strides_bytes[i];
    }
    CUresult r = fn(map, dt, rank, const_cast<void*>(base), gdims, gstr, gbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SVB_REQUIRE(r == CUDA_SUCCESS, SVB_ERR_CUDA,
                "cuTensorMapEncodeTiled failed (%d): rank %u dims [%llu,%llu,..] box [%u,%u,..]", (int)r, rank,
                (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0), box[0],
                rank > 1 ? box[1] : 0);
    return SVB_OK;
}

}  // namespace svb

extern "C" {
int svb_version(void) { return SVB_VERSION; }
const char* svb_last_error(void) { return svb::last_error_ref().c_str(); }
int svb_device_check(void) { return svb::check_device_sm100(); }
long long svb_launch_count(int reset) { return svb::launches_total(reset != 0); }
}
