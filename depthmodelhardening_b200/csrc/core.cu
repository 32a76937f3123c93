// Library-level entry points: thread-local error string, version, build arch.
#include <stdarg.h>

#include <atomic>
#include <map>
#include <mutex>
#include <utility>

#include "../../include/dmh_b200.h"
#include "dmh_common.cuh"

namespace dmh {
static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}
static std::atomic<long long> g_launches{0};

// ---- exhaustive check of the 3-instruction division by a launch constant (dmh_math.cuh div_const): all 2^24
// significands of the binades [1,2) and [2,4), both signs.  For a NORMAL quotient without intermediate underflow the
// result depends only on the significand of a, so this covers every a with 2^-100 <= |a| <= FLT_MAX (inf / NaN pass
// through in div_const); below that a * rc may lose bits to underflow and the quotient can differ from IEEE division
// by one subnormal ulp (~1e-45) -- far below anything floor() of a pixel coordinate can see.
__device__ unsigned g_const_div_bad;
__global__ void const_div_check_kernel(float c, float rc) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;          // 2^24 significands: binades [1,2) and [2,4)
    const float a = __uint_as_float(0x3f800000u + i);
    const float q = div_const(a, c, rc), ref = __fdiv_rn(a, c);
    const float qn = div_const(-a, c, rc), refn = __fdiv_rn(-a, c);
    if (__float_as_uint(q) != __float_as_uint(ref) || __float_as_uint(qn) != __float_as_uint(refn))
        atomicAdd(&g_const_div_bad, 1u);
}

bool const_div_exact(int c, float* rc_out, cudaStream_t caller) {
    static std::mutex mu;
    static std::map<std::pair<int, int>, bool> cache;               // (device, c) -> verified
    static std::map<int, cudaStream_t> check_stream;                // one private non-blocking stream per device
    const float rc = (float)(1.0 / (double)c);
    *rc_out = rc;
    if (c < 1) return false;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find({dev, c});
    if (it != cache.end()) return it->second;
    // The check waits for its result, and a synchronisation while the caller's stream is being captured is refused and
    // invalidates the capture (global capture mode, PyTorch's default).  So while the caller's stream captures, the
    // constant is reported as NOT verified and NOT cached, without any call that synchronises: the caller takes the
    // generic IEEE division (same bits), and the first call outside a capture verifies it.
    cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(caller, &capture) != cudaSuccess || capture != cudaStreamCaptureStatusNone) {
        cudaGetLastError();
        return false;
    }
    // First use of this constant on this device: one small launch + a 4-byte read-back, on a PRIVATE non-blocking
    // stream with asynchronous copies (never the legacy stream: no device-wide synchronisation).  If the check cannot
    // run, the constant is likewise reported as not verified and not cached.
    cudaStream_t& cs = check_stream[dev];
    bool ran = true;
    if (!cs) ran = cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking) == cudaSuccess;
    unsigned bad = 0;
    unsigned* dbad = nullptr;
    ran = ran && cudaGetSymbolAddress((void**)&dbad, g_const_div_bad) == cudaSuccess;
    ran = ran && cudaMemsetAsync(dbad, 0, sizeof(unsigned), cs) == cudaSuccess;
    if (ran) {
        const_div_check_kernel<<<(1u << 24) / 256, 256, 0, cs>>>((float)c, rc);
        bad = 1;
        ran = cudaMemcpyAsync(&bad, dbad, sizeof(bad), cudaMemcpyDeviceToHost, cs) == cudaSuccess &&
              cudaStreamSynchronize(cs) == cudaSuccess;
    }
    if (!ran) {
        cudaGetLastError();
        return false;
    }
    cache[{dev, c}] = (bad == 0);
    return bad == 0;
}
void count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- 8-bit frame transport: torchvision's to_tensor (`img.to(float32).div(255)`) on the device.  IEEE division:
// the k/255 the reference's loaders produce, bit for bit (a multiplication by 1/255 differs in the last place for
// about a third of the 256 values).  16 bytes in, 4 x 128-bit stores out per thread; HBM-bound (5 B per element).
__global__ void __launch_bounds__(256) unpack_u8_kernel(const uint8_t* __restrict__ in, long long n, float* __restrict__ out) {
    const long long nv = n >> 4;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
        const uint4 q = __ldg(reinterpret_cast<const uint4*>(in) + i);
        const unsigned w[4] = {q.x, q.y, q.z, q.w};
        float4* o = reinterpret_cast<float4*>(out) + 4 * i;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            o[j] = make_float4(div_rn((float)(w[j] & 0xffu), 255.0f), div_rn((float)((w[j] >> 8) & 0xffu), 255.0f),
                               div_rn((float)((w[j] >> 16) & 0xffu), 255.0f), div_rn((float)(w[j] >> 24), 255.0f));
    }
    // tail (n % 16 elements) by the first threads of the grid
    const long long t = (nv << 4) + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) out[t] = div_rn((float)in[t], 255.0f);
}
}  // namespace dmh

extern "C" {
long long dmh_launch_count(void) { return dmh::g_launches.load(std::memory_order_relaxed); }
const char* dmh_last_error(void) { return dmh::g_error; }
int dmh_version(void) { return 1; }
int dmh_build_arch(void) { return 100; }
int dmh_const_div_exact(int c) {
    float rc;
    return dmh::const_div_exact(c, &rc, cudaStreamPerThread) ? 1 : 0;
}
int dmh_unpack_u8(const uint8_t* in, long long n, float* out, dmh_stream_t stream) {
    DMH_REQUIRE(in && out, "dmh_unpack_u8: null pointer");
    DMH_REQUIRE(n >= 0, "dmh_unpack_u8: negative size");
    DMH_REQUIRE(((uintptr_t)in & 15) == 0 && ((uintptr_t)out & 15) == 0, "dmh_unpack_u8: buffers must be 16-byte aligned");
    if (n == 0) return DMH_OK;
    const long long nv = n >> 4;
    long long blocks = (nv + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;          // grid-stride over 16 CTAs per SM
    if (blocks < 1) blocks = 1;
    DMH_LAUNCH(dmh::unpack_u8_kernel, (int)blocks, 256, 0, (cudaStream_t)stream)(in, n, out);
    DMH_CHECK_LAUNCH("dmh_unpack_u8");
    return DMH_OK;
}
}
