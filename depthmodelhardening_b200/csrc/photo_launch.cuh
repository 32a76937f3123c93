// Host-side set-up shared by the launchers of the photometric kernels (photo_fast.cu, photo_ms.cu, photo_mf.cu,
// photo_objective.cu): the TMA descriptor of the target frames, the one-time kernel attributes per device, the
// disparity-to-depth constants and the wave split of the multi-scale kernels.
#pragma once
#include <cuda.h>
#include <string.h>

#include "../../include/dmh_b200.h"
#include "dmh_common.cuh"

using namespace dmh;

namespace {

// cuTensorMapEncodeTiled through the runtime's driver entry point lookup (no link-time libcuda dependency)
typedef CUresult (*TmaEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TmaEncodeFn tma_encoder() {
    static TmaEncodeFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return reinterpret_cast<TmaEncodeFn>(f);
    }();
    return fn;
}

// TMA descriptor of B frames (B,3,H,W) fp32 at `base`, viewed as a (W, H, 3, B) tensor, box (box_w, box_h, 3, 1);
// out-of-image elements are zero-filled.  false when TMA cannot take the frames: rows must be 16-byte aligned
// (W % 4 == 0 and an aligned base) and the driver must provide the encoder.
bool encode_frames_map(CUtensorMap* map, const float* base, int B, int H, int W, int box_w, int box_h) {
    memset(map, 0, sizeof(*map));
    if (W % 4 != 0 || (uintptr_t)base % 16 != 0 || tma_encoder() == nullptr) return false;
    const cuuint64_t gdim[4] = {(cuuint64_t)W, (cuuint64_t)H, 3, (cuuint64_t)B};
    const cuuint64_t gstr[3] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4, (cuuint64_t)W * H * 12};
    const cuuint32_t box[4] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 3, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return tma_encoder()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// One-time set-up per device of one launcher's kernels: the opt-in to `smem` bytes of dynamic shared memory.  Each
// launcher keeps one instance as a function-local static.  The attribute is idempotent, so racing first calls do no
// harm.
class KernelSetup {
  public:
    // The current device's SM count, or 0 after reporting the failure through set_error as `name`.
    template <typename Kernel>
    int sms(const char* name, const Kernel* kernels, int n, size_t smem) {
        int dev = 0;
        cudaGetDevice(&dev);
        int& sms = sms_[dev & 63];
        if (sms == 0) {
            cudaError_t e = cudaSuccess;
            for (int i = 0; i < n && e == cudaSuccess; ++i)
                e = cudaFuncSetAttribute(kernels[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            int count = 0;
            if (e == cudaSuccess) e = cudaDeviceGetAttribute(&count, cudaDevAttrMultiProcessorCount, dev);
            if (e != cudaSuccess) {
                set_error("%s: cudaFuncSetAttribute failed: %s", name, cudaGetErrorString(e));
                return 0;
            }
            sms = count;
        }
        return sms;
    }

  private:
    int sms_[64] = {};           // per device (ordinal & 63); 0 until configured
};

// disp_to_depth constants; a depth input (is_depth) is used as it is
DepthScale depth_scale(float min_depth, float max_depth, bool is_depth) {
    DepthScale ds;
    ds.min_disp = is_depth ? 0.f : (float)(1.0 / (double)max_depth);
    ds.range = is_depth ? 0.f : (float)(1.0 / (double)min_depth - 1.0 / (double)max_depth);
    return ds;
}

// Work split of the multi-scale kernels over n_tiles tiles and `slots` resident CTAs: tiles [0, n_full) walk all S
// scales.  The tiles of a partial last wave become S single-scale items each whenever that takes fewer "scale times"
// than one more wave of all-scale CTAs (a walk over S scales lasts S times longer): ceil(tail * S / slots) < S.
int split_last_wave(int n_tiles, int S, int slots) {
    if (S > 1 && slots > 0 && n_tiles > slots) {
        const int tail = n_tiles % slots;
        if (tail > 0 && (tail * S + slots - 1) / slots < S) return n_tiles - tail;
    }
    return n_tiles;
}

}  // namespace
