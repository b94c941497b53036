// ABI bookkeeping: version, error strings, device query, the once-per-process tuning table and the
// per-kernel dynamic-shared-memory attribute cache.
#include "sp_common.cuh"
#include <atomic>
#include <mutex>
#include <vector>

extern "C" int sp_abi_version(void) { return SP_ABI_VERSION; }

extern "C" const char* sp_error_string(int code) {
    switch (code) {
        case 0: return "ok";
        case SP_ERR_BAD_ARGUMENT: return "simple_pose_b200: bad argument (null pointer, bad size or unsupported value)";
        case SP_ERR_BAD_ALIGNMENT: return "simple_pose_b200: base pointer is not 16-byte aligned";
        case SP_ERR_WORKSPACE: return "simple_pose_b200: workspace too small";
        case SP_ERR_UNSUPPORTED: return "simple_pose_b200: shape not supported by the kernels";
        default: break;
    }
    if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
    return "simple_pose_b200: unknown error code";
}

extern "C" int sp_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    SP_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    SP_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return 0;
}

// ---- tuning table ---------------------------------------------------------------------------------
namespace {

std::mutex g_mutex;
SpTuning g_tuning;
std::atomic<bool> g_tuning_loaded{false};

int env_or_unset(const char* name) {
    const char* v = getenv(name);
    if (!v || !*v) return SP_UNSET;
    return atoi(v);
}

void load_tuning_locked() {
    SpTuning t;
    t.no_pdl = env_or_unset("SP_NO_PDL");
    t.encode_warps = env_or_unset("SP_ENCODE_WARPS");
    t.encode_parts = env_or_unset("SP_ENCODE_PARTS");
    t.loss_force_ldg = env_or_unset("SP_LOSS_FORCE_LDG");
    t.loss_chunk_quads = env_or_unset("SP_LOSS_CHUNK_QUADS");
    t.loss_ring = env_or_unset("SP_LOSS_RING");
    t.loss_warps = env_or_unset("SP_LOSS_WARPS");
    t.train_force_ldg = env_or_unset("SP_TRAIN_FORCE_LDG");
    t.train_chunk_quads = env_or_unset("SP_TRAIN_CHUNK_QUADS");
    t.train_no_tile = env_or_unset("SP_TRAIN_NO_TILE");
    t.train_static_pct = env_or_unset("SP_TRAIN_STATIC_PCT");
    t.train_warps = env_or_unset("SP_TRAIN_WARPS");
    t.train_ring = env_or_unset("SP_TRAIN_RING");
    t.decode_force_generic = env_or_unset("SP_DECODE_FORCE_GENERIC");
    t.decode_warps = env_or_unset("SP_DECODE_WARPS");
    t.decode_stages = env_or_unset("SP_DECODE_STAGES");
    t.decode_grid_wide = env_or_unset("SP_DECODE_GRID_WIDE");
    t.decode_runtime_ksize = env_or_unset("SP_DECODE_RUNTIME_KSIZE");
    t.decode_static_pct = env_or_unset("SP_DECODE_STATIC_PCT");
    t.step_warps = env_or_unset("SP_STEP_WARPS");
    t.step_static_pct = env_or_unset("SP_STEP_STATIC_PCT");
    t.nms_serial = env_or_unset("SP_NMS_SERIAL");
    g_tuning = t;
    g_tuning_loaded.store(true, std::memory_order_release);
}

struct SmemMark {
    const void* func;
    int device;
    size_t bytes;
};
std::vector<SmemMark> g_smem_marks;

}  // namespace

const SpTuning& sp_tuning() {
    if (!g_tuning_loaded.load(std::memory_order_acquire)) {
        std::lock_guard<std::mutex> lock(g_mutex);
        if (!g_tuning_loaded.load(std::memory_order_relaxed)) load_tuning_locked();
    }
    return g_tuning;
}

extern "C" int sp_reload_tuning(void) {
    std::lock_guard<std::mutex> lock(g_mutex);
    load_tuning_locked();
    return 0;
}

cudaError_t sp_ensure_dyn_smem(const void* func, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(g_mutex);
    for (SmemMark& m : g_smem_marks) {
        if (m.func == func && m.device == dev) {
            if (m.bytes >= bytes) return cudaSuccess;
            e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
            if (e == cudaSuccess) m.bytes = bytes;
            return e;
        }
    }
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) g_smem_marks.push_back(SmemMark{func, dev, bytes});
    return e;
}
