// Common device/host helpers for the B200 Pocket-TTS engine (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cmath>

#define PTTS_CUDA_CHECK(expr)                                                                          \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess) {                                                                       \
            fprintf(stderr, "ptts_b200: CUDA error %s at %s:%d: %s\n", cudaGetErrorName(_e), __FILE__, \
                    __LINE__, cudaGetErrorString(_e));                                                 \
            abort();                                                                                   \
        }                                                                                              \
    } while (0)

namespace ptts {

// Programmatic dependent launch (PDL): every kernel of the per-frame step starts with pdl_prologue(): it lets the NEXT kernel's
// CTAs be scheduled early (their prologue - barrier init, TMEM allocation, descriptor prefetch - overlaps this kernel's tail)
// and then waits until the PREVIOUS kernel has completed and flushed its memory before touching any data.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() { pdl_trigger(); pdl_wait(); }

template <typename... KArgs, typename... Args>
inline void launch_k(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t lc{};
    lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = smem; lc.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr; lc.numAttrs = pdl ? 1 : 0;
    PTTS_CUDA_CHECK(cudaLaunchKernelEx(&lc, kernel, KArgs(args)...));
}

// ---- model constants (reference src/config.h:53-87, models/defaults.h, modules/transformer.h:297-300) ----
constexpr int D_MODEL = 1024, N_HEADS = 16, D_HEAD = 64, N_LAYERS = 6, D_FF = 4096, LDIM = 32;
constexpr int D_FLOW = 512, N_RES = 6;
constexpr int M_DIM = 512, M_HEADS = 8, M_LAYERS = 2, M_FF = 2048, M_CTX = 250, M_T = 16;
constexpr int FRAME = 1920;

enum : int { DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2 };
enum : int { ACT_NONE = 0, ACT_GELU = 1, ACT_SILU = 2, ACT_ELU = 3 };
enum : int { OUT2_NONE = 0, OUT2_BF16 = 1, OUT2_F16 = 2, OUT2_F16_SPLIT = 3 };
enum : int { EPI_GENERIC = 0, EPI_FLOW_QKV = 1, EPI_MIMI_QKV = 2 };

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Activations. The epilogues evaluate ~150 M of these per frame batch, so they use the hardware exponential
// (ex2.approx via __expf, relative error ~2^-22) instead of libdevice's expm1f/tanhf (40+ instructions each): with those the
// SEANet GEMM epilogues were instruction-issue bound (ncu: 66 thread-instructions per output element, profiles/).
// Every result is rounded to f16/bf16 right after, which swamps the difference (parity unchanged, tests/test_gpu_parity.py).
//
// ggml_gelu on CPU: tanh form through an f16 table (input and output rounded to f16); reference
// modules/transformer.h:271, modules/mimi_transformer.h:959 + SURVEY.md Appendix C.
__device__ __forceinline__ float tanh_fast(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// tanh.approx (one MUFU op, relative error ~2^-11) saturates to +-1 for large |u|, which reproduces ggml's x <= -10 -> 0 and
// x >= 10 -> x special cases up to the final f16 rounding; the result is rounded to f16 and then to bf16 (the next GEMM operand).
__device__ __forceinline__ float gelu_ggml(float x) {
    const float xf = __half2float(__float2half_rn(x));
    const float u = 0.79788456080286535587989211986876f * xf * fmaf(0.044715f * xf, xf, 1.0f);
    const float hx = 0.5f * xf;
    return __half2float(__float2half_rn(fmaf(hx, tanh_fast(u), hx)));
}
__device__ __forceinline__ float silu_f(float x) { const float hx = 0.5f * x; return fmaf(hx, tanh_fast(hx), hx); }   // x * sigmoid(x)
// ELU through ex2.approx.ftz: __expf without -ftz wraps the same MUFU op in denormal scaling (2 FMUL + 2 FSETP + selects per call); for x <= 0
// both give exp(x) - 1 to ~2^-22, and a flushed denormal changes nothing once 1 is subtracted.
__device__ __forceinline__ float elu_f(float x) {
    float e; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 1.4426950408889634f));
    return x > 0.f ? x : e - 1.0f;
}
__device__ __forceinline__ float apply_act(float v, int act) {
    switch (act) {
        case ACT_GELU: return gelu_ggml(v);
        case ACT_SILU: return silu_f(v);
        case ACT_ELU: return elu_f(v);
        default: return v;
    }
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

// Row addressing shared by every batched op: GEMM row r belongs to slot-relative batch entry r / rps and
// is row r % rps inside it:   offset(r) = (r / rps) * slot_stride + (r % rps) * row_stride + base
struct RowMap {
    long long slot_stride = 0;
    long long row_stride = 0;
    long long base = 0;
    __host__ __device__ long long off(int r, int rps) const {
        return (long long)(r / rps) * slot_stride + (long long)(r % rps) * row_stride + base;
    }
};

// Fused GEMM epilogue description (see gemm.cuh).
struct Epi {
    int mode = EPI_GENERIC;
    int rps = 1 << 30;                 // rows per slot for the row maps
    const float* bias = nullptr;       // [N]
    const float* colscale = nullptr;   // [N]   (Mimi layer_scale)
    const float* rowmul = nullptr;     // [R][rowmul_ld] elementwise gate (flow head)
    int rowmul_ld = 0;
    const float* resid = nullptr; RowMap resid_map;   // v += resid
    float* out = nullptr; RowMap out_map;             // f32 output of v
    void* out2 = nullptr; RowMap out2_map;            // low-precision output of act(v)
    int out2_type = OUT2_NONE; int act = ACT_NONE;
    int split_off = 0;                 // OUT2_F16_SPLIT: lo part stored at +split_off columns
    // EPI_FLOW_QKV / EPI_MIMI_QKV
    const int* row_slot = nullptr;     // [R] absolute slot of each row
    const int* row_pos = nullptr;      // [R] absolute position of each row
    const float2* cs = nullptr;        // [R][32] (cos, sin) of pos * freq_i
    void* kcache = nullptr; void* vcache = nullptr;   // this layer's cache base
    long long kv_slot_stride = 0;      // elements between slots
    int kv_f32 = 0;                    // FlowLM cache dtype (1 = f32 like the reference, 0 = bf16)
    float* q_out_f32 = nullptr;        // FlowLM: [R][1024] f32 de-interleaved rotated q
    __nv_bfloat16* q_out_bf16 = nullptr;  // Mimi: [R][512] bf16 rotated q
    int kv_linear = 0;                 // EPI_MIMI_QKV only: k / v land in row `row` of kcache / vcache (no ring, no row_slot / row_pos)
};

}  // namespace ptts
