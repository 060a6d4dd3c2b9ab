// gemm_tc.cuh — the tensor-core implementation of the generic GEMM family (see gemm.cuh) for sm_100a:
//   * operands staged by TMA (cp.async.bulk.tensor, SWIZZLE_128B) into a multi-stage shared-memory ring,
//   * tcgen05.mma (kind::f16, bf16 or f16 inputs, fp32 accumulate) issued by ONE thread, accumulator in TMEM,
//   * epilogue warps read TMEM with tcgen05.ld (32 lanes x 32 columns) and run the fused epilogue.
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..9 = epilogue (TMEM lane group (warp & 3) * 32, two
// warps per lane group alternate 32-column chunks). Persistent over 128 x BN output tiles, accumulator double-buffered in TMEM and
// released right after the last tcgen05.ld of a tile; up to two CTAs per SM. One kernel instantiation per (BN, epilogue class).
//
// A operand: channel-last activations [slot][rows][C]. A causal conv window (K = taps * C) is NOT materialised:
// k-block kb = (tap, c0) is loaded at row offset +tap, so a conv is the same kernel as a linear (taps == 1).
// An M tile is ONE TMA box: 128 rows of one slot when a slot has >= 128 GEMM rows (the last tile of a slot is partly
// out of bounds = zero-filled, its extra rows are discarded), or {T rows x floor(128/T) slots} when a slot has T < 128 rows.
#pragma once
#include "common.cuh"
#include "gemm.cuh"
#include <cuda.h>
#include <cstring>
#include <algorithm>
#include <map>
#include <tuple>
#include <vector>

namespace ptts {

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// try_wait with a large suspend-time hint: the warp sleeps in hardware until the phase flips instead of spinning
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity), "r"(0x989680u) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"((uint64_t)tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"((uint64_t)tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* tm, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"((uint64_t)tm), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// TMA store of a shared-memory box (written by this warp through the generic proxy, made visible with fence.proxy.async) into a 3-D tensor
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"((uint64_t)tm), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }   // staging may be rewritten
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }          // writes are complete
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
                   "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
                   "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format: version 1, layout type 2): rows are 128 B,
// 8-row groups are SBO = 1024 B apart; the k-slice inside the 128-byte atom is selected by advancing the start address.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((1024 >> 4) & 0x3FFF) << 32;   // stride byte offset
    d |= 1ull << 46;                                // descriptor version (Blackwell)
    d |= 2ull << 61;                                // SWIZZLE_128B
    return d;
}

struct TcParams {
    int R, N, K;
    int kb_per_tap;       // C / 64
    int T;                // GEMM rows per slot (plain matrix: R)
    int SB;               // slots per M tile when T < 128 (tile = SB x T rows, one TMA box {64, T, SB}); 1 otherwise
    int tps;              // M tiles per slot when T >= 128 (tile = 128 rows of one slot, box {64, 128, 1})
    int tiles_m;
    uint32_t a_bytes;     // bytes one A box delivers (including zero-filled out-of-bounds rows)
    int stages;           // shared-memory ring depth (runtime: deeper when only one CTA fits per SM anyway)
    uint32_t idesc;
    int splits;           // deterministic split-K: work item = (tile, split); partial sums go to a workspace
    int kb_per_split;
    long long ws_split_stride;   // elements between the partial-sum planes of consecutive splits
    int epi_class;               // index into EPI_CLASSES (0 = fully dynamic epilogue)
    int prefetch;                // 1 = small-M GEMM: prefetch the first work item's whole weight stream into L2 up front
    int out_rps;                 // TMA-store epilogue: GEMM rows per output slot (>= R for a plain matrix)
};

// Epilogue staging per epilogue warp: a 32 x 32 f32 accumulator chunk transposed through shared memory (rows padded to 36 floats:
// 16-byte aligned and conflict-free for 128-bit stores by row and 128-bit loads by quarter-row) + (slot, row-in-slot) of its 32 rows.
constexpr int EPI_WARPS = 8, EPI_STG_LD = 36, EPI_STG_BYTES = 32 * EPI_STG_LD * 4, EPI_ROW_BYTES = 32 * 8;
constexpr int EPI_SMEM = EPI_WARPS * (EPI_STG_BYTES + EPI_ROW_BYTES);   // 38,912 B

// ---- GENERIC epilogue, specialised at compile time ----
// The epilogue description (Epi) is a runtime structure; evaluating its flags per element made the big conv GEMMs instruction-issue bound
// (ncu r1_v8: 12.7 k warp-instructions per 128x64 tile, issue slots 57 % busy, tensor pipe 2 %). The host therefore maps the Epi to one
// of a few flag sets (epi_class) that the kernel switches on ONCE per 32-column chunk; everything inside is straight-line code.
// EF_DYNAMIC keeps the fully general runtime version for anything not in the list.
enum : unsigned { EF_BIAS = 1, EF_COLSCALE = 2, EF_ROWMUL = 4, EF_RESID = 8, EF_OUT = 16, EF_OUT2_BF16 = 32, EF_OUT2_F16 = 64, EF_SPLIT = 128,
                  EF_GELU = 256, EF_SILU = 512, EF_ELU = 1024, EF_TMA = 1u << 30, EF_DYNAMIC = 1u << 31 };
// EF_TMA marks the instantiations that use the TMA-store epilogue (epi_chunk_tma) instead of the transposing one; the host picks the
// variant per launch (TcPlanCache::tma_epilogue && many M tiles). Measured on B200: the Mimi decoder alone 0.600 -> 0.563 ms per step at
// batch 256 (every large conv / linear GEMM 5-20 % faster), but inside the two-stream pipeline the step got SLOWER (1.054 -> 1.115 ms:
// the bulk stores of a co-resident Mimi CTA compete with the FlowLM stream's bulk loads for the SM's TMA path), and the decode-sized
// GEMMs of the FlowLM chain lose ~3 % to the extra tensor-map prefetch and the store drain at CTA exit. Hence: TMA variants for the
// Mimi-only / single-stream paths, transposing epilogue inside the pipeline and for all decode-sized GEMMs.
constexpr unsigned EPI_CLASSES[] = {
    EF_DYNAMIC,                                             // 0 = not supported by the tensor-core kernel (CUDA-core fallback)
    EF_ELU | EF_OUT2_F16,                                   // 1 SEANet conv
    EF_OUT | EF_ELU | EF_OUT2_F16,                          // 2 SEANet transposed conv (f32 skip copy + f16 next input)
    EF_RESID | EF_ELU | EF_OUT2_F16,                        // 3 SEANet residual-block tail
    EF_COLSCALE | EF_RESID | EF_OUT,                        // 4 Mimi out_proj / linear2 (layer scale + residual)
    EF_GELU | EF_OUT2_BF16,                                 // 5 linear1 (+GELU)
    EF_RESID | EF_OUT,                                      // 6 FlowLM out_proj / linear2 (unsplit), flow head final linear (+noise)
    EF_OUT,                                                 // 7 split-K partial sums, adaLN projections
    EF_COLSCALE | EF_RESID | EF_OUT2_F16,                   // 8 last Mimi linear2 (writes SEANet's f16 input)
    EF_SILU | EF_OUT2_BF16,                                 // 9 flow head mlp.0
    EF_ROWMUL | EF_RESID | EF_OUT,                          // 10 flow head mlp.2 (gate + residual)
    EF_RESID | EF_SILU | EF_OUT2_BF16,                      // 11 flow head cond_embed (+ t_combined, SiLU)
    EF_OUT | EF_ELU | EF_OUT2_BF16 | EF_TMA,                // 12 unit tests (bf16 flavour of class 2, TMA-store epilogue)
    EF_ELU | EF_OUT2_F16 | EF_SPLIT,                        // 13 convt_split=1: conv feeding a transposed conv (hi | lo f16)
    EF_RESID | EF_ELU | EF_OUT2_F16 | EF_SPLIT,             // 14 convt_split=1: residual-block tail feeding a transposed conv
    EF_GELU | EF_OUT2_BF16 | EF_TMA,                        // 15 = 5 with the TMA-store epilogue
    EF_ELU | EF_OUT2_F16 | EF_TMA,                          // 16 = 1
    EF_OUT | EF_ELU | EF_OUT2_F16 | EF_TMA,                 // 17 = 2
    EF_RESID | EF_ELU | EF_OUT2_F16 | EF_TMA,               // 18 = 3
    EF_COLSCALE | EF_RESID | EF_OUT | EF_TMA,               // 19 = 4
    EF_COLSCALE | EF_RESID | EF_OUT2_F16 | EF_TMA,          // 20 = 8
};
constexpr int EPI_NCLASSES = sizeof(EPI_CLASSES) / sizeof(EPI_CLASSES[0]);

// The bias is always a runtime option (one uniform branch per chunk), everything else is part of the class key.
inline unsigned epi_flags_of(const Epi& e) {
    unsigned f = 0;
    if (e.colscale) f |= EF_COLSCALE;
    if (e.rowmul) f |= EF_ROWMUL;
    if (e.resid) f |= EF_RESID;
    if (e.out) f |= EF_OUT;
    if (e.out2_type == OUT2_BF16) f |= EF_OUT2_BF16;
    if (e.out2_type == OUT2_F16 || e.out2_type == OUT2_F16_SPLIT) f |= EF_OUT2_F16;
    if (e.out2_type == OUT2_F16_SPLIT) f |= EF_SPLIT;
    if (e.out2_type != OUT2_NONE) { if (e.act == ACT_GELU) f |= EF_GELU; else if (e.act == ACT_SILU) f |= EF_SILU; else if (e.act == ACT_ELU) f |= EF_ELU; }
    return f;
}
// want_tma: prefer the TMA-store variant when both exist, the transposing one otherwise
inline int epi_class_of(const Epi& e, bool want_tma = false) {
    const unsigned f = epi_flags_of(e);
    int any = 0;
    for (int i = 1; i < EPI_NCLASSES; i++) {
        if ((EPI_CLASSES[i] & ~EF_TMA) != f) continue;
        if (((EPI_CLASSES[i] & EF_TMA) != 0) == want_tma) return i;
        if (!any) any = i;
    }
    return any;
}

// One 32x32 accumulator chunk, already transposed into `stg` ([32][EPI_STG_LD] f32): lane (sub, cq) handles rows 4i + sub, columns
// cq..cq+3, so that the 8 lanes sharing a row cover 128 contiguous bytes (f32) and every warp-level access touches 4 full lines.
template <unsigned F>
__device__ __forceinline__ void epi_chunk(const Epi& e, const float* stg, const int2* rowinfo, int sub, int cq, int col, int rows_left, int tile_row0, long long ws_off) {
    constexpr bool DYN = (F & EF_DYNAMIC) != 0;
    const bool has_bias = e.bias != nullptr;
    const bool has_cs = DYN ? e.colscale != nullptr : (F & EF_COLSCALE) != 0;
    const bool has_rm = DYN ? e.rowmul != nullptr : (F & EF_ROWMUL) != 0;
    const bool has_res = DYN ? e.resid != nullptr : (F & EF_RESID) != 0;
    const bool has_out = DYN ? e.out != nullptr : (F & EF_OUT) != 0;
    const bool o2_bf16 = DYN ? e.out2_type == OUT2_BF16 : (F & EF_OUT2_BF16) != 0;
    const bool o2_f16 = DYN ? (e.out2_type == OUT2_F16 || e.out2_type == OUT2_F16_SPLIT) : (F & EF_OUT2_F16) != 0;
    const bool o2_split = DYN ? e.out2_type == OUT2_F16_SPLIT : (F & EF_SPLIT) != 0;
    const int act = DYN ? e.act : ((F & EF_GELU) ? ACT_GELU : (F & EF_SILU) ? ACT_SILU : (F & EF_ELU) ? ACT_ELU : ACT_NONE);
    const float4 bias4 = has_bias ? __ldg(reinterpret_cast<const float4*>(e.bias + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 cs4 = has_cs ? __ldg(reinterpret_cast<const float4*>(e.colscale + col)) : make_float4(1.f, 1.f, 1.f, 1.f);
    // strides fit 32 bits (a slot's buffer is far below 2^31 elements): one IMAD.WIDE per term instead of 64 x 64 multiplies
    const int res_ss = (int)e.resid_map.slot_stride, res_rs = (int)e.resid_map.row_stride;
    const int out_ss = (int)e.out_map.slot_stride, out_rs = (int)e.out_map.row_stride;
    const int o2_ss = (int)e.out2_map.slot_stride, o2_rs = (int)e.out2_map.row_stride;
    // the residual loads of the 8 rows are issued before any store: the compiler cannot hoist them itself (stores through out/out2
    // may alias), and serialised load->store pairs cost ~1 us each
#pragma unroll
    for (int half = 0; half < 2; half++) {                      // two passes of 4 rows: 16 registers of residual prefetch instead of 32
        float4 rs4[4], rm4[4];
        if (has_res) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int r = 16 * half + 4 * i + sub;
                rs4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r < rows_left) {
                    const int2 ri = rowinfo[r];
                    rs4[i] = *reinterpret_cast<const float4*>(e.resid + ((long long)ri.x * res_ss + (long long)ri.y * res_rs + e.resid_map.base) + col);
                }
            }
        }
        if (has_rm) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int r = 16 * half + 4 * i + sub;
                rm4[i] = make_float4(1.f, 1.f, 1.f, 1.f);
                if (r < rows_left) rm4[i] = *reinterpret_cast<const float4*>(e.rowmul + (long long)(tile_row0 + r) * e.rowmul_ld + col);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int r = 16 * half + 4 * i + sub;
            if (r < rows_left) {
                const float4 w4 = *reinterpret_cast<const float4*>(stg + r * EPI_STG_LD + cq);
                const int2 ri = rowinfo[r];
                float v[4] = {w4.x, w4.y, w4.z, w4.w};
                // explicit round-to-nearest adds / multiplies (no FMA contraction): the transposing and the TMA-store epilogue must round
                // identically, a frame must not depend on which of them ran (synchronous step vs two-stream pipeline)
                if (has_bias) { v[0] = __fadd_rn(v[0], bias4.x); v[1] = __fadd_rn(v[1], bias4.y); v[2] = __fadd_rn(v[2], bias4.z); v[3] = __fadd_rn(v[3], bias4.w); }
                if (has_cs) { v[0] = __fmul_rn(v[0], cs4.x); v[1] = __fmul_rn(v[1], cs4.y); v[2] = __fmul_rn(v[2], cs4.z); v[3] = __fmul_rn(v[3], cs4.w); }
                if (has_rm) { v[0] = __fmul_rn(v[0], rm4[i].x); v[1] = __fmul_rn(v[1], rm4[i].y); v[2] = __fmul_rn(v[2], rm4[i].z); v[3] = __fmul_rn(v[3], rm4[i].w); }
                if (has_res) { v[0] = __fadd_rn(v[0], rs4[i].x); v[1] = __fadd_rn(v[1], rs4[i].y); v[2] = __fadd_rn(v[2], rs4[i].z); v[3] = __fadd_rn(v[3], rs4[i].w); }
                if (has_out) *reinterpret_cast<float4*>(e.out + ((long long)ri.x * out_ss + (long long)ri.y * out_rs + e.out_map.base + ws_off) + col) = make_float4(v[0], v[1], v[2], v[3]);
                if (o2_bf16 || o2_f16) {
                    if (act == ACT_GELU) {
#pragma unroll
                        for (int k = 0; k < 4; k++) v[k] = gelu_ggml(v[k]);
                    } else if (act == ACT_SILU) {
#pragma unroll
                        for (int k = 0; k < 4; k++) v[k] = silu_f(v[k]);
                    } else if (act == ACT_ELU) {
#pragma unroll
                        for (int k = 0; k < 4; k++) v[k] = elu_f(v[k]);
                    }
                    const long long r2 = (long long)ri.x * o2_ss + (long long)ri.y * o2_rs + e.out2_map.base + col;
                    if (o2_bf16) {
                        __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
                        uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
                        *reinterpret_cast<uint2*>((__nv_bfloat16*)e.out2 + r2) = pk;
                    } else {
                        const __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
                        uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&h0); pk.y = *reinterpret_cast<const uint32_t*>(&h1);
                        *reinterpret_cast<uint2*>((__half*)e.out2 + r2) = pk;
                        if (o2_split) {
                            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
                            const __half2 l0 = __floats2half2_rn(v[0] - f0.x, v[1] - f0.y), l1 = __floats2half2_rn(v[2] - f1.x, v[3] - f1.y);
                            uint2 pl; pl.x = *reinterpret_cast<const uint32_t*>(&l0); pl.y = *reinterpret_cast<const uint32_t*>(&l1);
                            *reinterpret_cast<uint2*>((__half*)e.out2 + r2 + e.split_off) = pl;
                        }
                    }
                }
            }
        }
    }
}

// ---- TMA-STORE epilogue (every generic class without a per-element gate / hi+lo split) ----
// The transposing epilogue above costs ~0.8 warp-instructions per output element (staging round trip + per-row address arithmetic +
// 8/16-byte global stores): the SEANet conv GEMMs were instruction-issue bound in it (ncu r1_v15: issue slots 52-59 % busy, tensor pipe
// 3-18 %). Here every lane keeps ITS row of the 32 x 32 accumulator chunk (TMEM lane = row): bias / scale / residual / activation in
// registers, the finished row goes to a swizzled shared-memory box (f32: 128-byte rows, SWIZZLE_128B; 16-bit: 64-byte rows, SWIZZLE_64B;
// both conflict-free for st.shared.v4 by row) and one elected lane hands the whole box to the TMA engine. Rows / slots outside the tensor
// are clipped by the tensor map, so ragged tails need no predicates. The residual is read with plain loads (one 128-byte line per lane).
template <unsigned F>
__device__ __forceinline__ void epi_chunk_tma(const Epi& e, float (&v)[32], uint8_t* stg, int lane, int col0, const CUtensorMap* tmO, const CUtensorMap* tmO2,
                                              int c_row, int c_slot, bool store, const float* resid_row) {
    constexpr bool has_cs = (F & EF_COLSCALE) != 0, has_res = (F & EF_RESID) != 0, has_out = (F & EF_OUT) != 0;
    constexpr bool o2_bf16 = (F & EF_OUT2_BF16) != 0, o2_f16 = (F & EF_OUT2_F16) != 0;
    constexpr int act = (F & EF_GELU) ? ACT_GELU : (F & EF_SILU) ? ACT_SILU : (F & EF_ELU) ? ACT_ELU : ACT_NONE;
    if (e.bias) {
#pragma unroll
        for (int j = 0; j < 8; j++) { const float4 b = __ldg(reinterpret_cast<const float4*>(e.bias + col0) + j); v[4 * j] = __fadd_rn(v[4 * j], b.x); v[4 * j + 1] = __fadd_rn(v[4 * j + 1], b.y); v[4 * j + 2] = __fadd_rn(v[4 * j + 2], b.z); v[4 * j + 3] = __fadd_rn(v[4 * j + 3], b.w); }
    }
    if (has_cs) {
#pragma unroll
        for (int j = 0; j < 8; j++) { const float4 b = __ldg(reinterpret_cast<const float4*>(e.colscale + col0) + j); v[4 * j] = __fmul_rn(v[4 * j], b.x); v[4 * j + 1] = __fmul_rn(v[4 * j + 1], b.y); v[4 * j + 2] = __fmul_rn(v[4 * j + 2], b.z); v[4 * j + 3] = __fmul_rn(v[4 * j + 3], b.w); }
    }
    if (has_res && resid_row) {
#pragma unroll
        for (int j = 0; j < 8; j++) { const float4 b = *(reinterpret_cast<const float4*>(resid_row + col0) + j); v[4 * j] = __fadd_rn(v[4 * j], b.x); v[4 * j + 1] = __fadd_rn(v[4 * j + 1], b.y); v[4 * j + 2] = __fadd_rn(v[4 * j + 2], b.z); v[4 * j + 3] = __fadd_rn(v[4 * j + 3], b.w); }
    }
    const uint32_t s32 = smem_u32(stg);
    if (has_out) {
        if (lane == 0) tma_store_wait_read();                   // the previous box has been read out of the staging buffer
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; j++) *reinterpret_cast<float4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && store) { tma_store_3d(tmO, s32, col0, c_row, c_slot); tma_store_commit(); }
    }
    if (o2_bf16 || o2_f16) {
        uint32_t pk[16];
#pragma unroll
        for (int k = 0; k < 16; k++) {
            float a = v[2 * k], b = v[2 * k + 1];
            if (act == ACT_GELU) { a = gelu_ggml(a); b = gelu_ggml(b); } else if (act == ACT_SILU) { a = silu_f(a); b = silu_f(b); } else if (act == ACT_ELU) { a = elu_f(a); b = elu_f(b); }
            if (o2_bf16) { const __nv_bfloat162 h = __floats2bfloat162_rn(a, b); pk[k] = *reinterpret_cast<const uint32_t*>(&h); }
            else { const __half2 h = __floats2half2_rn(a, b); pk[k] = *reinterpret_cast<const uint32_t*>(&h); }
        }
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; j++) *reinterpret_cast<uint4*>(stg + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && store) { tma_store_3d(tmO2, s32, col0, c_row, c_slot); tma_store_commit(); }
    }
}

// ---- QKV epilogue for 32 consecutive columns (= half a head): RoPE with vector loads/stores (see epi_apply for the math) ----
template <bool mimi>
__device__ __forceinline__ void epi_qkv32(const Epi& e, int row, int col0, float (&v)[32]) {
    const int D = mimi ? M_DIM : D_MODEL;
    if (e.bias) {
#pragma unroll
        for (int i = 0; i < 32; i++) v[i] += e.bias[col0 + i];
    }
    const int part = col0 / D, c = col0 - part * D;
    const int slot = e.kv_linear ? 0 : e.row_slot[row], pos = e.kv_linear ? row : e.row_pos[row];
    if (slot < 0) return;                                       // dead row (finished utterance): nothing is appended or handed on
    const long long cbase = (long long)slot * e.kv_slot_stride + (long long)(mimi && !e.kv_linear ? pos % M_CTX : pos) * D;
    if (part == 2) {
        if (!mimi && e.kv_f32) {
            float4* g = reinterpret_cast<float4*>((float*)e.vcache + cbase + c);
#pragma unroll
            for (int j = 0; j < 8; j++) g[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        } else {
            uint4* g = reinterpret_cast<uint4*>((__nv_bfloat16*)e.vcache + cbase + c);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                __nv_bfloat162 p[4];
#pragma unroll
                for (int i = 0; i < 4; i++) p[i] = __floats2bfloat162_rn(v[8 * j + 2 * i], v[8 * j + 2 * i + 1]);
                g[j] = *reinterpret_cast<uint4*>(p);
            }
        }
        return;
    }
    const int h = c >> 6, i0 = ((c & 63) >> 5) * 16;          // 16 rotation pairs i0..i0+15 of head h
    float re[16], im[16];
    const float4* cs4 = reinterpret_cast<const float4*>(e.cs + row * 32 + i0);
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const float4 t = cs4[j];                                // (cos, sin) of pairs 2j, 2j+1
        re[2 * j] = v[4 * j] * t.x - v[4 * j + 1] * t.y;          im[2 * j] = v[4 * j] * t.y + v[4 * j + 1] * t.x;
        re[2 * j + 1] = v[4 * j + 2] * t.z - v[4 * j + 3] * t.w;  im[2 * j + 1] = v[4 * j + 2] * t.w + v[4 * j + 3] * t.z;
    }
    const int i_re = (h << 6) + i0, i_im = i_re + 32;          // de-interleaved [re(0..31) | im(0..31)]
    const bool f32dst = !mimi && (part == 0 || e.kv_f32);
    if (f32dst) {
        float* dst = (part == 0) ? e.q_out_f32 + (long long)row * D : (float*)e.kcache + cbase;
        float4* gr = reinterpret_cast<float4*>(dst + i_re); float4* gi = reinterpret_cast<float4*>(dst + i_im);
#pragma unroll
        for (int j = 0; j < 4; j++) { gr[j] = make_float4(re[4 * j], re[4 * j + 1], re[4 * j + 2], re[4 * j + 3]); gi[j] = make_float4(im[4 * j], im[4 * j + 1], im[4 * j + 2], im[4 * j + 3]); }
    } else {
        __nv_bfloat16* dst = (part == 0) ? e.q_out_bf16 + (long long)row * D : (__nv_bfloat16*)e.kcache + cbase;
        uint4* gr = reinterpret_cast<uint4*>(dst + i_re); uint4* gi = reinterpret_cast<uint4*>(dst + i_im);
#pragma unroll
        for (int j = 0; j < 2; j++) {
            __nv_bfloat162 pr[4], pi[4];
#pragma unroll
            for (int i = 0; i < 4; i++) { pr[i] = __floats2bfloat162_rn(re[8 * j + 2 * i], re[8 * j + 2 * i + 1]); pi[i] = __floats2bfloat162_rn(im[8 * j + 2 * i], im[8 * j + 2 * i + 1]); }
            gr[j] = *reinterpret_cast<uint4*>(pr); gi[j] = *reinterpret_cast<uint4*>(pi);
        }
    }
}

template <int BN>
struct TcCfg {
    static constexpr int STAGES_2CTA = (BN >= 128) ? 2 : 3;     // two CTAs per SM (default): 2 x (ring + staging) must fit 228 KB
    static constexpr int MAX_STAGES = 8;
    static constexpr int A_BYTES = 128 * 128;
    static constexpr int W_BYTES = BN * 128;
    static constexpr int STAGE_BYTES = A_BYTES + W_BYTES;
    static constexpr int STAGES_1CTA = ((224 * 1024 - EPI_SMEM - 1280) / STAGE_BYTES) < MAX_STAGES ? ((224 * 1024 - EPI_SMEM - 1280) / STAGE_BYTES) : MAX_STAGES;
    static constexpr int smem_bytes(int stages) { return stages * STAGE_BYTES + EPI_SMEM + 1024 /*align*/ + 256 /*barriers*/; }
    static constexpr int TMEM_COLS = 2 * BN;                   // double-buffered accumulator
};

// Persistent: CTA b processes tiles b, b + gridDim.x, ... (tile = tile_m * tiles_n + tile_n). The accumulator is double
// buffered in TMEM so the epilogue of tile i overlaps the TMA/MMA of tile i+1.
// CLS > 0: generic epilogue class EPI_CLASSES[CLS]; CLS == -1: FlowLM QKV epilogue; CLS == -2: Mimi QKV epilogue. One instantiation per
// (BN, CLS) keeps each kernel's code small: with a runtime switch over all classes the kernel was 160 KB of SASS and the epilogue
// warps' top stall was instruction fetch (ncu r1_v11: stalled_no_instruction 2.2 per issue).
template <int BN, int CLS>
__global__ void __launch_bounds__(320, 2) gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                                                         const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmO2,
                                                         const TcParams p, const Epi epi) {
    using Cfg = TcCfg<BN>;
    constexpr bool GEN = CLS > 0;
    constexpr unsigned CF = EPI_CLASSES[GEN ? CLS : 0];
    constexpr bool TMAEPI = GEN && (CF & EF_TMA) != 0;   // see epi_chunk_tma
    const int STAGES = p.stages;
    pdl_trigger();                                             // the next kernel may start its prologue now
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA = base, sW = base + STAGES * Cfg::A_BYTES;
    const uint32_t stg0 = sW + STAGES * Cfg::W_BYTES;         // epilogue staging (EPI_SMEM bytes)
    const uint32_t bars = stg0 + EPI_SMEM;                     // full[S] | empty[S] | tfull[2] | tempty[2] | tmem_ptr
    const uint32_t full0 = bars, empty0 = bars + 8 * STAGES, tfull0 = bars + 16 * STAGES, tempty0 = tfull0 + 16, tptr = tempty0 + 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_kb = p.K / 64;
    const int tiles_n = p.N / BN;
    const int total_tiles = tiles_n * p.tiles_m * p.splits;                 // work items (tile, split), split fastest

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tmW) : "memory");
        if (TMAEPI) {
            asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tmO) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&tmO2) : "memory");
        }
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(tfull0 + 8 * b, 1); mbar_init(tempty0 + 8 * b, 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tptr), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tptr) : "memory");
    if (p.prefetch && warp == 0 && lane == 0 && (int)blockIdx.x < total_tiles) {
        // Decode-sized GEMMs read their weights cold from HBM (the KV stream has flushed L2) and the smem ring alone cannot cover
        // DRAM latency x bandwidth: ask L2 for this CTA's whole weight stream now. Weights do not depend on the previous kernel, so
        // under programmatic dependent launch this overlaps the predecessor's tail.
        const int work = blockIdx.x, split = work % p.splits, tile_n = (work / p.splits) % tiles_n;
        const int kb0 = split * p.kb_per_split, kb1 = min(num_kb, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; kb++) tma_prefetch_3d(&tmW, 0, tile_n * BN, kb);
    }
    pdl_wait();                                                // barriers/TMEM are set up; now wait for the producer kernel's data

    if (warp == 0) {
        if (lane == 0) {
            // ===== TMA producer: one A box + one W box per k-block =====
            uint32_t cnt = 0;
            const uint32_t bytes = p.a_bytes + (uint32_t)Cfg::W_BYTES;
            for (int work = blockIdx.x; work < total_tiles; work += gridDim.x) {
                const int split = work % p.splits, tile = work / p.splits;
                const int tile_n = tile % tiles_n, tile_m = tile / tiles_n;
                int slot, t0;
                if (p.T >= 128) { slot = tile_m / p.tps; t0 = (tile_m % p.tps) * 128; } else { slot = tile_m * p.SB; t0 = 0; }
                const int kb0 = split * p.kb_per_split, kb1 = min(num_kb, kb0 + p.kb_per_split);
                for (int kb = kb0; kb < kb1; kb++, cnt++) {
                    const int s = cnt % STAGES; const uint32_t ph = (cnt / STAGES) & 1;
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    const int tap = kb / p.kb_per_tap, c0 = (kb % p.kb_per_tap) * 64;
                    mbar_expect_tx(full0 + 8 * s, bytes);
                    tma_load_3d(sA + s * Cfg::A_BYTES, &tmA, full0 + 8 * s, c0, t0 + tap, slot);
                    tma_load_3d(sW + s * Cfg::W_BYTES, &tmW, full0 + 8 * s, 0, tile_n * BN, kb);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ===== MMA issuer =====
            uint32_t cnt = 0; int it = 0;
            for (int work = blockIdx.x; work < total_tiles; work += gridDim.x, it++) {
                const int buf = it & 1;
                mbar_wait(tempty0 + 8 * buf, ((it >> 1) & 1) ^ 1);   // epilogue has drained this accumulator buffer
                tc_fence_after();
                const uint32_t tacc = tmem_base + (uint32_t)(buf * BN);
                const int split = work % p.splits;
                const int kb0 = split * p.kb_per_split, kb1 = min(num_kb, kb0 + p.kb_per_split);
                for (int kb = kb0; kb < kb1; kb++, cnt++) {
                    const int s = cnt % STAGES; const uint32_t ph = (cnt / STAGES) & 1;
                    mbar_wait(full0 + 8 * s, ph);
                    tc_fence_after();
                    const uint64_t ad = make_smem_desc_sw128(sA + s * Cfg::A_BYTES), bd = make_smem_desc_sw128(sW + s * Cfg::W_BYTES);
#pragma unroll
                    for (int k = 0; k < 4; k++) tc_mma_f16(tacc, ad + 2 * k, bd + 2 * k, p.idesc, (kb > kb0 || k != 0) ? 1u : 0u);
                    tc_commit(empty0 + 8 * s);                   // frees the smem stage when these MMAs retire
                }
                tc_commit(tfull0 + 8 * buf);                     // accumulator complete
            }
        }
    } else {
        // ===== epilogue warps: lane group (warp & 3), 32-column chunks alternate between the two warps of a lane group =====
        const int ew = warp & 3, half = (warp - 2) >> 2;
        uint8_t* const smem_gen = smem_raw + (stg0 - smem_u32(smem_raw));
        float* const stg = reinterpret_cast<float*>(smem_gen + (warp - 2) * EPI_STG_BYTES);
        int2* const rowinfo = reinterpret_cast<int2*>(smem_gen + EPI_WARPS * EPI_STG_BYTES + (warp - 2) * EPI_ROW_BYTES);
        const int sub = lane >> 3, cq = (lane & 7) * 4;          // coalesced phase: row 4i + sub of the chunk, columns cq..cq+3
        int it = 0;
        for (int work = blockIdx.x; work < total_tiles; work += gridDim.x, it++) {
            const int split = work % p.splits, tile = work / p.splits;
            const int tile_n = tile % tiles_n, tile_m = tile / tiles_n;
            const int buf = it & 1;
            int row_base, nvalid;
            if (p.T >= 128) { const int slot = tile_m / p.tps, t0 = (tile_m % p.tps) * 128; row_base = slot * p.T + t0; nvalid = min(128, p.T - t0); }
            else { row_base = tile_m * p.SB * p.T; nvalid = min(p.SB * p.T, p.R - row_base); }
            const int ri = ew * 32 + lane;
            const int row = row_base + ri;
            const bool live = ri < nvalid;
            if constexpr (GEN && !TMAEPI) {
                rowinfo[lane] = make_int2(row / epi.rps, row % epi.rps);
                __syncwarp();
            }
            // TMA-store epilogue: this warp's 32 rows start at GEMM row g0 -> (slot, row) of the output tensor; its own row's residual line
            const int g0 = row_base + ew * 32;
            const bool w_store = ew * 32 < nvalid;
            const int c_slot = g0 / p.out_rps, c_row = g0 % p.out_rps;
            const float* resid_row = nullptr;
            if constexpr (TMAEPI && (CF & EF_RESID) != 0) {
                if (live) {
                    resid_row = epi.resid + epi.resid_map.off(row, epi.rps);
                    // the residual line(s) of this lane's row: ask L2 for them now, the accumulator is not ready yet
                    for (int c0 = half * 32; c0 < BN; c0 += 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(resid_row + tile_n * BN + c0));
                }
            }
            mbar_wait(tfull0 + 8 * buf, (it >> 1) & 1);
            tc_fence_after();
            const long long ws_off = (long long)split * p.ws_split_stride;
            if (half * 32 >= BN) {                                 // BN = 32: the second warp of a lane group has no chunk, it only releases the buffer
                tc_fence_before();
                __syncwarp();
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tempty0 + 8 * buf) : "memory");
            }
#pragma unroll 1
            for (int c0 = half * 32; c0 < BN; c0 += 64) {
                float v[32];
                tc_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(buf * BN + c0), v);
                if (c0 + 64 >= BN) {
                    // This warp's last chunk of the tile is now in registers: hand the accumulator buffer back to the MMA warp BEFORE the slow
                    // global phase of the epilogue, so tile i+2's mainloop never waits for tile i's loads and stores.
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tempty0 + 8 * buf) : "memory");
                }
                if constexpr (TMAEPI) {
                    epi_chunk_tma<CF>(epi, v, smem_gen + (warp - 2) * 4096, lane, tile_n * BN + c0, &tmO, &tmO2, c_row, c_slot + split, w_store, resid_row);   // split-K: plane `split` of the plain workspace
                } else if constexpr (GEN) {
                    float4* sp = reinterpret_cast<float4*>(stg + lane * EPI_STG_LD);
#pragma unroll
                    for (int j = 0; j < 8; j++) sp[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    __syncwarp();
                    const int col = tile_n * BN + c0 + cq, rows_left = nvalid - ew * 32, tile_row0 = row_base + ew * 32;
                    epi_chunk<CF>(epi, stg, rowinfo, sub, cq, col, rows_left, tile_row0, ws_off);
                    __syncwarp();                                  // the staging tile is overwritten by the next chunk
                } else {
                    if (live) epi_qkv32<CLS == -2>(epi, row, tile_n * BN + c0, v);
                }
            }
        }
    }
    if constexpr (TMAEPI) { if (warp >= 2 && lane == 0) tma_store_wait_all(); }   // every box this lane handed to the TMA engine has been written
    tc_fence_before();
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
}

using TcKernelFn = void (*)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const TcParams, const Epi);
template <int BN>
inline TcKernelFn tc_kernel_for(int cls) {
    switch (cls) {
        case -2: return gemm_tc_kernel<BN, -2>;
        case -1: return gemm_tc_kernel<BN, -1>;
        case 1: return gemm_tc_kernel<BN, 1>;
        case 2: return gemm_tc_kernel<BN, 2>;
        case 3: return gemm_tc_kernel<BN, 3>;
        case 4: return gemm_tc_kernel<BN, 4>;
        case 5: return gemm_tc_kernel<BN, 5>;
        case 6: return gemm_tc_kernel<BN, 6>;
        case 7: return gemm_tc_kernel<BN, 7>;
        case 8: return gemm_tc_kernel<BN, 8>;
        case 9: return gemm_tc_kernel<BN, 9>;
        case 10: return gemm_tc_kernel<BN, 10>;
        case 11: return gemm_tc_kernel<BN, 11>;
        case 12: return gemm_tc_kernel<BN, 12>;
        case 13: return gemm_tc_kernel<BN, 13>;
        case 14: return gemm_tc_kernel<BN, 14>;
        case 15: return gemm_tc_kernel<BN, 15>;
        case 16: return gemm_tc_kernel<BN, 16>;
        case 17: return gemm_tc_kernel<BN, 17>;
        case 18: return gemm_tc_kernel<BN, 18>;
        case 19: return gemm_tc_kernel<BN, 19>;
        case 20: return gemm_tc_kernel<BN, 20>;
        default: return nullptr;
    }
}
inline TcKernelFn tc_kernel(int bn, int cls) { return bn == 128 ? tc_kernel_for<128>(cls) : bn == 64 ? tc_kernel_for<64>(cls) : tc_kernel_for<32>(cls); }

// Deterministic split-K reduction: sums the partial planes in a fixed order and applies the real epilogue.
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ ws, int splits, long long plane, int R, int N, const Epi epi) {
    pdl_prologue();
    const long long idx = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (idx >= (long long)R * N) return;
    const int row = (int)(idx / N), col = (int)(idx % N);
    float4 a = *reinterpret_cast<const float4*>(ws + idx);
    for (int s = 1; s < splits; s++) {
        const float4 b = *reinterpret_cast<const float4*>(ws + (long long)s * plane + idx);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    const float v[4] = {a.x, a.y, a.z, a.w};
    epi_apply<4>(epi, row, col, v, N);
}

// Same, one warp per row of C columns, followed by the LayerNorm that consumes this GEMM's output (ggml_norm semantics, see
// layernorm_kernel): the row is already in registers, so the separate LN launch and its read of the row disappear.
struct LnFuse { const float* w = nullptr; const float* b = nullptr; float eps = 0.f; __nv_bfloat16* out = nullptr; };

template <int C>
__global__ void __launch_bounds__(C / 4) splitk_reduce_ln_kernel(const float* __restrict__ ws, int splits, long long plane, int R, const Epi epi, const LnFuse ln) {
    // One CTA per row, one float4 (4 columns) per thread: R CTAs keep enough loads in flight to stream the partial planes at HBM/L2
    // speed (one warp per row left 32 CTAs on 148 SMs and took 34 us for linear2's 16 planes).
    pdl_prologue();
    constexpr int NW = C / 128;                                 // warps per CTA
    __shared__ float red[2][NW];
    const int row = blockIdx.x, col = threadIdx.x * 4, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* p = ws + (long long)row * C + col;
    float4 a = *reinterpret_cast<const float4*>(p);
    int s = 1;
    for (; s + 3 < splits; s += 4) {                            // four independent loads in flight per thread
        const float4 b0 = *reinterpret_cast<const float4*>(p + (long long)s * plane), b1 = *reinterpret_cast<const float4*>(p + (long long)(s + 1) * plane);
        const float4 b2 = *reinterpret_cast<const float4*>(p + (long long)(s + 2) * plane), b3 = *reinterpret_cast<const float4*>(p + (long long)(s + 3) * plane);
        a.x += b0.x; a.y += b0.y; a.z += b0.z; a.w += b0.w;    // fixed order s, s+1, ...: deterministic
        a.x += b1.x; a.y += b1.y; a.z += b1.z; a.w += b1.w;
        a.x += b2.x; a.y += b2.y; a.z += b2.z; a.w += b2.w;
        a.x += b3.x; a.y += b3.y; a.z += b3.z; a.w += b3.w;
    }
    for (; s < splits; s++) { const float4 b = *reinterpret_cast<const float4*>(p + (long long)s * plane); a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
    float v[4] = {a.x, a.y, a.z, a.w};
    if (epi.bias) { const float4 b = __ldg(reinterpret_cast<const float4*>(epi.bias + col)); v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w; }
    if (epi.colscale) { const float4 b = __ldg(reinterpret_cast<const float4*>(epi.colscale + col)); v[0] *= b.x; v[1] *= b.y; v[2] *= b.z; v[3] *= b.w; }
    if (epi.resid) { const float4 b = *reinterpret_cast<const float4*>(epi.resid + epi.resid_map.off(row, epi.rps) + col); v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w; }
    if (epi.out) *reinterpret_cast<float4*>(epi.out + epi.out_map.off(row, epi.rps) + col) = make_float4(v[0], v[1], v[2], v[3]);
    float s1 = warp_sum(v[0] + v[1] + v[2] + v[3]);
    if (lane == 0) red[0][warp] = s1;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < NW; w++) tot += red[0][w];
    const float mean = tot / C;
    float s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 4; i++) { v[i] -= mean; s2 += v[i] * v[i]; }
    s2 = warp_sum(s2);
    if (lane == 0) red[1][warp] = s2;
    __syncthreads();
    tot = 0.f;
#pragma unroll
    for (int w = 0; w < NW; w++) tot += red[1][w];
    const float rs = 1.0f / sqrtf(tot / C + ln.eps);
    float y[4];
#pragma unroll
    for (int i = 0; i < 4; i++) { y[i] = v[i] * rs; if (ln.w) y[i] *= ln.w[col + i]; if (ln.b) y[i] += ln.b[col + i]; }
    __nv_bfloat162 p0 = __floats2bfloat162_rn(y[0], y[1]), p1 = __floats2bfloat162_rn(y[2], y[3]);
    uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
    *reinterpret_cast<uint2*>(ln.out + (long long)row * C + col) = pk;
}

// ------------------------------------------------------------------------------------------------
// Host side: tensor-map cache + dispatch
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                        const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct TcPlanCache {
    PFN_tmapEncodeTiled encode = nullptr;
    std::map<std::tuple<const void*, long long, long long, long long, long long, long long, int, int>, CUtensorMap> maps;   // see tc_get_map
    int num_sms = 148;
    bool pdl_light = false;     // programmatic launch for the split-K reduction kernels only (see b200_engine::pdl_light)
    bool coreside = false;      // see tc_gemm_launch; switched on by the engine while it enqueues the two-stream pipeline
    bool coreside_allowed = true;   // PTTS_B200_CORESIDE=0: never (deep rings / two Mimi CTAs per SM everywhere)
    bool pdl = false;
    bool tma_epilogue = false;  // large-M GEMMs use the TMA-store epilogue (set by the engine outside the two-stream pipeline)
    float* ws_buf[2] = {nullptr, nullptr}; size_t ws_elems = (size_t)32 << 20;   // split-K partial sums, one workspace per engine stream
    int cur_ws = 0;
};

inline TcPlanCache* tc_plan_cache_create() {
    auto* c = new TcPlanCache;
    void* fn = nullptr; cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess) c->encode = (PFN_tmapEncodeTiled)fn;
    if (const char* v = getenv("PTTS_B200_CORESIDE")) c->coreside_allowed = atoi(v) != 0;
    // every (tile width, epilogue class) instantiation: opt in to the large dynamic smem and the uniform carve-out (see engine.cu)
    for (int bn : {128, 64, 32}) {
        const int st1 = bn == 128 ? TcCfg<128>::STAGES_1CTA : bn == 64 ? TcCfg<64>::STAGES_1CTA : TcCfg<32>::STAGES_1CTA;
        for (int cls = -2; cls < EPI_NCLASSES; cls++) {
            TcKernelFn k = tc_kernel(bn, cls);
            if (!k) continue;
            PTTS_CUDA_CHECK(cudaFuncSetAttribute((const void*)k, cudaFuncAttributeMaxDynamicSharedMemorySize, st1 * (128 * 128 + bn * 128) + EPI_SMEM + 1024 + 256));
            PTTS_CUDA_CHECK(cudaFuncSetAttribute((const void*)k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        }
    }
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) c->num_sms = sms;
    return c;
}
inline void tc_plan_cache_destroy(TcPlanCache* c) { if (c) for (float* w : c->ws_buf) if (w) cudaFree(w); delete c; }

struct TcGeom { int C, taps, T, SB, tps, tiles_m, n_slots, rows_per_slot_buf, box_rows; long long slot_stride; bool ok; };

inline TcGeom tc_geometry(int R, int K, const RowMap& amap, int a_rps) {
    TcGeom g{}; g.ok = false;
    const long long C = amap.row_stride;
    if (C <= 0 || C % 64 != 0 || K % C != 0 || amap.base != 0) return g;
    g.C = (int)C; g.taps = (int)(K / C);
    if (amap.slot_stride == 0) {                       // plain matrix (one "slot")
        if (g.taps != 1) return g;
        g.T = R; g.n_slots = 1; g.rows_per_slot_buf = R; g.slot_stride = (long long)R * C;
    } else {
        if (R % a_rps != 0 || amap.slot_stride % C != 0) return g;
        g.T = a_rps; g.n_slots = R / a_rps; g.slot_stride = amap.slot_stride; g.rows_per_slot_buf = (int)(amap.slot_stride / C);
        if (g.rows_per_slot_buf < g.T + g.taps - 1) return g;
    }
    if (g.T >= 128) { g.SB = 1; g.tps = (g.T + 127) / 128; g.tiles_m = g.n_slots * g.tps; g.box_rows = 128; }
    else { g.SB = 128 / g.T; g.tps = 0; g.tiles_m = (g.n_slots + g.SB - 1) / g.SB; g.box_rows = g.T; }
    g.ok = true; return g;
}

// Tile width and split-K factor.
// Small-M GEMMs (decode: R = utterances in flight, at most a few M tiles) cannot fill 148 SMs with output tiles alone and are
// bounded by fixed latencies, so the choice is made with a small cost model (microseconds):
//   GEMM    ~ 3 + CTAs-per-SM x bytes one CTA streams / (50 KB/us per SM)        (cold TMA ingest per SM, launch + pipeline fill)
//   reduce  ~ 4 + splits x R x N x 4 B / (3 MB/us)   when split (a second kernel; it also does a fused LayerNorm for free)
//   + 4.5 when a LayerNorm was requested but cannot be fused (no split)
// Calibrated on the ncu launch lists in profiles/ and on whole-step sweeps with PTTS_B200_PLAN (the step time moves by < 1 % over
// all sensible choices: these GEMMs are bounded by per-kernel fixed costs, not by the tile shape).
struct TcPlan { int bn; int splits; };
inline TcPlan tc_plan(int tiles_m, int R, int N, int K, int num_sms, bool want_ln) {
    TcPlan best{0, 1};
    const int num_kb = K / 64;
    // tuning hook: PTTS_B200_PLAN="NxK=BNxSPLITS;..." overrides the choice for small-M GEMMs of that shape
    if (tiles_m <= 4) {
        if (const char* ov = getenv("PTTS_B200_PLAN")) {
            char key[64]; snprintf(key, sizeof key, "%dx%d=", N, K);
            if (const char* q = strstr(ov, key)) {
                int bn = 0, sp = 0;
                if (sscanf(q + strlen(key), "%dx%d", &bn, &sp) == 2 && (bn == 32 || bn == 64 || bn == 128) && N % bn == 0 && sp >= 1 && sp <= 16) return TcPlan{bn, sp};
            }
        }
    }
    if (tiles_m <= 4) {
        double best_cost = 1e30;
        for (int bn : {128, 64, 32}) {
            if (N % bn != 0) continue;
            const int tiles = tiles_m * (N / bn);
            for (int sp : {1, 2, 4, 8, 16}) {
                const int kbps = (num_kb + sp - 1) / sp;
                if (sp > 1 && (kbps < 4 || (size_t)sp * R * N > ((size_t)32 << 20))) continue;
                const int ctas = tiles * ((num_kb + kbps - 1) / kbps);
                const double per_sm = (double)((ctas + num_sms - 1) / num_sms) * kbps * (16.0 + bn / 8.0);      // KB
                double cost = 3.0 + per_sm / 50.0;
                if (sp > 1) cost += 4.0 + (double)sp * R * N * 4.0 / 3.0e6;
                else if (want_ln) cost += 4.5;
                if (cost < best_cost) { best_cost = cost; best = TcPlan{bn, sp}; }
            }
        }
        return best;
    }
    if (const char* ov = getenv("PTTS_B200_PLAN")) {           // tuning hook for large GEMMs: "NxK=BNx1"
        char key[64]; snprintf(key, sizeof key, "%dx%d=", N, K);
        if (const char* q = strstr(ov, key)) {
            int bn = 0, sp = 0;
            if (sscanf(q + strlen(key), "%dx%d", &bn, &sp) == 2 && (bn == 32 || bn == 64 || bn == 128) && N % bn == 0) return TcPlan{bn, 1};
        }
    }
    for (int bn : {128, 64, 32}) {
        if (N % bn != 0) continue;
        if (tiles_m * (N / bn) >= 120 || bn == 32) { best.bn = bn; break; }
    }
    return best;
}

inline bool tc_tma_epilogue_geometry_ok(const Epi& e, int R);

template <typename T>
inline bool tc_gemm_supported(int R, int N, int K, const RowMap& amap, int a_rps, const Epi& epi) {
    // 1-2 rows: the GEMV kernel (one pass over the weights with plain loads) wins; from 3 rows on the split-K TMA stream of the tensor-core
    // kernel is faster even though its 128-row tile is almost empty (measured per decode step: batch 4 0.75 -> 0.54 ms, batch 8 1.21 -> 0.55 ms)
    static const int min_rows = getenv("PTTS_B200_TC_MIN_ROWS") ? atoi(getenv("PTTS_B200_TC_MIN_ROWS")) : 3;
    if (R < min_rows || K % 64 != 0 || N % 32 != 0) return false;
    if (epi.mode == EPI_GENERIC && epi_class_of(epi, false) == 0) {
        static bool warned = false;
        if (!warned) { warned = true; fprintf(stderr, "ptts_b200: warning: epilogue flags 0x%x have no tensor-core class; using the CUDA-core GEMM\n", epi_flags_of(epi)); }
        return false;
    }
    if (epi.mode == EPI_GENERIC && (EPI_CLASSES[epi_class_of(epi, false)] & EF_TMA) != 0 && !tc_tma_epilogue_geometry_ok(epi, R)) return false;   // TMA-only class
    const TcGeom g = tc_geometry(R, K, amap, a_rps);
    return g.ok;
}

// kind: 0 = bf16 operand, 1 = f16 operand (both SWIZZLE_128B), 2 = f32 output box (SWIZZLE_128B), 3 = 16-bit output box (SWIZZLE_64B)
inline const CUtensorMap* tc_get_map(TcPlanCache* c, const void* ptr, int kind, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                                     const cuuint32_t* box) {
    auto key = std::make_tuple(ptr, (long long)dims[0], (long long)dims[1], (long long)(rank > 2 ? dims[2] : 1),
                               (long long)strides_bytes[0], (long long)(rank > 2 ? strides_bytes[1] : 0),
                               (int)(box[1] | (box[0] << 12) | ((rank > 2 ? box[2] : 1) << 22)), kind);
    auto it = c->maps.find(key);
    if (it != c->maps.end()) return &it->second;
    CUtensorMap m;
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType dt = kind == 0 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : kind == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    CUresult r = c->encode(&m, dt, (cuuint32_t)rank, const_cast<void*>(ptr), dims,
                           strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, kind == 3 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { fprintf(stderr, "ptts_b200: cuTensorMapEncodeTiled failed (%d) kind %d dims %llu %llu %llu\n", (int)r, kind, (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)(rank > 2 ? dims[2] : 1)); abort(); }
    return &(c->maps[key] = m);
}

// Output side of the TMA-store epilogue: GEMM row g lands in slot g / rps, row g % rps of a [slots][rps][N] tensor (plain matrix: one slot
// of R rows). A warp's 32 consecutive rows must be one box: rps a multiple of 32, or a divisor of 32 (box = rps rows x 32/rps slots).
inline bool tc_tma_epilogue_geometry_ok(const Epi& e, int R) {
    const bool plain = e.rps >= R;
    if (!plain && e.rps % 32 != 0 && 32 % e.rps != 0) return false;
    auto ok_map = [&](const RowMap& m, int es) { return (m.row_stride * es) % 16 == 0 && (m.slot_stride * es) % 16 == 0 && (m.base * es) % 16 == 0 && (plain || m.slot_stride > 0); };
    if (e.out && !ok_map(e.out_map, 4)) return false;
    if (e.out2 && !ok_map(e.out2_map, 2)) return false;
    return true;
}
inline const CUtensorMap* tc_out_map(TcPlanCache* c, const void* base_ptr, const RowMap& m, int es, int R, int N, int rps, int planes, long long plane_stride_elems) {
    const bool plain = rps >= R;
    const int rows_o = plain ? R : rps, slots_o = plain ? planes : (R + rps - 1) / rps;
    cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)rows_o, (cuuint64_t)slots_o};
    const long long s2 = plain ? (planes > 1 ? plane_stride_elems : (long long)R * m.row_stride) : m.slot_stride;
    cuuint64_t str[2] = {(cuuint64_t)m.row_stride * es, (cuuint64_t)s2 * es};
    const int box_rows = std::min(32, rows_o), box_slots = plain ? 1 : std::max(1, std::min(32 / box_rows, slots_o));   // plain: planes are split-K partials
    cuuint32_t box[3] = {32, (cuuint32_t)box_rows, (cuuint32_t)box_slots};
    return tc_get_map(c, (const char*)base_ptr + m.base * es, es == 4 ? 2 : 3, 3, dims, str, box);
}

// [N][K] row-major -> [K/64][N][64] (host side, at weight upload)
template <typename T>
inline std::vector<T> tc_kblock_major(const std::vector<T>& w, int N, int K) {
    std::vector<T> o(w.size());
    const int nkb = K / 64;
    for (int kb = 0; kb < nkb; kb++)
        for (int n = 0; n < N; n++)
            for (int j = 0; j < 64; j++) o[((size_t)kb * N + n) * 64 + j] = w[(size_t)n * K + kb * 64 + j];
    return o;
}

template <typename T>
inline int tc_gemm_launch(TcPlanCache* c, const T* A, RowMap amap, int a_rps, const T* W, int R, int N, int K, const Epi& epi, cudaStream_t stream,
                          const LnFuse* ln = nullptr, bool* ln_done = nullptr) {
    if (!c || !c->encode) { fprintf(stderr, "ptts_b200: tensor-map encoder unavailable\n"); abort(); }
    constexpr bool f16 = std::is_same<T, __half>::value;
    const TcGeom g = tc_geometry(R, K, amap, a_rps);
    const bool ln_ok = ln && ln->out && epi.mode == EPI_GENERIC && !epi.rowmul && epi.out2_type == OUT2_NONE && (N == 1024 || N == 512);
    const TcPlan plan = tc_plan(g.tiles_m, R, N, K, c->num_sms, ln_ok);
    const int bn = plan.bn;
    cuuint64_t adims[3] = {(cuuint64_t)g.C, (cuuint64_t)g.rows_per_slot_buf, (cuuint64_t)g.n_slots};
    cuuint64_t astr[2] = {(cuuint64_t)g.C * 2, (cuuint64_t)g.slot_stride * 2};
    cuuint32_t abox[3] = {64, (cuuint32_t)g.box_rows, (cuuint32_t)g.SB};
    const CUtensorMap* ta = tc_get_map(c, A, f16 ? 1 : 0, 3, adims, astr, abox);
    // weights are stored k-block-major, [K/64][N][64] (tc_kblock_major): the box of any tile width is ONE contiguous bn x 128 B run,
    // so cold weight streams from HBM are page-friendly instead of bn separate 128-byte pieces 2*K bytes apart
    cuuint64_t wdims[3] = {64, (cuuint64_t)N, (cuuint64_t)(K / 64)};
    cuuint64_t wstr[2] = {128, (cuuint64_t)N * 128};
    cuuint32_t wbox[3] = {64, (cuuint32_t)bn, 1};
    const CUtensorMap* tw = tc_get_map(c, W, f16 ? 1 : 0, 3, wdims, wstr, wbox);
    TcParams p; p.R = R; p.N = N; p.K = K; p.kb_per_tap = g.C / 64; p.T = g.T; p.SB = g.SB; p.tps = g.tps; p.tiles_m = g.tiles_m;
    p.a_bytes = (uint32_t)(128 * g.box_rows * g.SB);
    // Small-M GEMMs (FlowLM decode: R = batch) cannot fill the SMs with output tiles alone: split K deterministically.
    const int num_kb = K / 64, tiles = (N / bn) * g.tiles_m;
    int splits = plan.splits;
    p.kb_per_split = (num_kb + splits - 1) / splits; p.ws_split_stride = 0;
    p.splits = (num_kb + p.kb_per_split - 1) / p.kb_per_split;   // no empty splits
    splits = p.splits;
    Epi kepi = epi;
    if (splits > 1) {
        // one fixed workspace for the engine's lifetime (its address is baked into captured CUDA graphs)
        if (!c->ws_buf[c->cur_ws]) PTTS_CUDA_CHECK(cudaMalloc(&c->ws_buf[c->cur_ws], c->ws_elems * sizeof(float)));
        kepi = Epi{}; kepi.out = c->ws_buf[c->cur_ws]; kepi.out_map.row_stride = N; p.ws_split_stride = (long long)R * N;
    } else { p.splits = 1; p.kb_per_split = num_kb; }
    p.epi_class = kepi.mode == EPI_GENERIC ? epi_class_of(kepi, c->tma_epilogue && R > 512 && tc_tma_epilogue_geometry_ok(kepi, R)) : 0;
    p.prefetch = g.tiles_m <= 4 ? 1 : 0;
    // instruction descriptor (kind::f16): D=f32, A/B = bf16|f16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
    p.idesc = (1u << 4) | ((f16 ? 0u : 1u) << 7) | ((f16 ? 0u : 1u) << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const int total_tiles = tiles * splits;
    // Co-residency mode (two-stream pipeline): every GEMM CTA takes at most half an SM (the 2-CTA ring depth), and GEMMs of the Mimi
    // stream launch at most one CTA per SM, so a decode-sized GEMM of the FlowLM chain always finds room next to a persistent Mimi CTA
    // instead of waiting for it to drain (CTAs are never preempted, stream priority only orders dispatch).
    const bool side = c->coreside && c->cur_ws == 1;
    dim3 grid(std::min(total_tiles, (side ? 1 : 2) * c->num_sms));
    const bool one_cta = !c->coreside && total_tiles <= c->num_sms;   // at most one CTA per SM anyway: spend the whole smem on a deeper ring
    const int cls = kepi.mode == EPI_GENERIC ? p.epi_class : (kepi.mode == EPI_MIMI_QKV ? -2 : -1);
    TcKernelFn kern = tc_kernel(bn, cls);
    if (!kern) { fprintf(stderr, "ptts_b200: no tensor-core kernel for epilogue class %d\n", cls); abort(); }
    const int st1 = bn == 128 ? TcCfg<128>::STAGES_1CTA : bn == 64 ? TcCfg<64>::STAGES_1CTA : TcCfg<32>::STAGES_1CTA;
    const int st2 = bn == 128 ? TcCfg<128>::STAGES_2CTA : bn == 64 ? TcCfg<64>::STAGES_2CTA : TcCfg<32>::STAGES_2CTA;
    const int stage_bytes = 128 * 128 + bn * 128;
    p.stages = one_cta ? st1 : st2;
    const CUtensorMap *to = ta, *to2 = ta;                    // unused by the other epilogues: any valid map
    p.out_rps = 1 << 30;
    if (cls > 0 && (EPI_CLASSES[cls] & EF_TMA) != 0) {
        const bool plain = kepi.rps >= R;
        p.out_rps = plain ? (1 << 30) : kepi.rps;
        if (kepi.out) to = tc_out_map(c, kepi.out, kepi.out_map, 4, R, N, kepi.rps, splits, p.ws_split_stride);
        if (kepi.out2) to2 = tc_out_map(c, kepi.out2, kepi.out2_map, 2, R, N, kepi.rps, 1, 0);
    }
    launch_k(c->pdl, kern, grid, dim3(320), (size_t)(p.stages * stage_bytes + EPI_SMEM + 1024 + 256), stream, *ta, *tw, *to, *to2, p, kepi);
    if (ln_done) *ln_done = false;
    if (splits > 1) {
        if (ln_ok) {
            if (N == 1024) launch_k(c->pdl || c->pdl_light, splitk_reduce_ln_kernel<1024>, dim3(R), dim3(256), 0, stream, (const float*)c->ws_buf[c->cur_ws], splits, (long long)R * N, R, epi, *ln);
            else launch_k(c->pdl || c->pdl_light, splitk_reduce_ln_kernel<512>, dim3(R), dim3(128), 0, stream, (const float*)c->ws_buf[c->cur_ws], splits, (long long)R * N, R, epi, *ln);
            if (ln_done) *ln_done = true;
        } else {
            const long long quads = (long long)R * N / 4;
            launch_k(c->pdl || c->pdl_light, splitk_reduce_kernel, dim3((unsigned)((quads + 255) / 256)), dim3(256), 0, stream, (const float*)c->ws_buf[c->cur_ws], splits, (long long)R * N, R, N, epi);
        }
        return 2;
    }
    return 1;
}

}  // namespace ptts
