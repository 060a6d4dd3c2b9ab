// head_fused.cuh — the six AdaLN residual blocks + final layer of the flow/LSD head (SimpleMLPAdaLN, reference modules/mlp.h:124-170,
// 233-251; models/flow_lm.h:141) as ONE kernel of 4-CTA thread-block clusters instead of 20 dependent launches.
//
// The head works on 512-wide rows and 512x512 weights: at decode batch sizes every one of its GEMMs is a ~5 us launch for < 1 us of
// work. Here a cluster of 4 CTAs owns 16 rows for the whole chain (256 utterances = 16 clusters = 64 SMs, one wave):
//   * CTA c of the cluster computes output columns [128c, 128c+128) of every GEMM (warp w: the 16 columns 128c+16w ..), on mma.sync
//     m16n8k16 (bf16 x bf16 -> f32). Its 16 x 512 weight slice of the NEXT GEMM is prefetched into registers (2 x 16 x LDG.128 per
//     lane, k permuted inside 32-wide blocks so that one 128-bit load feeds two k-steps) while the current epilogue / hand-off runs;
//   * activations never leave the SMs. The f32 residual x lives in the accumulator-fragment registers of the CTA that owns the column
//     slice; GEMM operands (bf16) are full 16 x 512 tiles in every CTA's shared memory, written slice by slice through distributed
//     shared memory with st.async: every remote store carries its byte count to an mbarrier of the RECEIVING CTA (complete_tx), the
//     receiver arms the barrier with the tile's total (expect_tx) and waits for the phase. No fences: a cluster barrier with release
//     semantics compiles to MEMBAR.ALL.GPU, which also waits for the weight prefetch in flight (measured: 112 us for this chain);
//   * LayerNorm + AdaLN modulate is distributed by rows: CTA c normalises rows 4c .. 4c+3 (it receives their f32 column slices from the
//     four column owners), two warps per row, ggml_norm two-pass arithmetic like layernorm_kernel, and broadcasts the bf16 result.
// The hand-offs are bound by the DSMEM port (~17 B/cycle per SM in + out, producer pays): an 8-CTA / 32-row cluster moved 64 KB per
// CTA and hand-off (53 us for the chain), this shape 32 KB.
// Three data-flow hand-offs per residual block, no global-memory round trip, no grid-wide synchronisation. Write-after-read safety
// follows from the data flow alone: a tile is rewritten only by CTAs that have consumed data derived from every reader's last read.
// Rounding points are those of the unfused path (LN output and SiLU output rounded to bf16; bias, gate and residual applied in f32 with
// separately rounded add / mul); the summation order inside a dot product differs (mma k order), as between any two GEMM paths here.
#pragma once
#include "common.cuh"
#include "kernels.cuh"

namespace ptts {

constexpr int HF_CLUSTER = 4, HF_ROWS = 16, HF_THREADS = 256;
constexpr int HF_NT = D_FLOW / HF_CLUSTER / 8 / (HF_THREADS / 32);   // 8-column tiles per warp (2)
constexpr int HF_CW = D_FLOW / HF_CLUSTER;     // columns per CTA (128)
constexpr int HF_OWN = HF_ROWS / HF_CLUSTER;   // rows normalised by one CTA
constexpr int HF_AS = D_FLOW + 32;      // bf16 row stride of the operand tiles: 1088 B puts rows g and g+1 sixteen banks apart (conflict-free LDS.128)
constexpr int HF_NLN = N_RES + 1;
constexpr int HF_HST = HF_CW + 8;
constexpr size_t HF_SMEM_BYTES = 2 * (size_t)HF_ROWS * HF_AS * 2 + (size_t)HF_OWN * D_FLOW * 4 + 2 * (size_t)HF_NLN * D_FLOW * 4 + 64 + 32 + (size_t)HF_ROWS * HF_HST * 2;

struct HfParams {
    int R;                               // rows (utterances of this step)
    const float* xh;                     // [R][512] input_proj(noise) (f32)
    const float* mod; int mod_ld;        // [R][mod_ld] adaLN projections: 6 x (shift | scale | gate), then (shift | scale)
    struct { const float *lnw, *lnb; const __nv_bfloat16* w0; const float* b0; const __nv_bfloat16* w2; const float* b2; } rb[N_RES];
    const float *fnw, *fnb; const __nv_bfloat16* wf; const float* bf;   // final layer (512 -> 32)
    const float* noise;                  // [R][32] the step's noise, or x_i of LSD substep i (latent = noise + flow)
    float* latent;                       // [R][32] (may alias noise: each element is read and written by the same thread)
    const float* stepw;                  // [R][32] multi-step LSD: latent = noise + flow * stepw (lsd_time_kernel); nullptr = one step
};

__device__ __forceinline__ uint32_t hf_mapa(const void* p, int rank) {     // address of the same shared-memory location in CTA `rank` of the cluster
    uint32_t r; const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
// st.async: store into (possibly another CTA's) shared memory and decrement the tx-count of that CTA's mbarrier `bar` by the bytes stored
__device__ __forceinline__ void hf_st_u32(uint32_t a, uint32_t v, uint32_t bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(a), "r"(v), "r"(bar) : "memory");
}
__device__ __forceinline__ void hf_st_f32x2(uint32_t a, float x, float y, uint32_t bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(a), "f"(x), "f"(y), "r"(bar) : "memory");
}
__device__ __forceinline__ void hf_st_u32x4(uint32_t a, uint4 v, uint32_t bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(bar) : "memory");
}
__device__ __forceinline__ void hf_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// receiver side: arm the next phase with its byte total (one thread), wait for a phase (everybody). The wait is the plain (CTA-scope
// acquire) form: everything handed over lives in THIS CTA's shared memory, which st.async has written before it completes the tx count.
// The .acquire.cluster form compiles to TRYWAIT + CCTL.IVALL (L1 invalidate), which also waits for the weight prefetch in flight.
__device__ __forceinline__ void hf_expect(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hf_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity), "r"(0x989680u) : "memory");
    } while (!ok);
}
// loads the compiler must not sink towards their use (issued a whole hand-off ahead of the epilogue that needs them)
__device__ __forceinline__ float2 hf_ldg_pinned(const float* p) {
    float2 v; asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ int hf_cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return (int)r; }

__device__ __forceinline__ void hf_load_w(uint4 (&wreg)[16], const __nv_bfloat16* __restrict__ W, int n, int t) {
    const uint4* src = reinterpret_cast<const uint4*>(W + (long long)n * D_FLOW + 8 * t);
#pragma unroll
    for (int kb = 0; kb < 16; kb++) wreg[kb] = __ldg(src + 4 * kb);
}
// acc[j] = A[16][512] (smem tile) x wreg[j] (8 columns each), NT column tiles.
// physical k = 32 kb + 8 t + 4 s + {0,1 | 2,3}  <->  fragment k = 2 t + {0,1 | 8,9} of k-step s (the same permutation on both operands)
template <int NT>
__device__ __forceinline__ void hf_mma_tile(float (&acc)[NT][4], const __nv_bfloat16* A, const uint4 (&wreg)[NT][16], int g, int t) {
    float acc2[NT][4];
#pragma unroll
    for (int j = 0; j < NT; j++)
#pragma unroll
        for (int i = 0; i < 4; i++) { acc[j][i] = 0.f; acc2[j][i] = 0.f; }
#pragma unroll
    for (int kb = 0; kb < 16; kb++) {
        const uint4 al = *reinterpret_cast<const uint4*>(A + g * HF_AS + 32 * kb + 8 * t);
        const uint4 ah = *reinterpret_cast<const uint4*>(A + (g + 8) * HF_AS + 32 * kb + 8 * t);
        const uint32_t a0[4] = {al.x, ah.x, al.y, ah.y}, a1[4] = {al.z, ah.z, al.w, ah.w};
#pragma unroll
        for (int j = 0; j < NT; j++) {
            mma_bf16_16816(acc[j], a0, wreg[j][kb].x, wreg[j][kb].y);       // two independent accumulation chains per column tile
            mma_bf16_16816(acc2[j], a1, wreg[j][kb].z, wreg[j][kb].w);
        }
    }
#pragma unroll
    for (int j = 0; j < NT; j++)
#pragma unroll
        for (int i = 0; i < 4; i++) acc[j][i] += acc2[j][i];
}

// shift / scale of the row-half this warp normalises (prefetched one GEMM ahead of the LayerNorm that uses them)
struct HfLnMod { float4 sh0, sh1, sc0, sc1; };
__device__ __forceinline__ HfLnMod hf_load_lnmod(const float* __restrict__ mod, int mod_ld, int mod_off, int row0, int R, int rank) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = warp >> 1, c = (warp & 1) * 256 + lane * 8;
    const int grow = min(row0 + HF_OWN * rank + i, R - 1);
    const float* mp = mod + (long long)grow * mod_ld + mod_off + c;
    HfLnMod m;
    m.sh0 = __ldg(reinterpret_cast<const float4*>(mp)); m.sh1 = __ldg(reinterpret_cast<const float4*>(mp + 4));
    m.sc0 = __ldg(reinterpret_cast<const float4*>(mp + D_FLOW)); m.sc1 = __ldg(reinterpret_cast<const float4*>(mp + D_FLOW + 4));
    return m;
}
// LayerNorm (eps 1e-6, optional affine) + modulate of this CTA's HF_OWN rows (f32, complete rows in Xo) -> bf16 -> row `4 rank + i` of
// the As tile of CTAs [peer0, peer1). Two warps per row (half a row each, 8 consecutive columns per lane).
__device__ __forceinline__ void hf_layernorm_rows(const float* Xo, __nv_bfloat16* As, float* red, const float* lw, const float* lb, const HfLnMod& m,
                                                  int rank, int peer0, int peer1, const void* bar) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = warp >> 1, c = (warp & 1) * 256 + lane * 8;
    const float4 sh0 = m.sh0, sh1 = m.sh1, sc0 = m.sc0, sc1 = m.sc1;
    const float4 x0 = *reinterpret_cast<const float4*>(Xo + i * D_FLOW + c), x1 = *reinterpret_cast<const float4*>(Xo + i * D_FLOW + c + 4);
    float v[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; j++) s += v[j];
    s = warp_sum(s);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    const float mean = (red[warp & ~1] + red[warp | 1]) / D_FLOW;
    float s2 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; j++) { v[j] -= mean; s2 += v[j] * v[j]; }
    s2 = warp_sum(s2);
    if (lane == 0) red[8 + warp] = s2;
    __syncthreads();
    const float rs = 1.0f / sqrtf((red[8 + (warp & ~1)] + red[8 + (warp | 1)]) / D_FLOW + 1e-6f);
    const float sh[8] = {sh0.x, sh0.y, sh0.z, sh0.w, sh1.x, sh1.y, sh1.z, sh1.w}, sc[8] = {sc0.x, sc0.y, sc0.z, sc0.w, sc1.x, sc1.y, sc1.z, sc1.w};
    uint32_t pk[4];
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
        const float y0 = (v[j] * rs * lw[c + j] + lb[c + j]) * (sc[j] + 1.f) + sh[j];
        const float y1 = (v[j + 1] * rs * lw[c + j + 1] + lb[c + j + 1]) * (sc[j + 1] + 1.f) + sh[j + 1];
        const __nv_bfloat162 p = __floats2bfloat162_rn(y0, y1);
        pk[j >> 1] = *reinterpret_cast<const uint32_t*>(&p);
    }
    const __nv_bfloat16* dst = As + (HF_OWN * rank + i) * HF_AS + c;
    for (int peer = peer0; peer < peer1; peer++) hf_st_u32x4(hf_mapa(dst, peer), make_uint4(pk[0], pk[1], pk[2], pk[3]), hf_mapa(bar, peer));
}

__global__ void __cluster_dims__(HF_CLUSTER, 1, 1) __launch_bounds__(HF_THREADS, 1) head_res_cluster_kernel(const HfParams p) {
    pdl_prologue();
    const int rank = hf_cluster_rank();
    const int row0 = (blockIdx.x / HF_CLUSTER) * HF_ROWS;
    extern __shared__ __align__(16) unsigned char hf_smem[];
    __nv_bfloat16* As = reinterpret_cast<__nv_bfloat16*>(hf_smem);                   // [16][HF_AS] LN output (operand of mlp.0 / final)
    __nv_bfloat16* Hs = As + HF_ROWS * HF_AS;                                        // [16][HF_AS] SiLU output (operand of mlp.2)
    float* Xo = reinterpret_cast<float*>(Hs + HF_ROWS * HF_AS);                      // [4][512] f32 residual rows this CTA normalises
    float* LW = Xo + HF_OWN * D_FLOW;                                                // [7][512] LN weights, [7][512] LN biases
    float* LB = LW + HF_NLN * D_FLOW;
    float* red = LB + HF_NLN * D_FLOW;                                               // [16]
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(red + 16);      // mbarriers: A tile, H tile, own x rows
    __nv_bfloat16* Hst = reinterpret_cast<__nv_bfloat16*>(bars + 4);                 // [16][HF_HST] this CTA's SiLU slice before it is sent
    const uint32_t barA = (uint32_t)__cvta_generic_to_shared(bars), barH = barA + 8, barX = barA + 16;
    constexpr uint32_t TILE_BYTES = HF_ROWS * D_FLOW * 2, XO_BYTES = HF_OWN * D_FLOW * 4;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int wcol = warp * 8 * HF_NT;                   // this warp's first column inside the CTA's slice
    const int ncol = rank * HF_CW + wcol;                // ... and in the 512-wide row; tile j: columns ncol + 8 j .., this lane's pair at + 2 t
    // fragment rows g and g + 8 of the cluster's 16 rows (rows >= R compute on a clamped copy and are never stored)
    const int grow[2] = {min(row0 + g, p.R - 1), min(row0 + 8 + g, p.R - 1)};

    uint4 wreg[HF_NT][16];
#pragma unroll
    for (int j = 0; j < HF_NT; j++) hf_load_w(wreg[j], p.rb[0].w0, ncol + 8 * j + g, t);
    HfLnMod lm = hf_load_lnmod(p.mod, p.mod_ld, 0, row0, p.R, rank);
    float xr[HF_NT][4];                                  // residual x of this lane's fragment positions
#pragma unroll
    for (int j = 0; j < HF_NT; j++)
#pragma unroll
        for (int hf = 0; hf < 2; hf++) {
            const float2 v = __ldg(reinterpret_cast<const float2*>(p.xh + (long long)grow[hf] * D_FLOW + ncol + 8 * j + 2 * t));
            xr[j][2 * hf] = v.x; xr[j][2 * hf + 1] = v.y;
        }
#pragma unroll
    for (int j = 0; j < HF_OWN * D_FLOW / 4 / HF_THREADS; j++) {
        const int i = tid + j * HF_THREADS, r = i / (D_FLOW / 4), c = (i % (D_FLOW / 4)) * 4;
        *reinterpret_cast<float4*>(Xo + r * D_FLOW + c) = __ldg(reinterpret_cast<const float4*>(p.xh + (long long)min(row0 + HF_OWN * rank + r, p.R - 1) * D_FLOW + c));
    }
#pragma unroll 4
    for (int i = tid; i < HF_NLN * D_FLOW; i += HF_THREADS) {
        const int l = i / D_FLOW, c = i % D_FLOW;
        const float* w = l < N_RES ? p.rb[l].lnw : p.fnw;
        const float* b = l < N_RES ? p.rb[l].lnb : p.fnb;
        LW[i] = w ? __ldg(w + c) : 1.f; LB[i] = b ? __ldg(b + c) : 0.f;
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n\tmbarrier.init.shared::cta.b64 [%1], 1;\n\tmbarrier.init.shared::cta.b64 [%2], 1;" ::"r"(barA), "r"(barH), "r"(barX) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        hf_expect(barA, TILE_BYTES); hf_expect(barH, TILE_BYTES); hf_expect(barX, XO_BYTES);
    }
    __syncthreads();
    hf_cluster_sync();                                   // every CTA of the cluster runs and has armed its barriers before anybody stores into it

    for (int b = 0; b < N_RES; b++) {
        // ---- a = LN(x) (1 + scale) + shift for this CTA's rows, broadcast ----
        hf_layernorm_rows(Xo, As, red, LW + b * D_FLOW, LB + b * D_FLOW, lm, rank, 0, HF_CLUSTER, bars);
        float2 bias0[HF_NT], bias2[HF_NT], gate[HF_NT][2];
        const float* gp = p.mod + b * 3 * D_FLOW + 2 * D_FLOW;
#pragma unroll
        for (int j = 0; j < HF_NT; j++) {
            const int c = ncol + 8 * j + 2 * t;
            bias0[j] = p.rb[b].b0 ? hf_ldg_pinned(p.rb[b].b0 + c) : make_float2(0.f, 0.f);
            bias2[j] = p.rb[b].b2 ? hf_ldg_pinned(p.rb[b].b2 + c) : make_float2(0.f, 0.f);
#pragma unroll
            for (int hf = 0; hf < 2; hf++) gate[j][hf] = hf_ldg_pinned(gp + (long long)grow[hf] * p.mod_ld + c);
        }
        hf_wait(barA, b & 1);
        if (tid == 0 && (b + 1 < N_RES || rank == 0)) hf_expect(barA, TILE_BYTES);
        // ---- h = silu(mlp.0(a)) ----
        float acc[HF_NT][4];
        hf_mma_tile<HF_NT>(acc, As, wreg, g, t);
#pragma unroll
        for (int j = 0; j < HF_NT; j++) hf_load_w(wreg[j], p.rb[b].w2, ncol + 8 * j + g, t);
#pragma unroll
        for (int j = 0; j < HF_NT; j++)
#pragma unroll
            for (int hf = 0; hf < 2; hf++) {
                const __nv_bfloat162 h = __floats2bfloat162_rn(silu_f(__fadd_rn(acc[j][2 * hf], bias0[j].x)), silu_f(__fadd_rn(acc[j][2 * hf + 1], bias0[j].y)));
                *reinterpret_cast<__nv_bfloat162*>(Hst + (8 * hf + g) * HF_HST + wcol + 8 * j + 2 * t) = h;
            }
        __syncthreads();
        {   // the CTA's 16 x 128 slice goes out as 16-byte stores (4-byte DSMEM stores straight from the fragments cost ~4x the store slots)
            const int r = tid >> 4, ch = tid & 15;
            const uint4 v = *reinterpret_cast<const uint4*>(Hst + r * HF_HST + ch * 8);
            const __nv_bfloat16* dst = Hs + r * HF_AS + rank * HF_CW + ch * 8;
#pragma unroll
            for (int peer = 0; peer < HF_CLUSTER; peer++) hf_st_u32x4(hf_mapa(dst, peer), v, hf_mapa(bars + 1, peer));
        }
        hf_wait(barH, b & 1);
        if (tid == 0 && b + 1 < N_RES) hf_expect(barH, TILE_BYTES);
        lm = hf_load_lnmod(p.mod, p.mod_ld, (b + 1) * 3 * D_FLOW, row0, p.R, rank);
        // ---- x += gate * mlp.2(h); the new x goes to the CTA that normalises the row ----
        hf_mma_tile<HF_NT>(acc, Hs, wreg, g, t);
        if (b + 1 < N_RES) {
#pragma unroll
            for (int j = 0; j < HF_NT; j++) hf_load_w(wreg[j], p.rb[b + 1].w0, ncol + 8 * j + g, t);
        } else if (rank == 0 && wcol < LDIM) {
#pragma unroll
            for (int j = 0; j < HF_NT; j++) hf_load_w(wreg[j], p.wf, wcol + 8 * j + g, t);
        }
#pragma unroll
        for (int j = 0; j < HF_NT; j++)
#pragma unroll
            for (int hf = 0; hf < 2; hf++) {
                float& x0 = xr[j][2 * hf]; float& x1 = xr[j][2 * hf + 1];
                x0 = __fadd_rn(__fmul_rn(__fadd_rn(acc[j][2 * hf], bias2[j].x), gate[j][hf].x), x0);
                x1 = __fadd_rn(__fmul_rn(__fadd_rn(acc[j][2 * hf + 1], bias2[j].y), gate[j][hf].y), x1);
                const int r = 8 * hf + g;                // cluster row -> CTA r / 4 normalises it
                hf_st_f32x2(hf_mapa(Xo + (r % HF_OWN) * D_FLOW + ncol + 8 * j + 2 * t, r / HF_OWN), x0, x1, hf_mapa(bars + 2, r / HF_OWN));
            }
        hf_wait(barX, b & 1);
        if (tid == 0 && b + 1 < N_RES) hf_expect(barX, XO_BYTES);
    }
    // ---- latent = noise + linear(LN(x) (1 + scale) + shift): 32 columns, computed by CTA 0 of the cluster ----
    hf_layernorm_rows(Xo, As, red, LW + N_RES * D_FLOW, LB + N_RES * D_FLOW, lm, rank, 0, 1, bars);
    if (rank != 0) return;                               // everything addressed to this CTA has arrived (its last wait was on barX)
    hf_wait(barA, N_RES & 1);
    if (wcol >= LDIM) return;
    float acc[HF_NT][4];
    hf_mma_tile<HF_NT>(acc, As, wreg, g, t);
#pragma unroll
    for (int j = 0; j < HF_NT; j++) {
        const int c = wcol + 8 * j + 2 * t;
        const float b0 = p.bf ? p.bf[c] : 0.f, b1 = p.bf ? p.bf[c + 1] : 0.f;
#pragma unroll
        for (int hf = 0; hf < 2; hf++) {
            const int row = row0 + 8 * hf + g;
            if (row < p.R) {
                const long long o = (long long)row * LDIM + c;
                if (p.stepw) {
                    p.latent[o] = __fadd_rn(__fmul_rn(__fadd_rn(acc[j][2 * hf], b0), p.stepw[o]), p.noise[o]);
                    p.latent[o + 1] = __fadd_rn(__fmul_rn(__fadd_rn(acc[j][2 * hf + 1], b1), p.stepw[o + 1]), p.noise[o + 1]);
                } else {
                    p.latent[o] = __fadd_rn(__fadd_rn(acc[j][2 * hf], b0), p.noise[o]);
                    p.latent[o + 1] = __fadd_rn(__fadd_rn(acc[j][2 * hf + 1], b1), p.noise[o + 1]);
                }
            }
        }
    }
}

}  // namespace ptts
