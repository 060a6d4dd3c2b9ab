// Non-GEMM kernels of the per-frame path: row preparation (RoPE tables), LayerNorm(+AdaLN modulate),
// FlowLM decode/prefill attention, Mimi ring attention, flow-head glue, Mimi front end, state upkeep.
#pragma once
#include "common.cuh"

namespace ptts {

// ------------------------------------------------------------------------------------------------
// Row preparation
// ------------------------------------------------------------------------------------------------
// (cos, sin)(pos * freq_i) per row. freq tables are computed on the host exactly like the reference's
// two RoPE flavours (rope.h:36-38 for FlowLM, ggml_timestep_embedding for Mimi rope.h:8-20).
__global__ void rope_table_kernel(const int* __restrict__ row_pos, const float* __restrict__ freq, float2* __restrict__ cs, int R) {
    pdl_prologue();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * 32) return;
    const float rad = (float)row_pos[idx >> 5] * freq[idx & 31];
    cs[idx] = make_float2(cosf(rad), sinf(rad));
}

// Decode step, Mimi side: 16 rows per slot (positions mimi_off .. mimi_off+15) and their RoPE table.
__global__ void prepare_mimi_kernel(int slot0, int n, const int* __restrict__ mimi_off, const float* __restrict__ freq,
                                    int* __restrict__ mrow_slot, int* __restrict__ mrow_pos, float2* __restrict__ mcs) {
    pdl_prologue();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * M_T * 32) return;
    const int r = idx >> 5, i = idx & 31, s = slot0 + r / M_T, pos = mimi_off[s] + r % M_T;
    if (i == 0) { mrow_slot[r] = s; mrow_pos[r] = pos; }
    const float rad = (float)pos * freq[i];
    mcs[idx] = make_float2(cosf(rad), sinf(rad));
}

// Text prefill: x[r] = float(embed[token[r]])   (ggml_get_rows, reference conditioners/text.h:29-37)
__global__ void embed_gather_kernel(const __nv_bfloat16* __restrict__ table, const int* __restrict__ tokens, float* __restrict__ x, int R) {
    pdl_prologue();
    const int r = blockIdx.x;
    if (r >= R) return;
    const __nv_bfloat16* src = table + (long long)tokens[r] * D_MODEL;
    for (int i = threadIdx.x; i < D_MODEL; i += blockDim.x) x[(long long)r * D_MODEL + i] = __bfloat162float(src[i]);
}

// ------------------------------------------------------------------------------------------------
// LayerNorm (ggml_norm: mean, biased variance of deviations, 1/sqrtf(var+eps); reference src/torch.h:49-60,
// modules/mlp.h:52-64) with optional affine and optional AdaLN modulate y*(1+scale)+shift (mlp.h:3-9).
// Writes a low-precision copy (the A operand of the following GEMM) and/or f32.
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(C / 4) layernorm_kernel(const float* __restrict__ x, RowMap xmap, int rps, int R, float eps,
                                                          const float* __restrict__ w, const float* __restrict__ b,
                                                          const float* __restrict__ shift, const float* __restrict__ scale, int mod_ld,
                                                          __nv_bfloat16* __restrict__ out_bf16, float* __restrict__ out_f32) {
    // One CTA (C/4 threads) per row, one float4 per thread: at decode batch sizes (R = 256) a warp-per-row layout leaves most SMs idle.
    pdl_prologue();
    constexpr int NW = C / 128;
    __shared__ float red[2][NW];
    const int row = blockIdx.x, col = threadIdx.x * 4, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (row >= R) return;
    const float4 a = *reinterpret_cast<const float4*>(x + xmap.off(row, rps) + col);
    float v[4] = {a.x, a.y, a.z, a.w};
    const float s1 = warp_sum(v[0] + v[1] + v[2] + v[3]);
    if (lane == 0) red[0][warp] = s1;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < NW; i++) tot += red[0][i];
    const float mean = tot / C;
    float s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 4; i++) { v[i] -= mean; s2 += v[i] * v[i]; }
    s2 = warp_sum(s2);
    if (lane == 0) red[1][warp] = s2;
    __syncthreads();
    tot = 0.f;
#pragma unroll
    for (int i = 0; i < NW; i++) tot += red[1][i];
    const float rs = 1.0f / sqrtf(tot / C + eps);
    float y[4];
#pragma unroll
    for (int i = 0; i < 4; i++) { y[i] = v[i] * rs; if (w) y[i] *= w[col + i]; if (b) y[i] += b[col + i]; }
    if (scale) {
        const float4 sc = *reinterpret_cast<const float4*>(scale + (long long)row * mod_ld + col), sh = *reinterpret_cast<const float4*>(shift + (long long)row * mod_ld + col);
        y[0] = y[0] * (sc.x + 1.f) + sh.x; y[1] = y[1] * (sc.y + 1.f) + sh.y; y[2] = y[2] * (sc.z + 1.f) + sh.z; y[3] = y[3] * (sc.w + 1.f) + sh.w;
    }
    if (out_bf16) {
        __nv_bfloat162 p0 = __floats2bfloat162_rn(y[0], y[1]), p1 = __floats2bfloat162_rn(y[2], y[3]);
        uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
        *reinterpret_cast<uint2*>(out_bf16 + (long long)row * C + col) = pk;
    }
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + (long long)row * C + col) = make_float4(y[0], y[1], y[2], y[3]);
}

// Many-row variant (Mimi: 16 rows per utterance, 4096 rows at batch 256): one WARP per row, eight rows per CTA, the row in registers
// (C / 32 values per lane), shuffles only. Same arithmetic (two-pass ggml_norm); contiguous [R][C] f32 in, bf16 out. The one-CTA-per-row
// kernel above needs 4096 CTAs of 128 threads and two block barriers for 2 KB of data per row (8 us per launch).
template <int C>
__global__ void __launch_bounds__(256) layernorm_rows_kernel(const float* __restrict__ x, int R, float eps, const float* __restrict__ w, const float* __restrict__ b,
                                                             __nv_bfloat16* __restrict__ out_bf16) {
    pdl_prologue();
    constexpr int NV = C / 128;                                  // float4 per lane
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= R) return;
    const float* xr = x + (long long)row * C;
    float4 v[NV]; float s = 0.f;
#pragma unroll
    for (int j = 0; j < NV; j++) { v[j] = *reinterpret_cast<const float4*>(xr + 128 * j + lane * 4); s += v[j].x + v[j].y + v[j].z + v[j].w; }
    const float mean = warp_sum(s) / C;
    float s2 = 0.f;
#pragma unroll
    for (int j = 0; j < NV; j++) { v[j].x -= mean; v[j].y -= mean; v[j].z -= mean; v[j].w -= mean; s2 += v[j].x * v[j].x + v[j].y * v[j].y + v[j].z * v[j].z + v[j].w * v[j].w; }
    const float rs = 1.0f / sqrtf(warp_sum(s2) / C + eps);
#pragma unroll
    for (int j = 0; j < NV; j++) {
        const int c = 128 * j + lane * 4;
        float y[4] = {v[j].x * rs, v[j].y * rs, v[j].z * rs, v[j].w * rs};
        if (w) { const float4 ww = *reinterpret_cast<const float4*>(w + c); y[0] *= ww.x; y[1] *= ww.y; y[2] *= ww.z; y[3] *= ww.w; }
        if (b) { const float4 bb = *reinterpret_cast<const float4*>(b + c); y[0] += bb.x; y[1] += bb.y; y[2] += bb.z; y[3] += bb.w; }
        const __nv_bfloat162 p0 = __floats2bfloat162_rn(y[0], y[1]), p1 = __floats2bfloat162_rn(y[2], y[3]);
        uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&p0); pk.y = *reinterpret_cast<const uint32_t*>(&p1);
        *reinterpret_cast<uint2*>(out_bf16 + (long long)row * C + c) = pk;
    }
}

// ------------------------------------------------------------------------------------------------
// FlowLM attention (reference modules/transformer.h:157-199, src/torch.h:128-150: scale 1/8, causal, softmax with f32
// probabilities, f32 PV). Two kernels share the work:
//   * attn_flow_split_kernel<KV>  — split-KV STREAMING kernel, one query row per CTA: the per-utterance part of the cache
//                                    (HBM bound; bf16 or the reference's f32 cache type);
//   * attn_tile_kernel            — tensor-core (mma.sync) flash tile: 64 query rows x one head against a key range that
//                                    MANY rows have in common (the shared voice prefix in decode) or that the rows of one
//                                    slot need under the causal mask (prefill, transformer.h:157-169).
// Both produce either the normalised bf16 output or a partial (max, sum, unnormalised acc) per (row, head) in a workspace
// [row][AF_WS_STRIDE entries]; the last streaming CTA of a row merges all partials of that row in a fixed order.
// Rows whose row_slot is negative are DEAD (finished utterances still inside the stepped slot range): nothing is read,
// appended or written for them.
// ------------------------------------------------------------------------------------------------
constexpr int AF_STAGES = 3, AF_KEYS = 8;
constexpr int AF_MAX_SPLITS = 16, AF_PFX_SPLITS = 8, AF_WS_STRIDE = AF_MAX_SPLITS + AF_PFX_SPLITS;

template <typename KV> struct AfCfg {
    static constexpr int ROW_BYTES = D_MODEL * (int)sizeof(KV);          // one cache row, all 16 heads: 2 KB (bf16) / 4 KB (f32)
    static constexpr int STAGE_BYTES = 2 * AF_KEYS * ROW_BYTES;          // 8 K rows + 8 V rows: 32 KB / 64 KB
    static constexpr int SMEM = AF_STAGES * STAGE_BYTES + 128;
    static constexpr int NCH = ROW_BYTES / 512;                          // 16-byte chunks per lane and row: 4 / 8
    static constexpr int EPC = 16 / (int)sizeof(KV);                     // elements per chunk: 8 / 4
    static constexpr int LPH = D_HEAD / EPC;                             // lanes sharing a head: 8 / 16
};

__device__ __forceinline__ uint32_t af_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void af_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity), "r"(0x989680u) : "memory");   // hardware sleep until the phase flips
    } while (!ok);
}
__device__ __forceinline__ void af_bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}

// The attention kernels keep their scores in the log2 domain (q pre-scaled by log2(e) / 8) so that every probability is ONE ex2.approx (plus the
// subtract): expf costs ~10 instructions, and at 32 of them per lane and 64-key block they outweighed the 80 MMAs of a
// tile-kernel block in issue slots. Maxima written to the merge workspace are converted back to the natural-log domain.
constexpr float AT_QSCALE = 0.125f * 1.4426950408889634f;
__device__ __forceinline__ float at_exp2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// Per-launch description of the keys a row attends to.
//   pfx_slot / pfx_len (per SLOT, may be null): keys [0, P) of the row live in ANOTHER slot's cache (the voice prefix shared by every
//   utterance of that voice, reference copy_states models/flow_lm.h:70-78 made a private copy instead); keys [P, pos] are the slot's own.
//   tiles_meta (may be null): {item count, prefix splits} of an attn_tile_kernel launch that ALREADY reduced keys [0, P) of every row with
//   P > 0 into workspace entries [AF_MAX_SPLITS, AF_MAX_SPLITS + prefix splits); this kernel then streams only [P, pos] and merges both.
//   defer_merge: the tile kernel runs CONCURRENTLY (forked stream), so its partials may not exist yet: this kernel only writes its own
//   partials and attn_merge_kernel, launched after the join, combines them (defer_merge = 1). defer_merge = 2: no merge launch either;
//   every CTA of both kernels counts into merge_cnt2[row][head] after it has published its partials, and whichever arrives LAST for a
//   (row, head) combines that head's partials (fixed entry order, same arithmetic as attn_merge_kernel: bit-identical) and writes the
//   bf16 output. Expected arrivals = streaming splits + prefix splits; dead rows are counted by nobody.
struct AfKeys { const int* pfx_slot; const int* pfx_len; const int* tiles_meta; int defer_merge; int* merge_cnt2; };

// One CTA per (KV split, query row), all 16 heads at once so that every cache row is read as one contiguous 2/4 KB line. Warp 8 lane 0
// is the producer: it streams groups of 8 consecutive K rows and V rows into a 3-stage shared-memory ring with cp.async.bulk + mbarrier
// complete_tx (bf16: two CTAs per SM = 192 KB in flight per SM; f32: one CTA of 192 KB). Consumer warp w owns key w of each stage: lane l,
// chunk i reads the 16 bytes at i*512 + l*16 of the row, so a row is NCH conflict-free LDS.128 per lane; the dot products are finished
// with shuffles inside each LPH-lane group; softmax is the online (running max / sum) form in fp32.
template <typename KV>
__global__ void __launch_bounds__(288, sizeof(KV) == 2 ? 2 : 1)
attn_flow_split_kernel(const float* __restrict__ q, const KV* __restrict__ kc, const KV* __restrict__ vc, long long kv_slot_stride,
                       const int* __restrict__ row_slot, const int* __restrict__ row_pos, const AfKeys keys, int splits,
                       float* __restrict__ ws_ml, float* __restrict__ ws_acc, __nv_bfloat16* __restrict__ out, int* __restrict__ merge_cnt) {
    using C = AfCfg<KV>;
    pdl_prologue();
    extern __shared__ __align__(128) uint8_t af_smem[];
    const int row = blockIdx.y, split = blockIdx.x;
    const int slot = row_slot[row];
    if (slot < 0) return;                                          // dead row: uniform for the whole CTA, before any barrier
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int len = row_pos[row] + 1;
    int P = 0, pslot = slot, n_extra = 0;
    if (keys.pfx_len) { P = min(keys.pfx_len[slot], len); pslot = keys.pfx_slot[slot]; }
    if (keys.tiles_meta && P > 0) n_extra = keys.tiles_meta[1];
    const int nA = n_extra > 0 ? 0 : P;                            // prefix keys streamed by this kernel
    const int ntot = nA + (len - P);                               // concatenated key space [A | B]
    int chunk = (ntot + splits - 1) / splits; chunk = (chunk + AF_KEYS - 1) / AF_KEYS * AF_KEYS;
    const int c_begin = split * chunk, c_end = min(ntot, c_begin + chunk);
    const int n_keys = max(0, c_end - c_begin);
    const int n_stages_total = (n_keys + AF_KEYS - 1) / AF_KEYS;
    const uint32_t sbase = af_smem_u32(af_smem);
    const uint32_t bars = sbase + AF_STAGES * C::STAGE_BYTES;      // full[3] | empty[3]
    if (threadIdx.x == 0) {
        for (int s = 0; s < AF_STAGES; s++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bars + 8 * s), "r"(1));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bars + 8 * (AF_STAGES + s)), "r"(8));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    if (warp == 8) {
        if (lane == 0) {
            // the per-utterance KV stream is read exactly once per step: mark it evict-first so that it does not push the Mimi stream's
            // operands (re-read by many tiles), the shared prefix and the next GEMM's prefetched weights out of L2
            uint64_t pol;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
            const char* kA = reinterpret_cast<const char*>(kc + (long long)pslot * kv_slot_stride);
            const char* vA = reinterpret_cast<const char*>(vc + (long long)pslot * kv_slot_stride);
            const char* kB = reinterpret_cast<const char*>(kc + (long long)slot * kv_slot_stride);
            const char* vB = reinterpret_cast<const char*>(vc + (long long)slot * kv_slot_stride);
            for (int it = 0; it < n_stages_total; it++) {
                const int s = it % AF_STAGES; const uint32_t ph = (it / AF_STAGES) & 1;
                af_mbar_wait(bars + 8 * (AF_STAGES + s), ph ^ 1);
                const int c0 = c_begin + it * AF_KEYS;
                const int nk = min(AF_KEYS, c_end - c0);
                const int na = max(0, min(nk, nA - c0));           // rows of this stage that come from the shared prefix
                const int nb = nk - na;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bars + 8 * s), "r"(2u * (uint32_t)nk * C::ROW_BYTES) : "memory");
                const uint32_t dk = sbase + s * C::STAGE_BYTES, dv = dk + AF_KEYS * C::ROW_BYTES;
                if (na > 0) {
                    af_bulk_load(dk, kA + (long long)c0 * C::ROW_BYTES, (uint32_t)na * C::ROW_BYTES, bars + 8 * s, pol);
                    af_bulk_load(dv, vA + (long long)c0 * C::ROW_BYTES, (uint32_t)na * C::ROW_BYTES, bars + 8 * s, pol);
                }
                if (nb > 0) {
                    const long long rb = (long long)(P + max(0, c0 - nA)) * C::ROW_BYTES;      // own rows start at position P
                    af_bulk_load(dk + na * C::ROW_BYTES, kB + rb, (uint32_t)nb * C::ROW_BYTES, bars + 8 * s, pol);
                    af_bulk_load(dv + na * C::ROW_BYTES, vB + rb, (uint32_t)nb * C::ROW_BYTES, bars + 8 * s, pol);
                }
            }
        }
        return;                                                    // the producer warp takes no part in the merge below (named barrier 1)
    }
    // ---- consumers: lane owns elements i * (512 / sizeof(KV)) + lane * EPC + e of the row, i.e. of head (that index) / 64 ----
    float qr[C::NCH][C::EPC];
#pragma unroll
    for (int i = 0; i < C::NCH; i++) {
        const float* qp = q + (long long)row * D_MODEL + i * (512 / (int)sizeof(KV)) + lane * C::EPC;
#pragma unroll
        for (int e = 0; e < C::EPC; e += 4) {
            const float4 a = *reinterpret_cast<const float4*>(qp + e);
            qr[i][e] = a.x * AT_QSCALE; qr[i][e + 1] = a.y * AT_QSCALE; qr[i][e + 2] = a.z * AT_QSCALE; qr[i][e + 3] = a.w * AT_QSCALE;   // log2 domain, see at_exp2
        }
    }
    float m[C::NCH], l[C::NCH], acc[C::NCH][C::EPC];
#pragma unroll
    for (int i = 0; i < C::NCH; i++) { m[i] = -INFINITY; l[i] = 0.f;
#pragma unroll
        for (int e = 0; e < C::EPC; e++) acc[i][e] = 0.f; }
    for (int it = 0; it < n_stages_total; it++) {
        const int s = it % AF_STAGES; const uint32_t ph = (it / AF_STAGES) & 1;
        af_mbar_wait(bars + 8 * s, ph);
        const int nk = min(AF_KEYS, n_keys - it * AF_KEYS);
        if (warp < nk) {
            const uint8_t* kr = af_smem + s * C::STAGE_BYTES + warp * C::ROW_BYTES + lane * 16;
            const uint8_t* vr = kr + AF_KEYS * C::ROW_BYTES;
            float sc[C::NCH];
#pragma unroll
            for (int i = 0; i < C::NCH; i++) {
                const uint4 kv = *reinterpret_cast<const uint4*>(kr + i * 512);
                float a = 0.f;
                if constexpr (sizeof(KV) == 2) {
                    const uint32_t w[4] = {kv.x, kv.y, kv.z, kv.w};
#pragma unroll
                    for (int t = 0; t < 4; t++) {
                        a = fmaf(__uint_as_float(w[t] << 16), qr[i][2 * t], a);
                        a = fmaf(__uint_as_float(w[t] & 0xffff0000u), qr[i][2 * t + 1], a);
                    }
                } else {
                    a = fmaf(__uint_as_float(kv.x), qr[i][0], a); a = fmaf(__uint_as_float(kv.y), qr[i][1], a);
                    a = fmaf(__uint_as_float(kv.z), qr[i][2], a); a = fmaf(__uint_as_float(kv.w), qr[i][3], a);
                }
#pragma unroll
                for (int o = C::LPH / 2; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                sc[i] = a;
            }
#pragma unroll
            for (int i = 0; i < C::NCH; i++) {
                const float mn = fmaxf(m[i], sc[i]);
                const float corr = at_exp2(m[i] - mn), p = at_exp2(sc[i] - mn);
                m[i] = mn; l[i] = l[i] * corr + p;
                const uint4 vv = *reinterpret_cast<const uint4*>(vr + i * 512);
                if constexpr (sizeof(KV) == 2) {
                    const uint32_t w[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
                    for (int t = 0; t < 4; t++) {
                        acc[i][2 * t] = fmaf(acc[i][2 * t], corr, p * __uint_as_float(w[t] << 16));
                        acc[i][2 * t + 1] = fmaf(acc[i][2 * t + 1], corr, p * __uint_as_float(w[t] & 0xffff0000u));
                    }
                } else {
                    acc[i][0] = fmaf(acc[i][0], corr, p * __uint_as_float(vv.x)); acc[i][1] = fmaf(acc[i][1], corr, p * __uint_as_float(vv.y));
                    acc[i][2] = fmaf(acc[i][2], corr, p * __uint_as_float(vv.z)); acc[i][3] = fmaf(acc[i][3], corr, p * __uint_as_float(vv.w));
                }
            }
        }
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bars + 8 * (AF_STAGES + s)) : "memory");
    }
    // ---- cross-warp merge through shared memory (ring is drained: every stage was consumed by all 8 warps) ----
    asm volatile("bar.sync 1, 256;" ::: "memory");
    float* sm_m = reinterpret_cast<float*>(af_smem);               // [8][16]
    float* sm_l = sm_m + 8 * 16;                                   // [8][16]
    float* sm_a = sm_l + 8 * 16;                                   // [8][1024]
#pragma unroll
    for (int i = 0; i < C::NCH; i++) {
        const int e0 = i * (512 / (int)sizeof(KV)) + lane * C::EPC;  // first element this lane owns in chunk i
        if ((lane % C::LPH) == 0) { sm_m[warp * 16 + (e0 >> 6)] = m[i]; sm_l[warp * 16 + (e0 >> 6)] = l[i]; }
        float* ap = sm_a + warp * D_MODEL + e0;
#pragma unroll
        for (int e = 0; e < C::EPC; e += 4) *reinterpret_cast<float4*>(ap + e) = make_float4(acc[i][e], acc[i][e + 1], acc[i][e + 2], acc[i][e + 3]);
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const int t = threadIdx.x;                                     // 0..255: dims 4t..4t+3, head t/16
    const int h = t >> 4;
    float M = -INFINITY;
#pragma unroll
    for (int w = 0; w < 8; w++) M = fmaxf(M, sm_m[w * 16 + h]);
    float L = 0.f, o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int w = 0; w < 8; w++) {
        const float mw = sm_m[w * 16 + h];
        const float sc = (mw == -INFINITY) ? 0.f : at_exp2(mw - M);
        L = fmaf(sm_l[w * 16 + h], sc, L);
        const float4 a = *reinterpret_cast<const float4*>(sm_a + w * D_MODEL + 4 * t);
        o[0] = fmaf(a.x, sc, o[0]); o[1] = fmaf(a.y, sc, o[1]); o[2] = fmaf(a.z, sc, o[2]); o[3] = fmaf(a.w, sc, o[3]);
    }
    if (splits == 1 && n_extra == 0 && !keys.defer_merge) {
        const float inv = 1.0f / L;
        __nv_bfloat162 p0 = __floats2bfloat162_rn(o[0] * inv, o[1] * inv), p1 = __floats2bfloat162_rn(o[2] * inv, o[3] * inv);
        uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
        *reinterpret_cast<uint2*>(out + (long long)row * D_MODEL + 4 * t) = pk;
        return;
    }
    const long long wrow = (long long)row * AF_WS_STRIDE;
    if ((t & 15) == 0) { ws_ml[(wrow + split) * 32 + h] = M * 0.69314718055994530942f; ws_ml[(wrow + split) * 32 + 16 + h] = L; }   // workspace maxima: natural-log domain
    *reinterpret_cast<float4*>(ws_acc + (wrow + split) * D_MODEL + 4 * t) = make_float4(o[0], o[1], o[2], o[3]);
    if (keys.defer_merge == 1) return;
    // The LAST split CTA of a row to finish merges all of the row's partials (fixed entry order: deterministic) and writes the bf16
    // output, which removes the separate merge launch from every layer. Release/acquire through the per-row counter. The prefix
    // partials (entries AF_MAX_SPLITS..) were written by an EARLIER kernel of the same stream, hence are already visible.
    // defer_merge == 2: the tile kernel runs concurrently and counts too, per (row, head); see AfKeys.
    __threadfence();
    asm volatile("bar.sync 1, 256;" ::: "memory");
    int* flag = reinterpret_cast<int*>(af_smem);                   // [16] (per head; one entry broadcast in the per-row scheme)
    if (keys.defer_merge == 2) {
        if (t < N_HEADS) {
            const int expect = splits + n_extra;
            const int prev = atomicAdd(keys.merge_cnt2 + row * N_HEADS + t, 1);
            flag[t] = (prev == expect - 1);
            if (prev == expect - 1) keys.merge_cnt2[row * N_HEADS + t] = 0;
        }
    } else if (t == 0) {
        const int prev = atomicAdd(merge_cnt + row, 1); const int last = (prev == splits - 1);
        if (last) merge_cnt[row] = 0;
        for (int i = 0; i < N_HEADS; i++) flag[i] = last;
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (!flag[h]) return;
    __threadfence();
    const int n_ent = splits + n_extra;
    float Mm = -INFINITY;
    for (int e = 0; e < n_ent; e++) { const int sp = e < splits ? e : AF_MAX_SPLITS + (e - splits); Mm = fmaxf(Mm, __ldcg(ws_ml + (wrow + sp) * 32 + h)); }
    float Lm = 0.f, om[4] = {0.f, 0.f, 0.f, 0.f};
    for (int e = 0; e < n_ent; e++) {
        const long long w2 = wrow + (e < splits ? e : AF_MAX_SPLITS + (e - splits));
        const float ms = __ldcg(ws_ml + w2 * 32 + h);
        const float sc = (ms == -INFINITY) ? 0.f : expf(ms - Mm);
        Lm = fmaf(__ldcg(ws_ml + w2 * 32 + 16 + h), sc, Lm);
        const float4 a = __ldcg(reinterpret_cast<const float4*>(ws_acc + w2 * D_MODEL + 4 * t));
        om[0] = fmaf(a.x, sc, om[0]); om[1] = fmaf(a.y, sc, om[1]); om[2] = fmaf(a.z, sc, om[2]); om[3] = fmaf(a.w, sc, om[3]);
    }
    const float inv = 1.0f / Lm;
    __nv_bfloat162 p0 = __floats2bfloat162_rn(om[0] * inv, om[1] * inv), p1 = __floats2bfloat162_rn(om[2] * inv, om[3] * inv);
    uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
    *reinterpret_cast<uint2*>(out + (long long)row * D_MODEL + 4 * t) = pk;
}

// ------------------------------------------------------------------------------------------------
// Tensor-core attention tile (bf16 cache): one CTA = 64 query rows x ONE head x a list of key blocks, flash style (online softmax,
// S = Q K^T and O += P V on mma.sync m16n8k16 bf16 -> f32; warp w owns query rows 16w .. 16w+15).
//   decode, shared voice prefix: the query rows are all utterances of one voice (row_list), the keys a split of that voice's prefix:
//     every prefix row is read once per 64 utterances (from L2) instead of once per utterance (from HBM). Output = partial.
//   prefill: the query rows are consecutive positions of one slot, keys = [shared prefix | own rows up to the row's position]
//     (causal mask key <= shift + query, transformer.h:157-169). Output = normalised bf16 rows.
// Precision: the reference computes attention in f32 on an f32 cache. K/V are bf16 here (cfg.kv_f32 = 0); q and the probabilities
// would lose another 8 bits as single bf16 MMA operands, so both are fed as hi + lo bf16 pairs (two MMAs each, ~16 mantissa bits).
// Against a float64 reference (tests/test_gpu_attention.py, values of order 1) the bf16 output of PREC 2 is within one bf16 ulp plus an
// absolute 9e-6, as close as the f32-FMA streaming kernel (1.3e-6); PREC 1 / 0 below need 2.3e-3 / 3.5e-2 beyond the ulp.
// No ldmatrix: the contraction index (QK^T) and the output-dim index (PV) are permuted so that every shared-memory access is a
// conflict-free LDS.128 (same fragment scheme as attn_mimi_mma4_kernel below):
//   * QK^T: lane (g, t) loads K[key 8j+g][32p + 8t .. +7]; its 8 values are the k-slots of two k16 steps, Q fragments use the same order;
//   * PV: output tile n holds dims {8c + n}: lane (g, t) loads V[key][8g .. 8g+7] for its four keys 16s + {2t, 2t+1, 8+2t, 9+2t};
//     PRMT interleaves key pairs. The lane ends up owning O[row][16t .. 16t+15].
// Shared memory: K and V blocks of 64 keys x 64 dims (8 KB each), double buffered with cp.async; the 16-byte chunk c of key row r is
// stored at chunk c ^ ((r & 1) << 2) for K and c ^ (((r >> 1) & 3) << 1) for V (both access patterns above hit 32 distinct banks).
// ------------------------------------------------------------------------------------------------
struct AtItem {
    int row0, nrows;               // query rows: row_list[row0 + i] (or row0 + i when row_list is null), i < nrows <= 64
    int a_slot, a_k0, a_k1;        // segment A: keys [a_k0, a_k1) of slot a_slot, visible to every row (shared prefix)
    int b_slot, b_k0, b_k1;        // segment B: keys [b_k0, b_k1) of slot b_slot, key k visible to a row iff k <= row_pos[row]
    int out_split;                 // >= 0: partial -> workspace entry out_split of each row; < 0: normalised bf16 -> out
    int pad0, pad1, pad2;
};

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void at_split2(float x, float y, uint32_t& hi, uint32_t& lo) {      // (x, y) -> bf16x2 hi, bf16x2 lo
    const __nv_bfloat162 h = __floats2bfloat162_rn(x, y);
    const float2 hf = __bfloat1622float2(h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x - hf.x, y - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h); lo = *reinterpret_cast<const uint32_t*>(&l);
}

constexpr int AT_ROWS = 64, AT_KEYS = 64, AT_TILE_BYTES = AT_KEYS * D_HEAD * 2;   // 8 KB

// PREC: 2 = q and the probabilities as hi + lo bf16 pairs, 1 = q only (P V with plain bf16 probabilities: their rounding errors are
// independent per key and average out over the keys a row attends to), 0 = plain bf16 operands.
template <int PREC>
__global__ void __launch_bounds__(128) attn_tile_kernel(const float* __restrict__ q, const __nv_bfloat16* __restrict__ kc, const __nv_bfloat16* __restrict__ vc,
                                                        long long kv_slot_stride, const AtItem* __restrict__ items, const int* __restrict__ meta,
                                                        const int* __restrict__ row_list, const int* __restrict__ row_pos,
                                                        float* __restrict__ ws_ml, float* __restrict__ ws_acc, __nv_bfloat16* __restrict__ out,
                                                        const int* __restrict__ row_slot, int* __restrict__ merge_cnt2, int stream_splits) {
    pdl_prologue();
    // log2-domain scores + ex2.approx for the decode-side tiles (PREC < 2), where the exponentials bound the kernel; the full-precision
    // variant (prefill: MMA / L2 bound, and its K/V rows feed every later frame) keeps expf on natural-log scores
    constexpr bool LOG2 = PREC < 2;
    constexpr float QS = LOG2 ? AT_QSCALE : 0.125f;
    auto EX = [](float x) { return LOG2 ? at_exp2(x) : expf(x); };
    __shared__ __align__(128) uint8_t sKV[2][2][AT_TILE_BYTES];    // [buffer][K | V]
    __shared__ int s_merge[AT_ROWS];                               // rows of this tile whose (row, head) this CTA completed (counted merge)
    if ((int)blockIdx.x >= meta[0]) return;
    const AtItem it = items[blockIdx.x];
    const int h = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const int i0 = 16 * warp + g, i1 = i0 + 8;
    const int r0 = i0 < it.nrows ? (row_list ? row_list[it.row0 + i0] : it.row0 + i0) : -1;
    const int r1 = i1 < it.nrows ? (row_list ? row_list[it.row0 + i1] : it.row0 + i1) : -1;
    const int rp0 = r0 >= 0 ? row_pos[r0] : -1, rp1 = r1 >= 0 ? row_pos[r1] : -1;
    // ---- Q fragments (scaled by 1/8, hi + lo) ----
    uint32_t qh[4][4], ql[4][4];
#pragma unroll
    for (int p = 0; p < 2; p++) {
        float x0[8], x1[8];
#pragma unroll
        for (int e = 0; e < 8; e++) { x0[e] = 0.f; x1[e] = 0.f; }
        if (r0 >= 0) {
            const float4 a = *reinterpret_cast<const float4*>(q + (long long)r0 * D_MODEL + h * D_HEAD + 32 * p + 8 * t), b = *reinterpret_cast<const float4*>(q + (long long)r0 * D_MODEL + h * D_HEAD + 32 * p + 8 * t + 4);
            x0[0] = a.x; x0[1] = a.y; x0[2] = a.z; x0[3] = a.w; x0[4] = b.x; x0[5] = b.y; x0[6] = b.z; x0[7] = b.w;
        }
        if (r1 >= 0) {
            const float4 a = *reinterpret_cast<const float4*>(q + (long long)r1 * D_MODEL + h * D_HEAD + 32 * p + 8 * t), b = *reinterpret_cast<const float4*>(q + (long long)r1 * D_MODEL + h * D_HEAD + 32 * p + 8 * t + 4);
            x1[0] = a.x; x1[1] = a.y; x1[2] = a.z; x1[3] = a.w; x1[4] = b.x; x1[5] = b.y; x1[6] = b.z; x1[7] = b.w;
        }
#pragma unroll
        for (int e = 0; e < 8; e++) { x0[e] *= QS; x1[e] *= QS; }
        // k16 step 2p: slots (2t, 2t+1) = values 0,1 and (2t+8, 2t+9) = values 2,3; step 2p+1: values 4,5 and 6,7
        at_split2(x0[0], x0[1], qh[2 * p][0], ql[2 * p][0]); at_split2(x1[0], x1[1], qh[2 * p][1], ql[2 * p][1]);
        at_split2(x0[2], x0[3], qh[2 * p][2], ql[2 * p][2]); at_split2(x1[2], x1[3], qh[2 * p][3], ql[2 * p][3]);
        at_split2(x0[4], x0[5], qh[2 * p + 1][0], ql[2 * p + 1][0]); at_split2(x1[4], x1[5], qh[2 * p + 1][1], ql[2 * p + 1][1]);
        at_split2(x0[6], x0[7], qh[2 * p + 1][2], ql[2 * p + 1][2]); at_split2(x1[6], x1[7], qh[2 * p + 1][3], ql[2 * p + 1][3]);
    }
    const int nblkA = (max(0, it.a_k1 - it.a_k0) + AT_KEYS - 1) / AT_KEYS, nblkB = (max(0, it.b_k1 - it.b_k0) + AT_KEYS - 1) / AT_KEYS;
    const int nblk = nblkA + nblkB;
    const uint32_t s_base = af_smem_u32(&sKV[0][0][0]);
    auto load_block = [&](int bi, int buf) {
        const bool segB = bi >= nblkA;
        const int k0 = segB ? it.b_k0 + (bi - nblkA) * AT_KEYS : it.a_k0 + bi * AT_KEYS;
        const int kend = segB ? it.b_k1 : it.a_k1;
        const long long sbase = (long long)(segB ? it.b_slot : it.a_slot) * kv_slot_stride + h * D_HEAD;
#pragma unroll
        for (int c = threadIdx.x; c < AT_KEYS * 8; c += 128) {
            const int key = c >> 3, ch = c & 7, kk = k0 + key;
            const uint32_t nbytes = kk < kend ? 16u : 0u;          // out-of-range rows are zero-filled
            const long long off = sbase + (long long)min(kk, kend - 1) * D_MODEL + ch * 8;
            const uint32_t dK = s_base + (uint32_t)(buf * 2) * AT_TILE_BYTES + key * 128 + ((ch ^ ((key & 1) << 2)) << 4);
            const uint32_t dV = s_base + (uint32_t)(buf * 2 + 1) * AT_TILE_BYTES + key * 128 + ((ch ^ (((key >> 1) & 3) << 1)) << 4);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dK), "l"(kc + off), "r"(nbytes) : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dV), "l"(vc + off), "r"(nbytes) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; n++) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
    if (nblk > 0) load_block(0, 0);
    for (int bi = 0; bi < nblk; bi++) {
        const int buf = bi & 1;
        if (bi + 1 < nblk) { load_block(bi + 1, buf ^ 1); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        const bool segB = bi >= nblkA;
        const int k0 = segB ? it.b_k0 + (bi - nblkA) * AT_KEYS : it.a_k0 + bi * AT_KEYS;
        const int kend = segB ? it.b_k1 : it.a_k1;
        const int lim0 = segB ? min(kend - 1, rp0) : kend - 1, lim1 = segB ? min(kend - 1, rp1) : kend - 1;   // last visible key per row
        const uint8_t* sK = &sKV[buf][0][0];
        const uint8_t* sV = &sKV[buf][1][0];
        // ---- S = Q K^T for 64 keys (8 tiles of 8) ----
        float S[8][4];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int key = 8 * j + g;
            const uint4 ka = *reinterpret_cast<const uint4*>(sK + key * 128 + ((t ^ ((key & 1) << 2)) << 4));
            const uint4 kb = *reinterpret_cast<const uint4*>(sK + key * 128 + (((4 + t) ^ ((key & 1) << 2)) << 4));
            float (&sc)[4] = S[j];
            sc[0] = sc[1] = sc[2] = sc[3] = 0.f;
            mma_bf16_16816(sc, qh[0], ka.x, ka.y); mma_bf16_16816(sc, qh[1], ka.z, ka.w);
            mma_bf16_16816(sc, qh[2], kb.x, kb.y); mma_bf16_16816(sc, qh[3], kb.z, kb.w);
            if (PREC >= 1) {
                mma_bf16_16816(sc, ql[0], ka.x, ka.y); mma_bf16_16816(sc, ql[1], ka.z, ka.w);
                mma_bf16_16816(sc, ql[2], kb.x, kb.y); mma_bf16_16816(sc, ql[3], kb.z, kb.w);
            }
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int kk = k0 + 8 * j + 2 * t + e;
                if (kk > lim0) sc[e] = -INFINITY;
                if (kk > lim1) sc[2 + e] = -INFINITY;
            }
        }
        // ---- online softmax (rows g and g+8; the four lanes of a quad share a row) ----
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int j = 0; j < 8; j++) { mx0 = fmaxf(mx0, fmaxf(S[j][0], S[j][1])); mx1 = fmaxf(mx1, fmaxf(S[j][2], S[j][3])); }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
        const float mu0 = mn0 == -INFINITY ? 0.f : mn0, mu1 = mn1 == -INFINITY ? 0.f : mn1;    // nothing visible yet: exp(-inf - 0) = 0
        const float c0 = EX(m0 - mu0), c1 = EX(m1 - mu1);
        m0 = mn0; m1 = mn1; l0 *= c0; l1 *= c1;
#pragma unroll
        for (int n = 0; n < 8; n++) { o[n][0] *= c0; o[n][1] *= c0; o[n][2] *= c1; o[n][3] *= c1; }
#pragma unroll
        for (int j = 0; j < 8; j++) {
            S[j][0] = EX(S[j][0] - mu0); S[j][1] = EX(S[j][1] - mu0); S[j][2] = EX(S[j][2] - mu1); S[j][3] = EX(S[j][3] - mu1);
            l0 += S[j][0] + S[j][1]; l1 += S[j][2] + S[j][3];
        }
        // ---- O += P V (4 key steps of 16) ----
#pragma unroll
        for (int s4 = 0; s4 < 4; s4++) {
            uint32_t ph[4], pl[4];
            at_split2(S[2 * s4][0], S[2 * s4][1], ph[0], pl[0]); at_split2(S[2 * s4][2], S[2 * s4][3], ph[1], pl[1]);
            at_split2(S[2 * s4 + 1][0], S[2 * s4 + 1][1], ph[2], pl[2]); at_split2(S[2 * s4 + 1][2], S[2 * s4 + 1][3], ph[3], pl[3]);
            const int ka = 16 * s4 + 2 * t;
            uint4 v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int key = ka + (u & 1) + 8 * (u >> 1);
                v[u] = *reinterpret_cast<const uint4*>(sV + key * 128 + ((g ^ (((key >> 1) & 3) << 1)) << 4));
            }
            const uint32_t a0[4] = {v[0].x, v[0].y, v[0].z, v[0].w}, a1[4] = {v[1].x, v[1].y, v[1].z, v[1].w};
            const uint32_t a2[4] = {v[2].x, v[2].y, v[2].z, v[2].w}, a3[4] = {v[3].x, v[3].y, v[3].z, v[3].w};
#pragma unroll
            for (int w = 0; w < 4; w++) {
                const uint32_t b0_lo = __byte_perm(a0[w], a1[w], 0x5410), b1_lo = __byte_perm(a2[w], a3[w], 0x5410);
                const uint32_t b0_hi = __byte_perm(a0[w], a1[w], 0x7632), b1_hi = __byte_perm(a2[w], a3[w], 0x7632);
                mma_bf16_16816(o[2 * w], ph, b0_lo, b1_lo);
                mma_bf16_16816(o[2 * w + 1], ph, b0_hi, b1_hi);
                if (PREC >= 2) { mma_bf16_16816(o[2 * w], pl, b0_lo, b1_lo); mma_bf16_16816(o[2 * w + 1], pl, b0_hi, b1_hi); }
            }
        }
        __syncthreads();                                           // this buffer is refilled two iterations from now
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    // o[n][e] = O[row g][16t + 8e + n], o[n][2+e] = O[row g+8][...]: the lane owns dims 16t .. 16t+15 of its two rows
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
        const int r = rr ? r1 : r0;
        if (r < 0) continue;
        const float mr = rr ? m1 : m0, lr = rr ? l1 : l0;
        if (it.out_split >= 0) {
            const long long w = (long long)r * AF_WS_STRIDE + it.out_split;
            if (t == 0) { ws_ml[w * 32 + h] = LOG2 ? mr * 0.69314718055994530942f : mr; ws_ml[w * 32 + 16 + h] = lr; }   // the merge works in the natural-log domain
            float* dst = ws_acc + w * D_MODEL + h * D_HEAD + 16 * t;
#pragma unroll
            for (int e = 0; e < 2; e++) {
                *reinterpret_cast<float4*>(dst + 8 * e) = make_float4(o[0][2 * rr + e], o[1][2 * rr + e], o[2][2 * rr + e], o[3][2 * rr + e]);
                *reinterpret_cast<float4*>(dst + 8 * e + 4) = make_float4(o[4][2 * rr + e], o[5][2 * rr + e], o[6][2 * rr + e], o[7][2 * rr + e]);
            }
        } else {
            const float inv = lr > 0.f ? 1.0f / lr : 0.f;
            __nv_bfloat162 pk[8];
#pragma unroll
            for (int e = 0; e < 2; e++)
#pragma unroll
                for (int n = 0; n < 8; n += 2) pk[e * 4 + n / 2] = __floats2bfloat162_rn(o[n][2 * rr + e] * inv, o[n + 1][2 * rr + e] * inv);
            __nv_bfloat16* dst = out + (long long)r * D_MODEL + h * D_HEAD + 16 * t;
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<uint4*>(&pk[0]);
            *reinterpret_cast<uint4*>(dst + 8) = *reinterpret_cast<uint4*>(&pk[4]);
        }
    }
    if (!merge_cnt2 || it.out_split < 0) return;
    // ---- counted merge (AfKeys::defer_merge == 2): arrive for every live row of the tile; rows this CTA completed are merged here ----
    __threadfence();
    __syncthreads();
    const int n_extra = meta[1], expect = stream_splits + n_extra;
    if ((int)threadIdx.x < AT_ROWS) {
        int mine = -1;
        if ((int)threadIdx.x < it.nrows) {
            const int r = row_list ? row_list[it.row0 + threadIdx.x] : it.row0 + (int)threadIdx.x;
            if (row_slot[r] >= 0) {                                  // dead rows are counted by nobody (their streaming CTA exits at once)
                const int prev = atomicAdd(merge_cnt2 + r * N_HEADS + h, 1);
                if (prev == expect - 1) { merge_cnt2[r * N_HEADS + h] = 0; mine = r; }
            }
        }
        s_merge[threadIdx.x] = mine;
    }
    __syncthreads();
    __threadfence();
    for (int i = threadIdx.x >> 1; i < it.nrows; i += 64) {          // two threads per row: 32 dims each
        const int r = s_merge[i];
        if (r < 0) continue;
        const long long wrow = (long long)r * AF_WS_STRIDE;
        const int d0 = h * D_HEAD + (threadIdx.x & 1) * 32;
        float Mm = -INFINITY;
        for (int e = 0; e < expect; e++) { const int sp = e < stream_splits ? e : AF_MAX_SPLITS + (e - stream_splits); Mm = fmaxf(Mm, __ldcg(ws_ml + (wrow + sp) * 32 + h)); }
        float Lm = 0.f, om[32];
#pragma unroll
        for (int j = 0; j < 32; j++) om[j] = 0.f;
        for (int e = 0; e < expect; e++) {
            const long long w2 = wrow + (e < stream_splits ? e : AF_MAX_SPLITS + (e - stream_splits));
            const float ms = __ldcg(ws_ml + w2 * 32 + h);
            const float sc = (ms == -INFINITY) ? 0.f : expf(ms - Mm);
            Lm = fmaf(__ldcg(ws_ml + w2 * 32 + 16 + h), sc, Lm);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 a = __ldcg(reinterpret_cast<const float4*>(ws_acc + w2 * D_MODEL + d0 + j));
                om[j] = fmaf(a.x, sc, om[j]); om[j + 1] = fmaf(a.y, sc, om[j + 1]); om[j + 2] = fmaf(a.z, sc, om[j + 2]); om[j + 3] = fmaf(a.w, sc, om[j + 3]);
            }
        }
        const float inv = 1.0f / Lm;
        __nv_bfloat16* dst = out + (long long)r * D_MODEL + d0;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
            __nv_bfloat162 pk[4];
#pragma unroll
            for (int u = 0; u < 4; u++) pk[u] = __floats2bfloat162_rn(om[j + 2 * u] * inv, om[j + 2 * u + 1] * inv);
            *reinterpret_cast<uint4*>(dst + j) = *reinterpret_cast<uint4*>(&pk[0]);
        }
    }
}

// Combines the partials of one row after the streaming kernel (entries [0, splits)) and the shared-prefix tile kernel (entries
// [AF_MAX_SPLITS, AF_MAX_SPLITS + prefix splits) for rows with a shared prefix) ran side by side. One CTA per row, fixed entry order.
__global__ void __launch_bounds__(256) attn_merge_kernel(const int* __restrict__ row_slot, const int* __restrict__ pfx_len, const int* __restrict__ tiles_meta, int splits,
                                                         const float* __restrict__ ws_ml, const float* __restrict__ ws_acc, __nv_bfloat16* __restrict__ out) {
    pdl_prologue();
    const int row = blockIdx.x, t = threadIdx.x, h = t >> 4;
    const int slot = row_slot[row];
    if (slot < 0) return;
    const int n_extra = pfx_len[slot] > 0 ? tiles_meta[1] : 0;
    const long long wrow = (long long)row * AF_WS_STRIDE;
    const int n_ent = splits + n_extra;
    float Mm = -INFINITY;
    for (int e = 0; e < n_ent; e++) { const int sp = e < splits ? e : AF_MAX_SPLITS + (e - splits); Mm = fmaxf(Mm, ws_ml[(wrow + sp) * 32 + h]); }
    float Lm = 0.f, om[4] = {0.f, 0.f, 0.f, 0.f};
    for (int e = 0; e < n_ent; e++) {
        const long long w2 = wrow + (e < splits ? e : AF_MAX_SPLITS + (e - splits));
        const float ms = ws_ml[w2 * 32 + h];
        const float sc = (ms == -INFINITY) ? 0.f : expf(ms - Mm);
        Lm = fmaf(ws_ml[w2 * 32 + 16 + h], sc, Lm);
        const float4 a = *reinterpret_cast<const float4*>(ws_acc + w2 * D_MODEL + 4 * t);
        om[0] = fmaf(a.x, sc, om[0]); om[1] = fmaf(a.y, sc, om[1]); om[2] = fmaf(a.z, sc, om[2]); om[3] = fmaf(a.w, sc, om[3]);
    }
    const float inv = 1.0f / Lm;
    __nv_bfloat162 p0 = __floats2bfloat162_rn(om[0] * inv, om[1] * inv), p1 = __floats2bfloat162_rn(om[2] * inv, om[3] * inv);
    uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
    *reinterpret_cast<uint2*>(out + (long long)row * D_MODEL + 4 * t) = pk;
}

// ------------------------------------------------------------------------------------------------
// Mimi ring attention: 16 queries of one slot x all 250 ring slots, additive 0/-inf bias taken from the
// reference's pattern (src/torch.h:168-221, called with the chunk's START offset, mimi_transformer.h:1198).
// mask_mode 0 = reference (non-causal quirk once offset > 250, SURVEY.md Appendix D.1), 1 = ideal causal ring.
// q (bf16), K/V ring (bf16), probabilities rounded to bf16 (ggml bf16 mul_mat), f32 accumulation.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool mimi_masked(int offset, int j, int c, int mask_mode) {
    if (mask_mode == 1) {
        const int last = offset + M_T - 1;
        const int p = last - (((last - c) % M_CTX + M_CTX) % M_CTX);   // newest position living in ring slot c
        return p < 0 || p > offset + j;
    }
    const int start = M_CTX * 2 - M_T;                                   // 484
    const int idx = (offset <= M_CTX ? start - offset : M_CTX - (offset % M_CTX)) + c;
    return idx >= start + 1 + j || (idx <= M_CTX - 1 && idx > M_CTX - 1 - (M_T - j - 1));
}

// One CTA (8 warps) per (slot, head). K and V of the head (250 x 64 bf16 each) are staged once in shared memory; warp w
// owns queries w and w+8. Scores: lane = ring slot (K rows read as 16-byte chunks, XOR-swizzled by row so that the 32 rows
// a warp touches spread over all banks), q broadcast from shared memory. Softmax per query row with warp shuffles, the
// probabilities are rounded to bf16 (ggml's bf16 mul_mat does that to the f32 operand), then PV with lane = 2 output dims.
constexpr int AM_SMEM = (2 * M_CTX * D_HEAD) * 2 + M_T * 256 * 4 + M_T * D_HEAD * 4;   // K,V bf16 + P f32 + Q f32 = 84,480 B

__global__ void __launch_bounds__(256) attn_mimi_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ kc,
                                                        const __nv_bfloat16* __restrict__ vc, long long kv_slot_stride, int slot0,
                                                        const int* __restrict__ mimi_off, int mask_mode, __nv_bfloat16* __restrict__ out) {
    pdl_prologue();
    extern __shared__ __align__(16) uint8_t am_smem[];
    uint4* sK = reinterpret_cast<uint4*>(am_smem);                               // [250][8 chunks], chunk index XOR (row & 7)
    uint4* sV = sK + M_CTX * 8;                                                  // [250][8 chunks]
    float* sP = reinterpret_cast<float*>(sV + M_CTX * 8);                        // [16][256]
    float* sQ = sP + M_T * 256;                                                  // [16][64]
    const int b = blockIdx.x, h = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int slot = slot0 + b;
    const int offset = mimi_off[slot];
    const uint4* Kg = reinterpret_cast<const uint4*>(kc + (long long)slot * kv_slot_stride + h * D_HEAD);   // row stride M_DIM*2 B = 64 uint4
    const uint4* Vg = reinterpret_cast<const uint4*>(vc + (long long)slot * kv_slot_stride + h * D_HEAD);
    for (int i = tid; i < M_CTX * 8; i += 256) {
        const int r = i >> 3, ch = i & 7;
        sK[r * 8 + (ch ^ (r & 7))] = Kg[(long long)r * (M_DIM / 8) + ch];
        sV[i] = Vg[(long long)r * (M_DIM / 8) + ch];
    }
    for (int i = tid; i < M_T * D_HEAD; i += 256) {
        const int t = i >> 6, d = i & 63;
        sQ[i] = __bfloat162float(q[((long long)b * M_T + t) * M_DIM + h * D_HEAD + d]);
    }
    __syncthreads();
    const int q0 = wid, q1 = wid + 8;
    // ---- scores (scale 1/8, additive 0/-inf bias) ----
    for (int c = lane; c < 256; c += 32) {
        float s0 = -INFINITY, s1 = -INFINITY;
        if (c < M_CTX) {
            const bool m0 = mimi_masked(offset, q0, c, mask_mode), m1 = mimi_masked(offset, q1, c, mask_mode);
            if (!(m0 && m1)) {
                float a0 = 0.f, a1 = 0.f;
#pragma unroll
                for (int ch = 0; ch < 8; ch++) {
                    const uint4 kv = sK[c * 8 + (ch ^ (c & 7))];
                    const uint32_t w[4] = {kv.x, kv.y, kv.z, kv.w};
                    const float4 qa0 = *reinterpret_cast<const float4*>(sQ + q0 * 64 + ch * 8), qb0 = *reinterpret_cast<const float4*>(sQ + q0 * 64 + ch * 8 + 4);
                    const float4 qa1 = *reinterpret_cast<const float4*>(sQ + q1 * 64 + ch * 8), qb1 = *reinterpret_cast<const float4*>(sQ + q1 * 64 + ch * 8 + 4);
                    const float k0 = __uint_as_float(w[0] << 16), k1 = __uint_as_float(w[0] & 0xffff0000u), k2 = __uint_as_float(w[1] << 16), k3 = __uint_as_float(w[1] & 0xffff0000u);
                    const float k4 = __uint_as_float(w[2] << 16), k5 = __uint_as_float(w[2] & 0xffff0000u), k6 = __uint_as_float(w[3] << 16), k7 = __uint_as_float(w[3] & 0xffff0000u);
                    a0 = fmaf(k0, qa0.x, a0); a0 = fmaf(k1, qa0.y, a0); a0 = fmaf(k2, qa0.z, a0); a0 = fmaf(k3, qa0.w, a0);
                    a0 = fmaf(k4, qb0.x, a0); a0 = fmaf(k5, qb0.y, a0); a0 = fmaf(k6, qb0.z, a0); a0 = fmaf(k7, qb0.w, a0);
                    a1 = fmaf(k0, qa1.x, a1); a1 = fmaf(k1, qa1.y, a1); a1 = fmaf(k2, qa1.z, a1); a1 = fmaf(k3, qa1.w, a1);
                    a1 = fmaf(k4, qb1.x, a1); a1 = fmaf(k5, qb1.y, a1); a1 = fmaf(k6, qb1.z, a1); a1 = fmaf(k7, qb1.w, a1);
                }
                if (!m0) s0 = a0 * 0.125f;
                if (!m1) s1 = a1 * 0.125f;
            }
        }
        sP[q0 * 256 + c] = s0; sP[q1 * 256 + c] = s1;
    }
    __syncwarp();
    // ---- softmax rows q0, q1 (this warp wrote them) ----
#pragma unroll
    for (int rsel = 0; rsel < 2; rsel++) {
        float* pr = sP + (rsel ? q1 : q0) * 256;
        float mx = -INFINITY;
        for (int c = lane; c < 256; c += 32) mx = fmaxf(mx, pr[c]);
        mx = warp_max(mx);
        float sum = 0.f;
        for (int c = lane; c < 256; c += 32) { const float e = expf(pr[c] - mx); pr[c] = e; sum += e; }
        sum = warp_sum(sum);
        const float inv = 1.0f / sum;
        for (int c = lane; c < 256; c += 32) pr[c] = __bfloat162float(__float2bfloat16_rn(pr[c] * inv));
    }
    __syncwarp();
    // ---- PV: lane owns output dims 2*lane, 2*lane+1 ----
    float o00 = 0.f, o01 = 0.f, o10 = 0.f, o11 = 0.f;
    const uint32_t* sV32 = reinterpret_cast<const uint32_t*>(sV);
    for (int c = 0; c < 248; c += 4) {
        const float4 p0 = *reinterpret_cast<const float4*>(sP + q0 * 256 + c), p1 = *reinterpret_cast<const float4*>(sP + q1 * 256 + c);
        const float pa[4] = {p0.x, p0.y, p0.z, p0.w}, pb[4] = {p1.x, p1.y, p1.z, p1.w};
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const uint32_t vv = sV32[(c + u) * 32 + lane];
            const float v0 = __uint_as_float(vv << 16), v1 = __uint_as_float(vv & 0xffff0000u);
            o00 = fmaf(pa[u], v0, o00); o01 = fmaf(pa[u], v1, o01); o10 = fmaf(pb[u], v0, o10); o11 = fmaf(pb[u], v1, o11);
        }
    }
    for (int c = 248; c < M_CTX; c++) {
        const uint32_t vv = sV32[c * 32 + lane];
        const float v0 = __uint_as_float(vv << 16), v1 = __uint_as_float(vv & 0xffff0000u);
        const float pa = sP[q0 * 256 + c], pb = sP[q1 * 256 + c];
        o00 = fmaf(pa, v0, o00); o01 = fmaf(pa, v1, o01); o10 = fmaf(pb, v0, o10); o11 = fmaf(pb, v1, o11);
    }
    *reinterpret_cast<__nv_bfloat162*>(out + ((long long)b * M_T + q0) * M_DIM + h * D_HEAD + 2 * lane) = __floats2bfloat162_rn(o00, o01);
    *reinterpret_cast<__nv_bfloat162*>(out + ((long long)b * M_T + q1) * M_DIM + h * D_HEAD + 2 * lane) = __floats2bfloat162_rn(o10, o11);
}

// ------------------------------------------------------------------------------------------------
// Mimi ring attention on the warp-level tensor cores (mma.sync m16n8k16, bf16 x bf16 -> f32): the 16 queries of one (slot, head) are
// exactly one M = 16 tile: S = Q K^T as key tiles of 8, softmax, O = P V as key steps of 16 x 8 output tiles. No ldmatrix: every global
// access is a 16-byte vector load/store because the contraction index (and the output-dim index) may be permuted freely:
//   * QK^T: lane (g, t) loads K[key 8j+g][32p + 8t .. +7]; its 8 values are used as the k-slots of two k16 steps, and the
//     Q fragments are loaded with the same permutation;
//   * PV: output tile n holds dims {8c + n}, so lane (g, t) needs V[key][8g .. 8g+7] (one 16-byte load) for its four keys
//     16s + {2t, 2t+1, 8+2t, 9+2t}; PRMT interleaves key pairs. The lane ends up owning O[q][16t .. 16t+15]: two 16-byte stores.
// The NORMALISED probabilities are rounded to bf16 before P V (ggml's bf16 mul_mat rounds its f32 operand), as in attn_mimi_kernel.
// (tcgen05 cannot be used here: its minimum M is 64 and a CTA pair per 16-row problem would idle 3/4 of the datapath.)
// ------------------------------------------------------------------------------------------------

struct MimiMaskRow { int lo; int a, b; };      // masked iff c >= lo || (a < c && c <= b) || c >= 250   (reference pattern, row j)
__device__ __forceinline__ MimiMaskRow mimi_mask_row(int offset, int j) {
    const int start = M_CTX * 2 - M_T;
    const int base = offset <= M_CTX ? start - offset : M_CTX - (offset % M_CTX);
    MimiMaskRow r; r.lo = start + 1 + j - base; r.a = M_CTX - 1 - (M_T - j - 1) - base; r.b = M_CTX - 1 - base;
    return r;
}
__device__ __forceinline__ bool mimi_masked_fast(const MimiMaskRow& r, int c) { return c >= r.lo || (c > r.a && c <= r.b) || c >= M_CTX; }

// ------------------------------------------------------------------------------------------------
// Mimi ring attention, four warps per (slot, head): warp w owns ring slots 64w .. 64w+63 (eight key tiles). K is read ONCE: the warp's
// 16 x 64 scores stay in registers while the row max / sum are combined across the four warps through shared memory, then P (normalised,
// rounded to bf16) x V for the warp's own keys and a fixed-order (deterministic) sum of the four partial outputs. A one-warp-per-(slot,
// head) version of the same fragments left ~14 warps per SM to hide HBM latency: 74 us per layer at 256 slots for 131 MB of K/V, vs 35 us.
// ------------------------------------------------------------------------------------------------
constexpr int AM4_LD = 68;                                   // padded row of the partial-output buffers (floats)

__global__ void __launch_bounds__(128) attn_mimi_mma4_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ kc,
                                                             const __nv_bfloat16* __restrict__ vc, long long kv_slot_stride, int slot0,
                                                             const int* __restrict__ mimi_off, int mask_mode, __nv_bfloat16* __restrict__ out) {
    pdl_prologue();
    __shared__ float s_max[4][16], s_sum[4][16];
    __shared__ __align__(16) float s_o[3][16][AM4_LD];          // partial outputs of warps 1..3
    const int b = blockIdx.x / M_HEADS, h = blockIdx.x % M_HEADS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int slot = slot0 + b;
    const int offset = mimi_off[slot];
    const __nv_bfloat16* K = kc + (long long)slot * kv_slot_stride + h * D_HEAD;
    const __nv_bfloat16* V = vc + (long long)slot * kv_slot_stride + h * D_HEAD;
    uint32_t qa[4][4];
#pragma unroll
    for (int p = 0; p < 2; p++) {
        const uint4 lo = *reinterpret_cast<const uint4*>(q + ((long long)b * M_T + g) * M_DIM + h * D_HEAD + 32 * p + 8 * t);
        const uint4 hi = *reinterpret_cast<const uint4*>(q + ((long long)b * M_T + g + 8) * M_DIM + h * D_HEAD + 32 * p + 8 * t);
        qa[2 * p][0] = lo.x; qa[2 * p][1] = hi.x; qa[2 * p][2] = lo.y; qa[2 * p][3] = hi.y;
        qa[2 * p + 1][0] = lo.z; qa[2 * p + 1][1] = hi.z; qa[2 * p + 1][2] = lo.w; qa[2 * p + 1][3] = hi.w;
    }
    const MimiMaskRow mr0 = mimi_mask_row(offset, g), mr1 = mimi_mask_row(offset, g + 8);
    // ---- scores of this warp's 8 key tiles (kept in registers) ----
    float S[8][4];
#pragma unroll
    for (int half = 0; half < 2; half++) {
        uint4 kv[4][2];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int krow = min(64 * warp + 8 * (4 * half + u) + g, M_CTX - 1);        // keys 250..255 do not exist: clamp, mask below
            const __nv_bfloat16* kr = K + (long long)krow * M_DIM + 8 * t;
            kv[u][0] = *reinterpret_cast<const uint4*>(kr);
            kv[u][1] = *reinterpret_cast<const uint4*>(kr + 32);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            float (&sc)[4] = S[4 * half + u];
            sc[0] = sc[1] = sc[2] = sc[3] = 0.f;
            mma_bf16_16816(sc, qa[0], kv[u][0].x, kv[u][0].y);
            mma_bf16_16816(sc, qa[1], kv[u][0].z, kv[u][0].w);
            mma_bf16_16816(sc, qa[2], kv[u][1].x, kv[u][1].y);
            mma_bf16_16816(sc, qa[3], kv[u][1].z, kv[u][1].w);
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int c = 64 * warp + 8 * (4 * half + u) + 2 * t + e;
                bool m0, m1;
                if (mask_mode == 0) { m0 = mimi_masked_fast(mr0, c); m1 = mimi_masked_fast(mr1, c); }
                else { m0 = c >= M_CTX || mimi_masked(offset, g, c, mask_mode); m1 = c >= M_CTX || mimi_masked(offset, g + 8, c, mask_mode); }
                sc[e] = m0 ? -INFINITY : sc[e] * AT_QSCALE;            // log2 domain: one ex2.approx per probability below
                sc[2 + e] = m1 ? -INFINITY : sc[2 + e] * AT_QSCALE;
            }
        }
    }
    // ---- V rows of this warp's 64 keys: issued now, consumed after the softmax (its two block barriers would otherwise sit between the
    //      K stream and the V stream: the kernel is HBM-latency bound, 135 MB per launch) ----
    uint4 vreg[4][4];
#pragma unroll
    for (int s4 = 0; s4 < 4; s4++) {
        const int k0 = 64 * warp + 16 * s4 + 2 * t;
        vreg[s4][0] = *reinterpret_cast<const uint4*>(V + (long long)min(k0, M_CTX - 1) * M_DIM + 8 * g);
        vreg[s4][1] = *reinterpret_cast<const uint4*>(V + (long long)min(k0 + 1, M_CTX - 1) * M_DIM + 8 * g);
        vreg[s4][2] = *reinterpret_cast<const uint4*>(V + (long long)min(k0 + 8, M_CTX - 1) * M_DIM + 8 * g);
        vreg[s4][3] = *reinterpret_cast<const uint4*>(V + (long long)min(k0 + 9, M_CTX - 1) * M_DIM + 8 * g);
    }
    // ---- row max over all 250 keys ----
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; j++) { mx0 = fmaxf(mx0, fmaxf(S[j][0], S[j][1])); mx1 = fmaxf(mx1, fmaxf(S[j][2], S[j][3])); }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    if (t == 0) { s_max[warp][g] = mx0; s_max[warp][g + 8] = mx1; }
    __syncthreads();
    mx0 = fmaxf(fmaxf(s_max[0][g], s_max[1][g]), fmaxf(s_max[2][g], s_max[3][g]));
    mx1 = fmaxf(fmaxf(s_max[0][g + 8], s_max[1][g + 8]), fmaxf(s_max[2][g + 8], s_max[3][g + 8]));
    // ---- exp and row sums (every row has at least its own position unmasked, so the max is finite) ----
    float l0 = 0.f, l1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        S[j][0] = at_exp2(S[j][0] - mx0); S[j][1] = at_exp2(S[j][1] - mx0); S[j][2] = at_exp2(S[j][2] - mx1); S[j][3] = at_exp2(S[j][3] - mx1);
        l0 += S[j][0] + S[j][1]; l1 += S[j][2] + S[j][3];
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    if (t == 0) { s_sum[warp][g] = l0; s_sum[warp][g + 8] = l1; }
    __syncthreads();
    const float inv0 = 1.0f / (((s_sum[0][g] + s_sum[1][g]) + s_sum[2][g]) + s_sum[3][g]);
    const float inv1 = 1.0f / (((s_sum[0][g + 8] + s_sum[1][g + 8]) + s_sum[2][g + 8]) + s_sum[3][g + 8]);
    // ---- O_w = P_w V_w over this warp's 64 keys ----
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; n++) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
#pragma unroll
    for (int s4 = 0; s4 < 4; s4++) {
        uint32_t pa[4];
        {
            __nv_bfloat162 x;
            x = __floats2bfloat162_rn(S[2 * s4][0] * inv0, S[2 * s4][1] * inv0); pa[0] = *reinterpret_cast<uint32_t*>(&x);
            x = __floats2bfloat162_rn(S[2 * s4][2] * inv1, S[2 * s4][3] * inv1); pa[1] = *reinterpret_cast<uint32_t*>(&x);
            x = __floats2bfloat162_rn(S[2 * s4 + 1][0] * inv0, S[2 * s4 + 1][1] * inv0); pa[2] = *reinterpret_cast<uint32_t*>(&x);
            x = __floats2bfloat162_rn(S[2 * s4 + 1][2] * inv1, S[2 * s4 + 1][3] * inv1); pa[3] = *reinterpret_cast<uint32_t*>(&x);
        }
        const uint4 v0 = vreg[s4][0], v1 = vreg[s4][1], v2 = vreg[s4][2], v3 = vreg[s4][3];
        const uint32_t a0[4] = {v0.x, v0.y, v0.z, v0.w}, a1[4] = {v1.x, v1.y, v1.z, v1.w}, a2[4] = {v2.x, v2.y, v2.z, v2.w}, a3[4] = {v3.x, v3.y, v3.z, v3.w};
#pragma unroll
        for (int w = 0; w < 4; w++) {
            const uint32_t b0_lo = __byte_perm(a0[w], a1[w], 0x5410), b1_lo = __byte_perm(a2[w], a3[w], 0x5410);
            const uint32_t b0_hi = __byte_perm(a0[w], a1[w], 0x7632), b1_hi = __byte_perm(a2[w], a3[w], 0x7632);
            mma_bf16_16816(o[2 * w], pa, b0_lo, b1_lo);
            mma_bf16_16816(o[2 * w + 1], pa, b0_hi, b1_hi);
        }
    }
    // ---- fixed-order sum of the four partial outputs: warps 1..3 publish, warp 0 adds them to its own (0 + 1 + 2 + 3) ----
    // o[n][e] = O[g][8(2t+e) + n], o[n][2+e] = O[g+8][...]: the lane owns dims 16t .. 16t+15 of rows g and g+8
    if (warp > 0) {
#pragma unroll
        for (int r = 0; r < 2; r++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                float* dst = &s_o[warp - 1][g + 8 * r][16 * t + 8 * e];
                *reinterpret_cast<float4*>(dst) = make_float4(o[0][2 * r + e], o[1][2 * r + e], o[2][2 * r + e], o[3][2 * r + e]);
                *reinterpret_cast<float4*>(dst + 4) = make_float4(o[4][2 * r + e], o[5][2 * r + e], o[6][2 * r + e], o[7][2 * r + e]);
            }
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int r = 0; r < 2; r++) {
            __nv_bfloat162 pk[8];
#pragma unroll
            for (int e = 0; e < 2; e++) {
                float acc[8];
#pragma unroll
                for (int n = 0; n < 8; n++) acc[n] = o[n][2 * r + e];
#pragma unroll
                for (int w = 0; w < 3; w++) {
                    const float* src = &s_o[w][g + 8 * r][16 * t + 8 * e];
                    const float4 x = *reinterpret_cast<const float4*>(src), y = *reinterpret_cast<const float4*>(src + 4);
                    acc[0] += x.x; acc[1] += x.y; acc[2] += x.z; acc[3] += x.w; acc[4] += y.x; acc[5] += y.y; acc[6] += y.z; acc[7] += y.w;
                }
#pragma unroll
                for (int n = 0; n < 8; n += 2) pk[e * 4 + n / 2] = __floats2bfloat162_rn(acc[n], acc[n + 1]);
            }
            __nv_bfloat16* dst = out + ((long long)b * M_T + g + 8 * r) * M_DIM + h * D_HEAD + 16 * t;
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<uint4*>(&pk[0]);
            *reinterpret_cast<uint4*>(dst + 8) = *reinterpret_cast<uint4*>(&pk[4]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Flow head glue
// ------------------------------------------------------------------------------------------------
// c = LN(h; out_norm) (bf16 copy for cond_embed) and EOS logit = out_eos(bf16(c)) + bias + 4
// (reference models/flow_lm.h:114-129). One CTA per row.
__global__ void __launch_bounds__(256) head_pre_kernel(const float* __restrict__ h, int R, const float* __restrict__ w, const float* __restrict__ b,
                                                       const __nv_bfloat16* __restrict__ w_eos, const float* __restrict__ b_eos,
                                                       __nv_bfloat16* __restrict__ c_bf16, float* __restrict__ eos) {
    pdl_prologue();
    __shared__ float red[3][8];
    const int row = blockIdx.x, col = threadIdx.x * 4, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (row >= R) return;
    const float4 a = *reinterpret_cast<const float4*>(h + (long long)row * D_MODEL + col);
    float v[4] = {a.x, a.y, a.z, a.w};
    const float s1 = warp_sum(v[0] + v[1] + v[2] + v[3]);
    if (lane == 0) red[0][warp] = s1;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) tot += red[0][i];
    const float mean = tot / D_MODEL;
    float s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 4; i++) { v[i] -= mean; s2 += v[i] * v[i]; }
    s2 = warp_sum(s2);
    if (lane == 0) red[1][warp] = s2;
    __syncthreads();
    tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) tot += red[1][i];
    const float rs = 1.0f / sqrtf(tot / D_MODEL + 1e-5f);
    float dot = 0.f;
    __nv_bfloat16 yb[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float y = v[i] * rs * w[col + i];
        if (b) y += b[col + i];
        yb[i] = __float2bfloat16_rn(y);
        dot = fmaf(__bfloat162float(yb[i]), __bfloat162float(w_eos[col + i]), dot);
    }
    *reinterpret_cast<uint2*>(c_bf16 + (long long)row * D_MODEL + col) = *reinterpret_cast<uint2*>(yb);
    dot = warp_sum(dot);
    if (lane == 0) red[2][warp] = dot;
    __syncthreads();
    if (threadIdx.x == 0) {
        float d = 0.f;
#pragma unroll
        for (int i = 0; i < 8; i++) d += red[2][i];
        eos[row] = d + (b_eos ? b_eos[0] : 0.f) + 4.0f;
    }
}

// noise -> (f32, bf16) per row. Noise is either injected by the caller (identical-noise parity runs, the
// reference's injection point is GraphContext::normal_, src/context.h:465-509) or drawn on the device from a
// counter-based generator keyed by (seed, sentence stream id, generation step): Philox-4x32-10 + Box-Muller, std = sqrt(temp).
__device__ __forceinline__ void philox4x32_10(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// One CTA (128 threads) per row: the first 32 threads draw the row's noise, then every thread computes 4 of the 512 outputs of
// input_proj(bf16(noise)) (32 -> 512, reference modules/mlp.h:236; bf16 operands, fp32 accumulation like every linear here).
__global__ void __launch_bounds__(128) noise_inproj_kernel(int slot0, int n, const float* __restrict__ injected, const unsigned long long* __restrict__ seed_ptr,
                                                           const float* __restrict__ temp, const int* __restrict__ gen_step, const unsigned int* __restrict__ rng_id,
                                                           float* __restrict__ noise_f32,
                                                           const __nv_bfloat16* __restrict__ w_in_t, const float* __restrict__ b_in, float* __restrict__ xh) {
    pdl_prologue();
    __shared__ float zs[LDIM];
    const int r = blockIdx.x, slot = slot0 + r, i = threadIdx.x;
    if (r >= n) return;
    if (i < LDIM) {
        float z;
        if (injected) {
            z = injected[r * LDIM + i];
        } else {
            const float std = sqrtf(temp[slot]);
            if (std == 0.f) z = 0.f;
            else {
                uint32_t o[4];
                const unsigned long long seed = *seed_ptr;
                // counter = (sentence stream id, generation step, draw pair): the id defaults to the slot; a batch scheduler sets it to the
                // sentence's global index so that the audio does not depend on the slot / GPU the sentence happens to land on
                philox4x32_10((uint32_t)seed, (uint32_t)(seed >> 32), rng_id[slot], (uint32_t)gen_step[slot], (uint32_t)(i >> 1), 0x5054545Au, o);
                const float u1 = ((float)(o[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);
                const float u2 = ((float)(o[1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
                const float rad = sqrtf(-2.0f * logf(u1));
                float sn, cn; sincosf(6.28318530717958647692f * u2, &sn, &cn);
                z = ((i & 1) ? rad * sn : rad * cn) * std;
            }
        }
        noise_f32[r * LDIM + i] = z;
        zs[i] = __bfloat162float(__float2bfloat16_rn(z));
    }
    __syncthreads();
    // w_in_t is input_proj.weight transposed to [32][512]: thread i reads 8 contiguous bytes per input k, a warp 256 contiguous bytes
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < LDIM; k++) {
        const uint2 wv = __ldg(reinterpret_cast<const uint2*>(w_in_t + (long long)k * D_FLOW + i * 4));
        const float z = zs[k];
        acc[0] = fmaf(__uint_as_float(wv.x << 16), z, acc[0]); acc[1] = fmaf(__uint_as_float(wv.x & 0xffff0000u), z, acc[1]);
        acc[2] = fmaf(__uint_as_float(wv.y << 16), z, acc[2]); acc[3] = fmaf(__uint_as_float(wv.y & 0xffff0000u), z, acc[3]);
    }
    if (b_in) { const float4 b = *reinterpret_cast<const float4*>(b_in + i * 4); acc[0] += b.x; acc[1] += b.y; acc[2] += b.z; acc[3] += b.w; }
    *reinterpret_cast<float4*>(xh + (long long)r * D_FLOW + i * 4) = make_float4(acc[0], acc[1], acc[2], acc[3]);
}

// Decode-step entry of the FlowLM backbone, one CTA (256 threads) per utterance: h = input_linear(bf16(previous latent)) (32 -> 1024,
// reference models/flow_lm.h:99) followed by layer 0's norm1 (src/torch.h:49-60) -> bf16 A operand of the first in_proj.
__global__ void __launch_bounds__(256) flow_in_kernel(int slot0, int n, const __nv_bfloat16* __restrict__ lat_in, const __nv_bfloat16* __restrict__ w_in_t,
                                                      const float* __restrict__ b_in, const float* __restrict__ lnw, const float* __restrict__ lnb,
                                                      float* __restrict__ h, __nv_bfloat16* __restrict__ n_bf,
                                                      const int* __restrict__ cur_len, const int* __restrict__ active, const float* __restrict__ freq,
                                                      int* __restrict__ row_slot, int* __restrict__ row_pos, float2* __restrict__ cs) {
    pdl_prologue();
    __shared__ float xs[LDIM];
    __shared__ float red[2][8];
    const int r = blockIdx.x, i = threadIdx.x, warp = i >> 5, lane = i & 31;
    if (r >= n) return;
    if (i < LDIM) xs[i] = __bfloat162float(lat_in[(long long)(slot0 + r) * LDIM + i]);
    if (warp == 1) {                                           // row bookkeeping for the QKV epilogues: slot, position, RoPE table
        const int pos = cur_len[slot0 + r];
        // a finished utterance inside the stepped range is a DEAD row (row_slot < 0): no KV append (its position may already equal the
        // cache capacity), no attention; the rest of the step computes on finite garbage that nothing consumes
        if (lane == 0) { row_slot[r] = active[slot0 + r] ? slot0 + r : -1; row_pos[r] = pos; }
        const float rad = (float)pos * freq[lane];
        cs[r * 32 + lane] = make_float2(cosf(rad), sinf(rad));
    }
    __syncthreads();
    float v[4] = {0.f, 0.f, 0.f, 0.f};                         // w_in_t = input_linear.weight transposed to [32][1024] (coalesced)
#pragma unroll
    for (int k = 0; k < LDIM; k++) {
        const uint2 wv = __ldg(reinterpret_cast<const uint2*>(w_in_t + (long long)k * D_MODEL + i * 4));
        const float z = xs[k];
        v[0] = fmaf(__uint_as_float(wv.x << 16), z, v[0]); v[1] = fmaf(__uint_as_float(wv.x & 0xffff0000u), z, v[1]);
        v[2] = fmaf(__uint_as_float(wv.y << 16), z, v[2]); v[3] = fmaf(__uint_as_float(wv.y & 0xffff0000u), z, v[3]);
    }
    if (b_in) { const float4 b = *reinterpret_cast<const float4*>(b_in + i * 4); v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w; }
    *reinterpret_cast<float4*>(h + (long long)r * D_MODEL + i * 4) = make_float4(v[0], v[1], v[2], v[3]);
    const float s1 = warp_sum(v[0] + v[1] + v[2] + v[3]);
    if (lane == 0) red[0][warp] = s1;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; w++) tot += red[0][w];
    const float mean = tot / D_MODEL;
    float s2 = 0.f;
#pragma unroll
    for (int j = 0; j < 4; j++) { v[j] -= mean; s2 += v[j] * v[j]; }
    s2 = warp_sum(s2);
    if (lane == 0) red[1][warp] = s2;
    __syncthreads();
    tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; w++) tot += red[1][w];
    const float rs = 1.0f / sqrtf(tot / D_MODEL + 1e-5f);
    __nv_bfloat16 yb[4];
#pragma unroll
    for (int j = 0; j < 4; j++) { float y = v[j] * rs * lnw[i * 4 + j]; if (lnb) y += lnb[i * 4 + j]; yb[j] = __float2bfloat16_rn(y); }
    *reinterpret_cast<uint2*>(n_bf + (long long)r * D_MODEL + i * 4) = *reinterpret_cast<uint2*>(yb);
}

// ------------------------------------------------------------------------------------------------
// Mimi front end: z = latent*emb_std + emb_mean; e = Wq . f16(z) (1x1 conv, f16 operands; reference
// src/pocket_tts.cpp:472-478, models/mimi.h:77-83); depthwise x16 upsampler on one step with carried state
// (modules/conv.h:283-331): x[k][c] = e[c]*w[c][k] + e_prev[c]*w[c][16+k] (+bias). State kept = e_prev.
// ------------------------------------------------------------------------------------------------
// wq_t is the quantizer projection transposed to [32][512], wup_t the upsampler taps transposed to [32][512]: lane = channel, so
// every weight load and every store is a coalesced line.
__global__ void __launch_bounds__(512) mimi_front_kernel(int slot0, const float* __restrict__ lat_f32, const float* __restrict__ emb_std,
                                                         const float* __restrict__ emb_mean, const __half* __restrict__ wq_t,
                                                         const float* __restrict__ wup_t, const float* __restrict__ bup,
                                                         float* __restrict__ e_prev, float* __restrict__ x) {
    pdl_prologue();
    __shared__ float z[LDIM];
    const int slot = slot0 + blockIdx.x, c = threadIdx.x;
    if (c < LDIM) z[c] = __half2float(__float2half_rn(__fadd_rn(__fmul_rn(emb_std[c], lat_f32[slot * LDIM + c]), emb_mean[c])));
    __syncthreads();
    float e = 0.f;
#pragma unroll
    for (int i = 0; i < LDIM; i++) e = fmaf(__half2float(wq_t[i * M_DIM + c]), z[i], e);
    const float ep = e_prev[(long long)slot * M_DIM + c];
    e_prev[(long long)slot * M_DIM + c] = e;
    const float bias = bup ? bup[c] : 0.f;
    float* xo = x + (long long)slot * M_T * M_DIM + c;
#pragma unroll
    for (int k = 0; k < M_T; k++) {
        const float y = __fadd_rn(__fmul_rn(e, wup_t[k * M_DIM + c]), __fmul_rn(ep, wup_t[(16 + k) * M_DIM + c]));
        xo[(long long)k * M_DIM] = y + bias;
    }
}

// Stop rule + bookkeeping after the head (reference src/pocket_tts.cpp:457-467,487-489) and the Mimi front end in one launch. Per slot:
//   eos_step = first step with logit+4 > 0; stop when gen_step >= eos_step + frames_after_eos; hard cap max_gen_len.
// produced[r] = 1 when this step emits a frame. Hands the new latent to the next step (bf16 copy = the A operand of input_linear),
// advances the FlowLM position, then runs mimi_front_kernel's math on the latent this step produced.
__global__ void __launch_bounds__(512) step_front_kernel(int slot0, int n, const float* __restrict__ eos, const float* __restrict__ latent,
                                                         int* __restrict__ cur_len, int* __restrict__ gen_step, int* __restrict__ eos_step,
                                                         const int* __restrict__ max_gen, const int* __restrict__ fae, int* __restrict__ active,
                                                         __nv_bfloat16* __restrict__ lat_in_bf16, float* __restrict__ lat_f32, int* __restrict__ produced,
                                                         float* __restrict__ eos_out, const float* __restrict__ emb_std, const float* __restrict__ emb_mean,
                                                         const __half* __restrict__ wq_t, const float* __restrict__ wup_t, const float* __restrict__ bup,
                                                         float* __restrict__ e_prev, float* __restrict__ x) {
    pdl_prologue();
    __shared__ float z[LDIM];
    __shared__ int emit;
    const int r = blockIdx.x, slot = slot0 + r, c = threadIdx.x;
    if (r >= n) return;
    if (c == 0) {
        int e = 0;
        if (active[slot]) {
            const int g = gen_step[slot];
            int es = eos_step[slot];
            if (eos[r] > 0.f && es == -1) es = g;
            eos_step[slot] = es;
            cur_len[slot] += 1;                                   // increment_states (pocket_tts.cpp:96)
            if (es != -1 && g >= es + fae[slot]) { gen_step[slot] = max_gen[slot]; active[slot] = 0; }
            else {
                e = 1; gen_step[slot] = g + 1;
                if (g + 1 >= max_gen[slot]) active[slot] = 0;     // next receive would hit the cap (pocket_tts.cpp:450-453,495)
            }
        }
        emit = e; produced[r] = e; if (eos_out) eos_out[r] = eos[r];
    }
    __syncthreads();
    if (c < LDIM) {
        float v;
        if (emit) { v = latent[r * LDIM + c]; lat_f32[slot * LDIM + c] = v; lat_in_bf16[slot * LDIM + c] = __float2bfloat16_rn(v); }
        else v = lat_f32[slot * LDIM + c];
        z[c] = __half2float(__float2half_rn(__fadd_rn(__fmul_rn(emb_std[c], v), emb_mean[c])));
    }
    __syncthreads();
    float e = 0.f;
#pragma unroll
    for (int i = 0; i < LDIM; i++) e = fmaf(__half2float(wq_t[i * M_DIM + c]), z[i], e);
    const float ep = e_prev[(long long)slot * M_DIM + c];
    e_prev[(long long)slot * M_DIM + c] = e;
    const float bias = bup ? bup[c] : 0.f;
    float* xo = x + (long long)slot * M_T * M_DIM + c;
#pragma unroll
    for (int k = 0; k < M_T; k++) {
        const float y = __fadd_rn(__fmul_rn(e, wup_t[k * M_DIM + c]), __fmul_rn(ep, wup_t[(16 + k) * M_DIM + c]));
        xo[(long long)k * M_DIM] = y + bias;
    }
}

// End-of-step upkeep for the streaming convs: every conv input buffer is [slot][S + T][C] with the S carried
// rows first (reference modules/conv.h:60-76 keeps the last K-stride inputs; the transposed convs keep the last
// input row instead of the reference's partial output, see DESIGN.md). Copies the last S rows to the front.
struct ShiftDesc { __half* buf; long long slot_stride; int S, T, C; };
struct ShiftAll { ShiftDesc d[9]; int n; };
__global__ void shift_states_kernel(ShiftAll sa, int slot0, int* __restrict__ mimi_off) {
    pdl_prologue();
    const ShiftDesc d = sa.d[blockIdx.y];
    const int slot = slot0 + blockIdx.x;
    __half* base = d.buf + (long long)slot * d.slot_stride;
    const int n8 = d.S * d.C / 8;                               // 16-byte pieces (every C here is a multiple of 8)
    // source rows [T, T+S) and destination rows [0, S) never overlap because T >= S for every conv here.
    const uint4* src = reinterpret_cast<const uint4*>(base + (long long)d.T * d.C);
    uint4* dst = reinterpret_cast<uint4*>(base);
    for (int i = threadIdx.x; i < n8; i += blockDim.x) dst[i] = src[i];
    if (blockIdx.y == 0 && threadIdx.x == 0) mimi_off[slot] += M_T;
}

// Sentence start (reference src/pocket_tts.cpp:416-444, models/mimi.h:71-75): zero the carried conv state rows
// and the upsampler state, reset the Mimi offset. The KV prefix restore is done with device copies by the host.
__global__ void reset_slot_kernel(ShiftAll sa, int slot, float* __restrict__ e_prev, int* __restrict__ mimi_off) {
    pdl_prologue();
    const ShiftDesc d = sa.d[blockIdx.y];
    __half* base = d.buf + (long long)slot * d.slot_stride;
    for (int i = threadIdx.x; i < d.S * d.C; i += blockDim.x) base[i] = __float2half_rn(0.f);
    if (blockIdx.y == 0) {
        for (int i = threadIdx.x; i < M_DIM; i += blockDim.x) e_prev[(long long)slot * M_DIM + i] = 0.f;
        if (threadIdx.x == 0) mimi_off[slot] = 0;
    }
}

}  // namespace ptts
