// Generic "rows x weights^T" GEMM family with one fused epilogue:
//     C[r][n] = sum_k A(r)[k] * W[n][k]        A(r) = A + amap.off(r, rps)   (rows may OVERLAP: a causal
//                                               conv window over channel-last data is one contiguous A row)
// Operands are bf16 x bf16 (linears: reference torch_nn_linear, src/torch.h:79-87, with a BF16 checkpoint
// ggml rounds the activation operand to bf16) or f16 x f16 (convs: ggml_conv_1d = im2col(F16) + f16 mul_mat,
// src/pocket_tts/modules/conv.h:81), always with fp32 accumulation.
//
// This file holds the CUDA-core implementations (any R, any N) used for small batches and as the
// validation path; gemm_tc.cuh holds the tcgen05/TMEM/TMA implementation selected for large R.
#pragma once
#include "common.cuh"

namespace ptts {

// ------------------------------------------------------------------------------------------------
// Fused epilogue. NV consecutive columns [col0, col0+NV) of one row; col0 % NV == 0, NV even.
// ------------------------------------------------------------------------------------------------
template <int NV>
__device__ __forceinline__ void epi_apply(const Epi& e, int row, int col0, const float (&acc)[NV], int N) {
    if (e.mode == EPI_GENERIC) {
        const long long ro = e.out ? e.out_map.off(row, e.rps) : 0;
        const long long r2 = e.out2 ? e.out2_map.off(row, e.rps) : 0;
        const long long rr = e.resid ? e.resid_map.off(row, e.rps) : 0;
#pragma unroll
        for (int i = 0; i < NV; i++) {
            const int col = col0 + i;
            if (col >= N) break;
            float v = acc[i];
            if (e.bias) v += e.bias[col];
            if (e.colscale) v *= e.colscale[col];
            if (e.rowmul) v *= e.rowmul[(long long)row * e.rowmul_ld + col];
            if (e.resid) v += e.resid[rr + col];
            if (e.out) e.out[ro + col] = v;
            if (e.out2_type != OUT2_NONE) {
                const float a = apply_act(v, e.act);
                if (e.out2_type == OUT2_BF16) {
                    ((__nv_bfloat16*)e.out2)[r2 + col] = __float2bfloat16_rn(a);
                } else if (e.out2_type == OUT2_F16) {
                    ((__half*)e.out2)[r2 + col] = __float2half_rn(a);
                } else {  // OUT2_F16_SPLIT: a ~= hi + lo, both f16 (near-fp32 operand for the f32 convT of the reference)
                    const __half hi = __float2half_rn(a);
                    ((__half*)e.out2)[r2 + col] = hi;
                    ((__half*)e.out2)[r2 + col + e.split_off] = __float2half_rn(a - __half2float(hi));
                }
            }
        }
        return;
    }
    // ---- QKV epilogues: RoPE + cache append (reference modules/transformer.h:64-153, rope.h:183-272;
    //      Mimi: modules/mimi_transformer.h:586-712, rope.h:86-181) ----
    const bool mimi = (e.mode == EPI_MIMI_QKV);
    const int D = mimi ? M_DIM : D_MODEL;
    const int slot = e.kv_linear ? 0 : e.row_slot[row];
    const int pos = e.kv_linear ? row : e.row_pos[row];
    if (slot < 0) return;                 // dead row (finished utterance): nothing is appended or handed on
#pragma unroll
    for (int p = 0; p < NV; p += 2) {
        const int col = col0 + p;
        if (col >= N) break;
        float a = acc[p], b = acc[p + 1];
        if (e.bias) { a += e.bias[col]; b += e.bias[col + 1]; }
        const int part = col / D;             // 0 q, 1 k, 2 v
        const int c = col - part * D;         // even column inside the part
        if (part < 2) {
            const int h = c >> 6, i = (c & 63) >> 1;
            const float2 cs = e.cs[row * 32 + i];
            const float re = a * cs.x - b * cs.y;
            const float im = a * cs.y + b * cs.x;
            const int i_re = (h << 6) + i, i_im = i_re + 32;   // de-interleaved [re(0..31) | im(0..31)]
            if (part == 0) {
                if (mimi) { e.q_out_bf16[(long long)row * D + i_re] = __float2bfloat16_rn(re); e.q_out_bf16[(long long)row * D + i_im] = __float2bfloat16_rn(im); }
                else      { e.q_out_f32[(long long)row * D + i_re] = re; e.q_out_f32[(long long)row * D + i_im] = im; }
            } else {
                const long long base = (long long)slot * e.kv_slot_stride + (long long)(mimi && !e.kv_linear ? pos % M_CTX : pos) * D;
                if (!mimi && e.kv_f32) { ((float*)e.kcache)[base + i_re] = re; ((float*)e.kcache)[base + i_im] = im; }
                else { ((__nv_bfloat16*)e.kcache)[base + i_re] = __float2bfloat16_rn(re); ((__nv_bfloat16*)e.kcache)[base + i_im] = __float2bfloat16_rn(im); }
            }
        } else {
            const long long base = (long long)slot * e.kv_slot_stride + (long long)(mimi && !e.kv_linear ? pos % M_CTX : pos) * D + c;
            if (!mimi && e.kv_f32) { ((float*)e.vcache)[base] = a; ((float*)e.vcache)[base + 1] = b; }
            else { ((__nv_bfloat16*)e.vcache)[base] = __float2bfloat16_rn(a); ((__nv_bfloat16*)e.vcache)[base + 1] = __float2bfloat16_rn(b); }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// CUDA-core tiled GEMM (any R): 64x64x32 tiles, 256 threads, 4x4 micro-tiles, fp32 FFMA.
// Requires K % 32 == 0 and 16-byte aligned A rows / W rows.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) gemm_ffma_kernel(const T* __restrict__ A, RowMap amap, int a_rps,
                                                        const T* __restrict__ W, int R, int N, int K, Epi epi) {
    pdl_prologue();
    constexpr int BM = 64, BN = 64, BK = 32, LD = BM + 4;
    __shared__ __align__(16) float As[BK][LD];
    __shared__ __align__(16) float Ws[BK][LD];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int lr = tid >> 2, lk = (tid & 3) * 8;      // this thread stages row lr, k-segment lk..lk+7
    const int arow = m0 + lr, wrow = n0 + lr;
    const T* ap = (arow < R) ? A + amap.off(arow, a_rps) + lk : nullptr;
    const T* wp = (wrow < N) ? W + (long long)wrow * K + lk : nullptr;
    const int ty = tid >> 4, tx = tid & 15;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += BK) {
        uint4 av = make_uint4(0, 0, 0, 0), wv = make_uint4(0, 0, 0, 0);
        if (ap) av = *reinterpret_cast<const uint4*>(ap + k0);
        if (wp) wv = __ldg(reinterpret_cast<const uint4*>(wp + k0));
        const T* ae = reinterpret_cast<const T*>(&av);
        const T* we = reinterpret_cast<const T*>(&wv);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; j++) { As[lk + j][lr] = to_f32<T>(ae[j]); Ws[lk + j][lr] = to_f32<T>(we[j]); }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; k++) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int row = m0 + ty * 4 + i;
        if (row < R) epi_apply<4>(epi, row, n0 + tx * 4, acc[i], N);
    }
}

// ------------------------------------------------------------------------------------------------
// Small-R GEMV-like kernel (R <= RMAX): one warp per column PAIR, weights streamed once with 128-bit
// loads, warp-shuffle reductions. This is the low-batch path: it is weight-bandwidth bound.
// Requires K % 8 == 0, N even.
// ------------------------------------------------------------------------------------------------
template <typename T, int RMAX>
__global__ void __launch_bounds__(256) gemv_small_kernel(const T* __restrict__ A, RowMap amap, int a_rps,
                                                         const T* __restrict__ W, int R, int N, int K, Epi epi) {
    pdl_prologue();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int n0 = warp * 2;
    if (n0 >= N) return;
    const T* w0 = W + (long long)n0 * K;
    const T* w1 = w0 + K;
    float acc[RMAX][2];
#pragma unroll
    for (int r = 0; r < RMAX; r++) acc[r][0] = acc[r][1] = 0.f;
    for (int k = lane * 8; k < K; k += 256) {
        const uint4 wv0 = __ldg(reinterpret_cast<const uint4*>(w0 + k));
        const uint4 wv1 = __ldg(reinterpret_cast<const uint4*>(w1 + k));
        const T* e0 = reinterpret_cast<const T*>(&wv0);
        const T* e1 = reinterpret_cast<const T*>(&wv1);
        float f0[8], f1[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { f0[j] = to_f32<T>(e0[j]); f1[j] = to_f32<T>(e1[j]); }
#pragma unroll
        for (int r = 0; r < RMAX; r++) {
            if (r < R) {
                const uint4 av = *reinterpret_cast<const uint4*>(A + amap.off(r, a_rps) + k);
                const T* ae = reinterpret_cast<const T*>(&av);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const float a = to_f32<T>(ae[j]);
                    acc[r][0] = fmaf(a, f0[j], acc[r][0]);
                    acc[r][1] = fmaf(a, f1[j], acc[r][1]);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < RMAX; r++) {
        if (r < R) {
            const float v0 = warp_sum(acc[r][0]), v1 = warp_sum(acc[r][1]);
            if (lane == 0) { const float v[2] = {v0, v1}; epi_apply<2>(epi, r, n0, v, N); }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// GEMV with the LayerNorm that produces its input fused in (batch 1-2 decode): x is the f32 row, every CTA first normalises the
// R <= 2 rows into shared memory (ggml_norm semantics like layernorm_kernel, optional affine, optional AdaLN modulate, result rounded
// to bf16 exactly as the separate LN kernel stores it), then each warp computes two output columns. The redundant per-CTA LN costs
// ~1 us of latency per launch and removes one launch (~4.7 us at this batch size) per LayerNorm: the step is launch bound there.
// ------------------------------------------------------------------------------------------------
struct LnArgs { const float* w = nullptr; const float* b = nullptr; float eps = 0.f; const float* shift = nullptr; const float* scale = nullptr; int mod_ld = 0; };

template <int K>
__global__ void __launch_bounds__(256) gemv_ln_kernel(const float* __restrict__ x, LnArgs ln, const __nv_bfloat16* __restrict__ W, int R, int N, Epi epi) {
    pdl_prologue();
    constexpr int PER = K / 256;                                 // elements per thread and row in the LN prologue
    __shared__ float xs[2][K];
    __shared__ float red[2][8];
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    for (int r = 0; r < R; r++) {
        float v[PER]; float s = 0.f;
#pragma unroll
        for (int i = 0; i < PER; i++) { v[i] = x[(long long)r * K + tid * PER + i]; s += v[i]; }
        s = warp_sum(s);
        if (lane == 0) red[0][wid] = s;
        __syncthreads();
        float tot = 0.f;
#pragma unroll
        for (int w = 0; w < 8; w++) tot += red[0][w];
        const float mean = tot / K;
        float s2 = 0.f;
#pragma unroll
        for (int i = 0; i < PER; i++) { v[i] -= mean; s2 += v[i] * v[i]; }
        s2 = warp_sum(s2);
        if (lane == 0) red[1][wid] = s2;
        __syncthreads();
        tot = 0.f;
#pragma unroll
        for (int w = 0; w < 8; w++) tot += red[1][w];
        const float rs = 1.0f / sqrtf(tot / K + ln.eps);
#pragma unroll
        for (int i = 0; i < PER; i++) {
            const int c = tid * PER + i;
            float y = v[i] * rs;
            if (ln.w) y *= ln.w[c];
            if (ln.b) y += ln.b[c];
            if (ln.scale) y = y * (ln.scale[(long long)r * ln.mod_ld + c] + 1.f) + ln.shift[(long long)r * ln.mod_ld + c];
            xs[r][c] = __bfloat162float(__float2bfloat16_rn(y));
        }
        __syncthreads();
    }
    const int n0 = (blockIdx.x * 8 + wid) * 2;
    if (n0 >= N) return;
    const __nv_bfloat16* w0 = W + (long long)n0 * K;
    const __nv_bfloat16* w1 = w0 + K;
    float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    for (int k = lane * 8; k < K; k += 256) {
        const uint4 wv0 = __ldg(reinterpret_cast<const uint4*>(w0 + k)), wv1 = __ldg(reinterpret_cast<const uint4*>(w1 + k));
        const uint32_t a0[4] = {wv0.x, wv0.y, wv0.z, wv0.w}, a1[4] = {wv1.x, wv1.y, wv1.z, wv1.w};
#pragma unroll
        for (int r = 0; r < 2; r++) {
            if (r < R) {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const float xa = xs[r][k + 2 * j], xb = xs[r][k + 2 * j + 1];
                    acc[r][0] = fmaf(xa, __uint_as_float(a0[j] << 16), acc[r][0]); acc[r][0] = fmaf(xb, __uint_as_float(a0[j] & 0xffff0000u), acc[r][0]);
                    acc[r][1] = fmaf(xa, __uint_as_float(a1[j] << 16), acc[r][1]); acc[r][1] = fmaf(xb, __uint_as_float(a1[j] & 0xffff0000u), acc[r][1]);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; r++) {
        if (r < R) {
            const float v0 = warp_sum(acc[r][0]), v1 = warp_sum(acc[r][1]);
            if (lane == 0) { const float v[2] = {v0, v1}; epi_apply<2>(epi, r, n0, v, N); }
        }
    }
}

// Final SEANet conv (64 -> 1 channel, k=3; reference seanet.h:208, defaults.h:113-118). Four lanes per output sample
// (16 channels x 3 taps each, two shuffles to finish), eight consecutive samples per warp so every global load
// instruction covers 1 KB of contiguous channel-last rows. f16 operands, fp32 accumulation like every other conv.
__global__ void __launch_bounds__(256) conv_n1_kernel(const __half* __restrict__ A, RowMap amap, int rps,
                                                      const __half* __restrict__ W, const float* __restrict__ bias,
                                                      int R, int K, float* __restrict__ out) {
    pdl_prologue();
    const int gl = blockIdx.x * blockDim.x + threadIdx.x;
    const int row = gl >> 2, g = gl & 3;                       // output sample, channel group (16 channels)
    const bool live = row < R;
    float acc = 0.f;
    if (live) {
        const __half* a = A + amap.off(row, rps) + g * 16;     // window = 3 consecutive rows of 64 channels (K == 192)
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const uint4 a0 = *reinterpret_cast<const uint4*>(a + k * 64), a1 = *reinterpret_cast<const uint4*>(a + k * 64 + 8);
            const uint4 w0 = __ldg(reinterpret_cast<const uint4*>(W + k * 64 + g * 16)), w1 = __ldg(reinterpret_cast<const uint4*>(W + k * 64 + g * 16 + 8));
            const __half2* ah0 = reinterpret_cast<const __half2*>(&a0); const __half2* ah1 = reinterpret_cast<const __half2*>(&a1);
            const __half2* wh0 = reinterpret_cast<const __half2*>(&w0); const __half2* wh1 = reinterpret_cast<const __half2*>(&w1);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float2 x = __half22float2(ah0[j]), y = __half22float2(wh0[j]), x2 = __half22float2(ah1[j]), y2 = __half22float2(wh1[j]);
                acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc); acc = fmaf(x2.x, y2.x, acc); acc = fmaf(x2.y, y2.y, acc);
            }
        }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (live && g == 0) out[row] = acc + (bias ? bias[0] : 0.f);
}

}  // namespace ptts
