// encoder.cuh — kernels of the voice-cloning encoder (DESIGN.md §4.6): 24 kHz PCM -> SEANet encoder -> encoder transformer -> strided
// downsample -> speaker projection -> audio_prompt rows. Everything that is a GEMM runs through the engine's GEMM family (strided convs as
// 2-tap windows over rows of r*C channels); the kernels here are the pieces that are not a GEMM.
#pragma once
#include "common.cuh"

namespace ptts {

constexpr int ENC_WIN = M_CTX;               // encoder attention: key j is visible to query i iff 0 <= i - j < ENC_WIN
constexpr int ENC_HOP = 1920;                // samples per 12.5 Hz output row
constexpr int ENC_FRONT_K = 7;

// Front conv k7 1 -> 64 (C = 1 is no GEMM: K % 64 != 0). pcm = 6 zero samples of causal padding followed by the (zero-padded) signal.
// y[t][c] = b[c] + sum_j w[c][j] * f16(pcm[t + j]) (f16 operands, f32 accumulation like every conv); writes the f32 residual row and
// the f16 ELU row that the first residual block reads.
__global__ void __launch_bounds__(256) enc_front_kernel(const float* __restrict__ pcm, const __half* __restrict__ w, const float* __restrict__ b, int L,
                                                        float* __restrict__ y, __half* __restrict__ a) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)L * 64) return;
    const int t = (int)(idx >> 6), c = (int)(idx & 63);
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < ENC_FRONT_K; j++) acc = fmaf(__half2float(w[c * ENC_FRONT_K + j]), __half2float(__float2half_rn(pcm[t + j])), acc);
    const float v = acc + (b ? b[c] : 0.f);
    y[idx] = v;
    a[idx] = __float2half_rn(elu_f(v));
}

// RoPE table of rows 0 .. R-1 at positions 0 .. R-1 (same arithmetic as prepare_mimi_kernel).
__global__ void enc_rope_kernel(const float* __restrict__ freq, float2* __restrict__ cs, int R) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * 32) return;
    const float rad = (float)(idx >> 5) * freq[idx & 31];
    cs[idx] = make_float2(cosf(rad), sinf(rad));
}

// Downsample input: f16 rows of the transformer output behind 16 copies of row 0 (causal padding with pad_mode = "replicate").
__global__ void enc_ds_pad_kernel(const float* __restrict__ x, int R, __half* __restrict__ ds) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)(R + 16) * M_DIM) return;
    const long long r = idx / M_DIM, c = idx % M_DIM;
    ds[idx] = __float2half_rn(x[(r < 16 ? 0 : r - 16) * M_DIM + c]);
}

__global__ void enc_to_bf16_kernel(const float* __restrict__ x, long long n, __nv_bfloat16* __restrict__ o) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) o[i] = __float2bfloat16_rn(x[i]);
}

// Causal sliding-window attention over R rows (8 heads x 64, positions = row indices): q, k rotated and de-interleaved per head like
// the Mimi decoder's, v plain, all bf16 [R][512]. One CTA = 64 consecutive queries x one head; the keys they can see (at most
// 64 + 249 rows) are staged in shared memory. One warp per query: lane l scores keys l, l+32, ... of the window (f32 dot products of
// the bf16 operands, scale 1/8), the window's max and sum come from warp reductions, the probabilities exp(s - max) are rounded to bf16
// and multiply v (lane l owns output dims 2l, 2l+1); out = that sum / (f32 sum of the unrounded probabilities), stored as bf16.
constexpr int AW_Q = 64, AW_WARPS = 8, AW_KROWS = AW_Q + ENC_WIN - 1, AW_KLD = 66;   // K rows padded to 33 words: conflict-free per-lane rows
constexpr int AW_SLOTS = (ENC_WIN + 31) / 32;
constexpr size_t AW_KBYTES = ((size_t)AW_KROWS * AW_KLD * 2 + 15) / 16 * 16;   // v rows behind it take 16-byte stores
constexpr size_t AW_SMEM = AW_KBYTES + (size_t)AW_KROWS * 64 * 2 + AW_WARPS * 64 * 4 + AW_WARPS * AW_SLOTS * 32 * 4;

__global__ void __launch_bounds__(AW_WARPS * 32) attn_window_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                                                                    const __nv_bfloat16* __restrict__ v, int R, __nv_bfloat16* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char aw_smem[];
    __nv_bfloat16* ks = reinterpret_cast<__nv_bfloat16*>(aw_smem);
    __nv_bfloat16* vs = reinterpret_cast<__nv_bfloat16*>(aw_smem + AW_KBYTES);
    float* qs = reinterpret_cast<float*>(vs + AW_KROWS * 64);
    float* ps = qs + AW_WARPS * 64;
    const int h = blockIdx.y, q0 = blockIdx.x * AW_Q, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kbase = max(0, q0 - (ENC_WIN - 1)), kend = min(R, q0 + AW_Q), nk = kend - kbase;
    for (int i = tid; i < nk * 8; i += blockDim.x) {          // 8 x 16 bytes per 64-dim row
        const int r = i >> 3, part = i & 7;
        const long long g = (long long)(kbase + r) * M_DIM + h * 64 + part * 8;
        const uint4 kv = *reinterpret_cast<const uint4*>(k + g), vv = *reinterpret_cast<const uint4*>(v + g);
        uint32_t* kd = reinterpret_cast<uint32_t*>(ks + r * AW_KLD + part * 8);
        kd[0] = kv.x; kd[1] = kv.y; kd[2] = kv.z; kd[3] = kv.w;
        *reinterpret_cast<uint4*>(vs + r * 64 + part * 8) = vv;
    }
    __syncthreads();
    float* qw = qs + warp * 64;
    float* pw = ps + warp * AW_SLOTS * 32;
    for (int qi = q0 + warp; qi < kend; qi += AW_WARPS) {
        const __nv_bfloat162 qv = reinterpret_cast<const __nv_bfloat162*>(q + (long long)qi * M_DIM + h * 64)[lane];
        qw[2 * lane] = __low2float(qv); qw[2 * lane + 1] = __high2float(qv);
        __syncwarp();
        const int j0 = qi - (ENC_WIN - 1);                    // key of window slot 0 (may be negative: masked)
        float s[AW_SLOTS], mx = -INFINITY;
#pragma unroll
        for (int m = 0; m < AW_SLOTS; m++) {
            const int kk = lane + 32 * m, j = j0 + kk;
            s[m] = -INFINITY;
            if (kk < ENC_WIN && j >= 0) {
                const __nv_bfloat162* kr = reinterpret_cast<const __nv_bfloat162*>(ks + (j - kbase) * AW_KLD);
                float acc = 0.f;
#pragma unroll
                for (int d = 0; d < 32; d++) { const float2 kf = __bfloat1622float2(kr[d]); acc = fmaf(qw[2 * d], kf.x, acc); acc = fmaf(qw[2 * d + 1], kf.y, acc); }
                s[m] = acc * 0.125f;
            }
            mx = fmaxf(mx, s[m]);
        }
        mx = warp_max(mx);
        float l = 0.f;
#pragma unroll
        for (int m = 0; m < AW_SLOTS; m++) {
            const float p = s[m] == -INFINITY ? 0.f : __expf(s[m] - mx);
            l += p;
            pw[lane + 32 * m] = __bfloat162float(__float2bfloat16_rn(p));
        }
        l = warp_sum(l);
        __syncwarp();
        float o0 = 0.f, o1 = 0.f;
        const int kk0 = max(0, -j0);
        for (int kk = kk0; kk < ENC_WIN; kk++) {
            const float p = pw[kk];
            const float2 vf = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(vs + (j0 + kk - kbase) * 64)[lane]);
            o0 = fmaf(p, vf.x, o0); o1 = fmaf(p, vf.y, o1);
        }
        const float inv = 1.f / l;
        reinterpret_cast<__nv_bfloat162*>(out + (long long)qi * M_DIM + h * 64)[lane] = __floats2bfloat162_rn(o0 * inv, o1 * inv);
        __syncwarp();                                          // qw / pw are rewritten by this warp's next query
    }
}

}  // namespace ptts
