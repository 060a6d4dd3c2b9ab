// encoder.cuh — kernels of the voice-cloning encoder (DESIGN.md §4.6): PCM resampled to 24 kHz -> SEANet encoder -> encoder transformer -> strided
// downsample -> speaker projection -> audio_prompt rows. Everything that is a GEMM runs through the engine's GEMM family (strided convs as
// 2-tap windows over rows of r*C channels); the kernels here are the pieces that are not a GEMM.
#pragma once
#include <algorithm>
#include "common.cuh"

namespace ptts {

constexpr int ENC_WIN = M_CTX;               // encoder attention: key j is visible to query i iff 0 <= i - j < ENC_WIN
constexpr int ENC_HOP = 1920;                // samples per 12.5 Hz output row
constexpr int ENC_FRONT_K = 7;
constexpr int ENC_SR = 24000, ENC_SR_MIN = 8000, ENC_SR_MAX = 192000;   // the encoder's rate; accepted input rates (integers)

// ---- resampling to 24 kHz in front of the encoder: torchaudio.functional.resample(x, sr, 24000) with its defaults (sinc_interp_hann,
// lowpass_filter_width L = 6, rolloff 0.99), its float64 filter rounded to f32. With o = sr / g and m = 24000 / g (g = gcd), output
// j = q m + i is sum_k K[i][k] xpad[q o + k], xpad = [w zeros | x | w + o zeros], w = ceil(L o / base), base = 0.99 min(o, m), and
// K[i][k] = sinc(pi t) cos^2(pi t / 2L) base / o with t = ((k - w) / o - i / m) base clamped to +-L. A tap is nonzero in f32 only for
// |t| < L, i.e. |(k - w) m - i o| <= X = floor(600 max(o, m) / 99) (exact integers), so phase i is a band of taps starting at
// d = k - w = ceil((i o - X) / m): output j reads x[s(j) .. s(j) + W - 1] with s(j) = ceil((j o - X) / m), and W is the widest band.
constexpr int RS_L = 6, RS_THREADS = 256;

__host__ __device__ inline long long rs_ceil_div(long long a, long long b) { return a >= 0 ? (a + b - 1) / b : -((-a) / b); }
__host__ __device__ inline long long rs_floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

struct ResamplePlan {
    int sr = 0, o = 0, m = 0, w = 0, W = 0; long long X = 0;
    long long first_tap(long long j) const { return rs_ceil_div(j * o - X, m); }
    int span_max() const { return (int)rs_ceil_div((long long)(RS_THREADS - 1) * o, m) + W; }   // input samples one CTA stages
};
inline ResamplePlan resample_plan(int sr) {
    ResamplePlan p; p.sr = sr;
    long long a = sr, b = ENC_SR;
    while (b) { const long long r = a % b; a = b; b = r; }
    p.o = (int)(sr / a); p.m = (int)(ENC_SR / a);
    const double base = (double)std::min(p.o, p.m) * 0.99;
    p.w = (int)std::ceil((double)(RS_L * p.o) / base);
    p.X = 600LL * std::max(p.o, p.m) / 99;
    for (int i = 0; i < p.m; i++)
        p.W = std::max(p.W, (int)(rs_floor_div((long long)i * p.o + p.X, p.m) - rs_ceil_div((long long)i * p.o - p.X, p.m) + 1));
    return p;
}

// coef[i][b] = K[i][w + ceil((i o - X) / m) + b] for b < W (0 past the phase's band), evaluated in float64 in torchaudio's operation
// order and rounded once.
__global__ void resample_table_kernel(int o, int m, int w, int W, long long X, float* __restrict__ coef) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)m * W) return;
    const int i = (int)(idx / W), b = (int)(idx % W);
    const long long d = rs_ceil_div((long long)i * o - X, m) + b;
    float c = 0.f;
    if (d <= rs_floor_div((long long)i * o + X, m) && d >= -w && d < w + o) {
        const double base = (double)min(o, m) * 0.99;
        double t = (double)(-i) / m + (double)d / o;
        t *= base;
        t = fmin(fmax(t, -(double)RS_L), (double)RS_L);
        const double cw = cos(t * M_PI / RS_L / 2), window = cw * cw;
        t *= M_PI;
        double k = t == 0.0 ? 1.0 : sin(t) / t;
        k *= window * (base / o);
        c = __double2float_rn(k);
    }
    coef[idx] = c;
}

// One thread per 24 kHz output y[j], j < L0 (= 1920 T): sum_b coef[j % m][b] x[s(j) + b] over the band in increasing b (f32 FMA), x = 0
// outside [0, n); outputs n24 .. L0-1 are the encoder's zero right padding. Each CTA stages the input span its 256 outputs read.
__global__ void __launch_bounds__(RS_THREADS) resample_kernel(const float* __restrict__ x, long long n, const float* __restrict__ coef, int o, int m,
                                                             int W, long long X, long long n24, long long L0, float* __restrict__ y) {
    extern __shared__ float rs_span[];
    const long long j0 = (long long)blockIdx.x * RS_THREADS, j = j0 + threadIdx.x;
    if (j0 >= n24) { if (j < L0) y[j] = 0.f; return; }
    const long long s0 = rs_ceil_div(j0 * o - X, m), jl = min(j0 + RS_THREADS, n24) - 1;
    const int span = (int)(rs_ceil_div(jl * o - X, m) + W - s0);
    for (int p = threadIdx.x; p < span; p += RS_THREADS) {
        const long long g = s0 + p;
        rs_span[p] = g >= 0 && g < n ? x[g] : 0.f;
    }
    __syncthreads();
    if (j < n24) {
        const float* c = coef + (j % m) * W;
        const float* xs = rs_span + (rs_ceil_div(j * o - X, m) - s0);
        float acc = 0.f;
        for (int b = 0; b < W; b++) acc = fmaf(c[b], xs[b], acc);
        y[j] = acc;
    } else if (j < L0) {
        y[j] = 0.f;
    }
}

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
