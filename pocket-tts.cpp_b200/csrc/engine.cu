// engine.cu — device layer of the B200 Pocket-TTS engine: weights, per-utterance slots, ragged prefill and the
// batched per-frame step (FlowLM backbone -> LSD flow head -> Mimi decoder -> 1920 PCM samples), replayed as CUDA
// graphs on two streams (run_step: the Mimi decode of frame t overlaps the FlowLM step of frame t+1).
// C ABI declared in include/ptts_b200.h. No CPU fallback: everything below runs on the device or aborts.
#include "../../include/ptts_b200.h"
#include "common.cuh"
#include "gemm.cuh"
#include "gemm_tc.cuh"
#include "kernels.cuh"
#include "persistent.cuh"
#include "head_fused.cuh"
#include "seanet_tail.cuh"
#include "seanet_res.cuh"
#include "encoder.cuh"

#include <cuda_profiler_api.h>
#include <nvtx3/nvToolsExt.h>
#include <algorithm>
#include <map>
#include <string>
#include <tuple>
#include <vector>
#include <cstring>

using namespace ptts;

namespace {

// NVTX ranges around the host-side phases (sentence start, prefill, step enqueue, collect): visible in Nsight Systems / ncu --nvtx; the
// reference only has wall-clock prints around send / receive (demos/pocket-tts.cpp:456-520). Header-only NVTX3: no-ops without a tool.
struct NvtxRange { explicit NvtxRange(const char* name) { nvtxRangePushA(name); } ~NvtxRange() { nvtxRangePop(); } };

struct HostTensor { std::vector<float> f; std::vector<int64_t> shape; int dtype; };

inline float h_bf16r(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
inline float h_silu(float x) { return x / (1.0f + expf(-x)); }

// w: [out][in] row-major (GEMV / CUDA-core paths), wk: k-block-major copy for the tensor-core path (nullptr when in % 64 != 0)
struct LinW { __nv_bfloat16* w = nullptr; __nv_bfloat16* wk = nullptr; float* b = nullptr; int out = 0, in = 0; };
struct ConvW { __half* w = nullptr; __half* wk = nullptr; float* b = nullptr; int N = 0, K = 0; };

// Decode-side work list of attn_tile_kernel for rows [0, n) whose shared prefix is (row_pfx_slot[r], row_pfx_len[r]) (0 rows: none): rows
// grouped by prefix, 64-row tiles, every prefix cut into `splits` key ranges so that tiles x splits x 16 heads fill the machine about twice.
// The longest prefix sets `splits`; a shorter one can end before its last ranges, whose items are empty (a_k0 == a_k1) and write m = -inf,
// l = 0 partials that the merges skip. Returns splits (0: no row has a prefix); rows receives the tile rows, items reference them.
int plan_prefix_tiles(const int* row_pfx_slot, const int* row_pfx_len, int n, int sms, std::vector<AtItem>& items, std::vector<int>& rows) {
    items.clear(); rows.clear();
    std::map<std::pair<int, int>, std::vector<int>> groups;
    for (int r = 0; r < n; r++) if (row_pfx_len[r] > 0) groups[{row_pfx_slot[r], row_pfx_len[r]}].push_back(r);
    int tiles = 0, max_p = 0;
    for (auto& g : groups) { tiles += ((int)g.second.size() + AT_ROWS - 1) / AT_ROWS; max_p = std::max(max_p, g.first.second); }
    if (tiles == 0) return 0;
    // ONE wave of tile CTAs (tiles x splits x 16 heads <= two resident CTAs per SM): a second, partly filled wave would cost a whole CTA time
    int splits = std::min(AF_PFX_SPLITS, std::max(1, (2 * sms) / (N_HEADS * tiles)));
    splits = std::max(1, std::min(splits, max_p / AT_KEYS));
    for (auto& g : groups) {
        const int plen = g.first.second;
        int chunk = (plen + splits - 1) / splits; chunk = (chunk + AT_KEYS - 1) / AT_KEYS * AT_KEYS;
        for (size_t i0 = 0; i0 < g.second.size(); i0 += AT_ROWS) {
            const int nr = (int)std::min<size_t>(AT_ROWS, g.second.size() - i0);
            for (int sp = 0; sp < splits; sp++) {
                AtItem it{}; it.row0 = (int)(rows.size()); it.nrows = nr; it.a_slot = g.first.first; it.a_k0 = std::min(plen, sp * chunk); it.a_k1 = std::min(plen, (sp + 1) * chunk);
                it.b_slot = 0; it.b_k0 = 0; it.b_k1 = 0; it.out_split = AF_MAX_SPLITS + sp;
                items.push_back(it);
            }
            for (int i = 0; i < nr; i++) rows.push_back(g.second[i0 + i]);
        }
    }
    return splits;
}
// Capacity of that list for max_slots rows of at most max_voices distinct prefixes.
int prefix_tiles_capacity(int max_slots, int max_voices) { return ((max_slots + AT_ROWS - 1) / AT_ROWS + max_voices + 1) * AF_PFX_SPLITS + 8; }

// Prefill work list of attn_tile_kernel (bf16 cache): the rows (slot-major, ascending positions) are cut into chunks of chunk_rows; inside a
// chunk, one item per run of <= 64 consecutive positions of one slot, with keys [0, P) of the slot's prefix slot and its own rows [P, last
// position of the run]. pfx_slot / pfx_len are indexed by slot. chunk_item0[c] = first item of chunk c (nchunks + 1 entries).
void plan_prefill_items(const int* slots, const int* pos, int total, int chunk_rows, const int* pfx_slot, const int* pfx_len,
                        std::vector<AtItem>& items, std::vector<int>& chunk_item0) {
    const int nchunks = (total + chunk_rows - 1) / chunk_rows;
    items.clear(); chunk_item0.assign(nchunks + 1, 0);
    for (int c = 0; c < nchunks; c++) {
        const int r0 = c * chunk_rows, R = std::min(chunk_rows, total - r0);
        chunk_item0[c] = (int)items.size();
        for (int i = 0; i < R;) {
            int j = i + 1;
            while (j < R && j - i < AT_ROWS && slots[r0 + j] == slots[r0 + i] && pos[r0 + j] == pos[r0 + j - 1] + 1) j++;
            const int slot = slots[r0 + i], P = pfx_len[slot];
            AtItem it{}; it.row0 = i; it.nrows = j - i; it.out_split = -1;
            it.a_slot = pfx_slot[slot]; it.a_k0 = 0; it.a_k1 = P;                                  // shared prefix rows (none: P = 0)
            it.b_slot = slot; it.b_k0 = P; it.b_k1 = pos[r0 + j - 1] + 1;                            // own rows, causal
            items.push_back(it);
            i = j;
        }
    }
    chunk_item0[nchunks] = (int)items.size();
}

}  // namespace

struct b200_engine {
    b200_config cfg{};
    cudaStream_t stream = nullptr;
    // Two-stream pipeline: the Mimi decode of frame t (tensor/ALU bound) runs on stream_m while the FlowLM step of frame t+1 (latency
    // bound small GEMMs + the HBM-bound KV stream) runs on the main stream. Hand-off buffer mx2[t & 1], events per parity.
    cudaStream_t stream_m = nullptr;
    cudaStream_t stream_c = nullptr;     // device->host PCM copies of b200_submit frames (beside the next frame's Mimi decode instead of in front of it)
    cudaStream_t stream_n = nullptr;     // host->device noise uploads of b200_submit (its own stream: behind a PCM copy they would wait for a Mimi decode)
    cudaStream_t stream_t = nullptr;     // forked branch of the main stream: the shared-prefix tile kernel runs beside the per-utterance KV stream
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool tma_epilogue_allowed = getenv("PTTS_B200_TMA_EPILOGUE") ? atoi(getenv("PTTS_B200_TMA_EPILOGUE")) != 0 : true;   // tuning hook
    bool fork_tiles = getenv("PTTS_B200_FORK_TILES") ? atoi(getenv("PTTS_B200_FORK_TILES")) != 0 : true;   // tuning hook
    // 1: no attn_merge_kernel; the last CTA (of either attention kernel) to arrive for a (row, head) merges it. Bit-identical output, but no
    // gain: the tile CTAs usually arrive last and their extra fence + merge tail costs what the 7 us launch saved (0.9405 vs 0.9341 ms per step).
    bool counted_merge = getenv("PTTS_B200_COUNTED_MERGE") ? atoi(getenv("PTTS_B200_COUNTED_MERGE")) != 0 : false;
    cudaEvent_t ev_main[2] = {nullptr, nullptr}, ev_mimi[2] = {nullptr, nullptr};
    bool ev_mimi_valid[2] = {false, false};
    unsigned long long pipe_t = 0;       // frames enqueued through the pipeline
    bool mimi_pending = false;           // stream_m holds work the main stream has not waited for
    int last_mimi_par = 0;               // parity of the newest frame whose Mimi decode was enqueued
    std::map<std::string, HostTensor> host;
    std::vector<void*> allocs;
    bool finalized = false;
    bool pdl_active = false;   // programmatic dependent launch for the kernels being enqueued (see run_graphed)
    bool pdl_small = false, pdl_chain = false;
    bool debug_skip_mimi = getenv("PTTS_B200_DEBUG_SKIP_MIMI") != nullptr;   // diagnosis only: time the FlowLM graph alone
    int af_splits_override = getenv("PTTS_B200_AF_SPLITS") ? atoi(getenv("PTTS_B200_AF_SPLITS")) : 0;   // tuning hook
    void set_pdl(bool on) { pdl_active = on; if (tc) tc->pdl = on; }
    // "Light" PDL: above 128 utterances only the small glue kernels (norms, split-K reductions, stop rule, state shifts: a few hundred threads, no
    // TMEM, little shared memory) are launched programmatically. Their early-resident CTAs cost nothing while the previous GEMM drains; the heavy
    // kernels keep plain stream order (with PDL on everything the waiting GEMM / attention CTAs of one stream starve the other: 1.09 ms per step).
    bool pdl_light = false, pdl_light_allowed = getenv("PTTS_B200_PDL_LIGHT") ? atoi(getenv("PTTS_B200_PDL_LIGHT")) != 0 : true;
    bool pdl_l() const { return pdl_active || pdl_light; }
    long long launches = 0;
    uint64_t seed = 0; unsigned long long* d_seed = nullptr;
    // CUDA graphs of the per-frame step, keyed by (kind, slot0, n, injected); first use runs eagerly (warm-up), second captures
    struct GraphEntry { cudaGraphExec_t exec = nullptr; int seen = 0; long long nlaunch = 0; unsigned long long last_use = 0; };
    std::map<std::tuple<int, int, int, int, int>, GraphEntry> graphs;
    // The cache is keyed by the batch range, so a server that varies (slot0, n) would otherwise grow it without bound: least-recently
    // used entries are evicted beyond graph_cache_cap (26 graphs per range and noise mode; callers should use few distinct ranges).
    size_t graph_cache_cap = getenv("PTTS_B200_GRAPH_CACHE") ? (size_t)atoi(getenv("PTTS_B200_GRAPH_CACHE")) : 512;
    unsigned long long graph_clock = 0;
    void evict_graphs() {
        while (graphs.size() > graph_cache_cap) {
            auto victim = graphs.end();
            for (auto it = graphs.begin(); it != graphs.end(); ++it) if (victim == graphs.end() || it->second.last_use < victim->second.last_use) victim = it;
            if (victim == graphs.end()) return;
            if (victim->second.exec) {
                // a graph launch still in flight keeps its resources alive (cudaGraphExecDestroy defers the release)
                PTTS_CUDA_CHECK(cudaGraphExecDestroy(victim->second.exec));
            }
            graphs.erase(victim);
        }
    }
    int n_voices = 0;
    std::vector<int> voice_len;
    int total_slots = 0;       // max_slots + max_voices (voice prefixes live in the extra KV slots)
    int max_rows = 0;          // scratch rows for the FlowLM forward (decode: slots, prefill: chunk rows)
    int n_embed = 0;

    // ---- weights ----
    __nv_bfloat16* embed = nullptr;
    float *emb_std = nullptr, *emb_mean = nullptr;
    std::vector<float> h_bos; float* d_bos = nullptr;
    LinW input_linear, cond_embed, input_proj, ada_all, final_lin;
    __nv_bfloat16 *input_linear_t = nullptr, *input_proj_t = nullptr;   // [32][out] transposed copies for the fused decode-entry kernels
    float *onw = nullptr, *onb = nullptr; __nv_bfloat16* w_eos = nullptr; float* b_eos = nullptr;
    struct { LinW in_proj, out_proj, lin1, lin2; float *n1w, *n1b, *n2w, *n2b; } fl[N_LAYERS];
    struct { float *lnw, *lnb; LinW mlp0, mlp2; } rb[N_RES];
    float *fnw = nullptr, *fnb = nullptr, *t_combined = nullptr;
    __half* wq = nullptr; float *wup = nullptr, *bup = nullptr;
    struct { LinW in_proj, out_proj, lin1, lin2; float *n1w, *n1b, *n2w, *n2b, *ls1, *ls2; } ml[M_LAYERS];
    ConvW c0, t2, r3a, r3b, t5, r6a, r6b, t8, r9a, r9b, c11;
    float *freq_flow = nullptr, *freq_mimi = nullptr;

    // ---- per-slot state ----
    void *kc = nullptr, *vc = nullptr;                 // FlowLM KV [layer][total_slots][cap][1024]
    long long kv_slot_stride = 0, kv_layer_stride = 0; // elements
    __nv_bfloat16 *mkc = nullptr, *mvc = nullptr;      // Mimi ring [layer][max_slots][250][512]
    long long mkv_slot_stride = 0, mkv_layer_stride = 0;
    int *cur_len = nullptr, *mimi_off = nullptr, *gen_step = nullptr, *eos_step = nullptr, *max_gen = nullptr, *fae = nullptr, *active = nullptr;
    float* temp = nullptr; unsigned int* rng_id = nullptr;   // per-slot sampling temperature, RNG stream id of the sentence in the slot
    __nv_bfloat16* lat_in_bf16 = nullptr; float* lat_f32 = nullptr;   // [slot][32] backbone input / last latent
    float* e_prev = nullptr;                                          // upsampler state [slot][512]
    std::vector<int> h_cur_len;                                       // host mirror of cur_len

    // ---- scratch ----
    float *h = nullptr, *q = nullptr; __nv_bfloat16 *n_bf = nullptr, *att_bf = nullptr, *ff_bf = nullptr;
    int *row_slot = nullptr, *row_pos = nullptr, *tok = nullptr; float2* cs = nullptr;
    float *af_ml = nullptr, *af_acc = nullptr;   // split-KV attention workspace [rows][splits][32] / [rows][splits][1024]
    int* af_cnt = nullptr;                       // per-row arrival counters of the in-kernel split merge (zero between launches)
    int* af_cnt2 = nullptr;                      // per (row, head) arrival counters of the counted merge (streaming + tile kernel side by side)
    // ---- shared voice prefix (cfg.prefix_share): per-slot {slot holding the prefix rows, number of prefix rows}; 0 rows = private cache ----
    int *pfx_slot = nullptr, *pfx_len = nullptr; std::vector<int> h_pfx_slot, h_pfx_len;
    unsigned long long pfx_version = 1;          // bumped whenever a slot's prefix assignment changes
    // decode-side work list of attn_tile_kernel (prefix x rows of a voice), rebuilt when the stepped range or the assignment changes
    AtItem* dec_items = nullptr; int* dec_meta = nullptr; int* dec_rows = nullptr; int dec_items_cap = 0;
    int dec_key_slot0 = -1, dec_key_n = -1; unsigned long long dec_key_version = 0; int dec_grid_items = 0;
    int tile_prec = getenv("PTTS_B200_TILE_PREC") ? atoi(getenv("PTTS_B200_TILE_PREC")) : 1;   // operand precision of the decode-side tile kernel (see attn_tile_kernel): q as
    // hi + lo (the scores go through exp), plain bf16 probabilities; measured on the bench context 2 -> 1 -> 0: 1.084 / 1.067 / 1.054 ms per step,
    // latent max-abs 0.020 / 0.018 / 0.020 and SNR 44.9 / 46.4 / 45.4 dB against the CPU restatement (no measurable parity difference)
    int prefill_prec = getenv("PTTS_B200_PREFILL_PREC") ? atoi(getenv("PTTS_B200_PREFILL_PREC")) : 2;   // operand precision of the prefill tiles (same scale)
    int tile_min_rows = getenv("PTTS_B200_TILE_MIN_ROWS") ? atoi(getenv("PTTS_B200_TILE_MIN_ROWS")) : 4;   // below: the streaming kernel reads the prefix itself
    // attention context of the forward being enqueued (decode: the fixed scratch arrays; prefill: this call's staging)
    struct AttnCtx { const int* row_slot = nullptr; const int* row_pos = nullptr; const float2* cs = nullptr;
                     const AtItem* items = nullptr; const int* meta = nullptr; int n_items = 0; bool prefill = false; } actx;
    // prefill staging on the device (grown on demand): [slot | pos | token] per row, tile items + meta per chunk, voice rows
    int* pf_int = nullptr; size_t pf_int_cap = 0; AtItem* pf_items = nullptr; size_t pf_items_cap = 0; int* pf_meta = nullptr; size_t pf_meta_cap = 0;
    float* pf_x = nullptr; size_t pf_x_cap = 0;
    __nv_bfloat16 *c_bf = nullptr, *sy_bf = nullptr, *hn_bf = nullptr, *h1_bf = nullptr;
    float *eos = nullptr, *ycond = nullptr, *mod = nullptr, *xh = nullptr, *noise_f32 = nullptr, *noise_inj = nullptr, *latent = nullptr;
    int* produced = nullptr; float* eos_out = nullptr;
    // Mimi
    float* mx = nullptr; float* mx2[2] = {nullptr, nullptr}; __nv_bfloat16 *mn_bf = nullptr, *mq_bf = nullptr, *matt_bf = nullptr, *mff_bf = nullptr;
    int *mrow_slot = nullptr, *mrow_pos = nullptr; float2* mcs = nullptr;
    __half *buf0 = nullptr, *buf2 = nullptr, *buf3a = nullptr, *buf3b = nullptr, *buf5 = nullptr, *buf6a = nullptr, *buf6b = nullptr,
           *buf8 = nullptr, *buf9a = nullptr, *buf9b = nullptr, *buf11 = nullptr;
    float *y3 = nullptr, *y6 = nullptr, *y9 = nullptr, *pcm = nullptr;
    // b200_submit frames decode into pcm_alt[frame parity] so that the copy of frame t can run while frame t+1 is decoded; every other path
    // (b200_step, b200_step_enqueue + b200_device_ptr("pcm"), b200_mimi_decode) writes `pcm`. pcm_out = the buffer the enqueued decode writes.
    float* pcm_alt[2] = {nullptr, nullptr}; float* pcm_out = nullptr;
    // Same idea for the injected noise of b200_submit: uploaded on the copy stream into noise_alt[frame parity] (ahead of the step, not between two
    // graph launches of the main stream); noise_src = the buffer the enqueued step reads.
    float* noise_alt[2] = {nullptr, nullptr}; float* noise_src = nullptr; cudaEvent_t ev_noise[2] = {nullptr, nullptr};
    cudaEvent_t ev_dec[2] = {nullptr, nullptr}, ev_copy[2] = {nullptr, nullptr}; bool ev_copy_valid[2] = {false, false}; int last_copy_par = -1;
    float* dtail = nullptr;   // [slot][2 + 1920][4] per-row tap products of the output conv (seanet_tail.cuh), two carried rows in front
    bool fused_tail_allowed = getenv("PTTS_B200_FUSED_TAIL") ? atoi(getenv("PTTS_B200_FUSED_TAIL")) != 0 : true;   // tuning hook
    // The tap "seanet.res9" reads the f16 a3 rows, which only the unfused launches produce. (Switching taps in the middle of a sentence leaves a
    // stale two-row output-conv state for one frame: the two paths carry it in different buffers. Debug only.)
    // Off by default: correct (82-84 dB against the unfused launches, state handling unchanged) but SLOWER, Mimi decode 0.484 -> 0.494 ms at batch
    // 256: at this stage the 64-channel intermediate (31 MB) and the skip tensor stay in L2 between the two tcgen05 GEMMs, so fusing them saves
    // no HBM traffic and trades tcgen05 for mma.sync. (Stage 3, where the tensors are 4x larger than L2 can hold, is where seanet_tail.cuh pays.)
    bool fused_res6_allowed = getenv("PTTS_B200_FUSED_RES6") ? atoi(getenv("PTTS_B200_FUSED_RES6")) != 0 : false;
    bool use_fused_res6() const { return fused_res6_allowed && cfg.gemm_path == 0 && !cfg.convt_split; }
    int tail_ipw = getenv("PTTS_B200_TAIL_IPW") ? atoi(getenv("PTTS_B200_TAIL_IPW")) : 0;   // tuning hook: work items per warp of seanet_tail_kernel (0 = persistent)
    int tail_ctas_per_sm = getenv("PTTS_B200_TAIL_CTAS") ? atoi(getenv("PTTS_B200_TAIL_CTAS")) : 2;   // tuning hook: persistent CTAs per SM of seanet_tail_kernel
    bool use_fused_tail() const { return fused_tail_allowed && cfg.gemm_path == 0 && !taps_on; }
    int C2 = 512, C5 = 256, C8 = 128;
    ShiftAll shifts{};
    // pinned staging
    float* pin_f = nullptr; int* pin_i = nullptr; size_t pin_f_n = 0, pin_i_n = 0;
    // ring of pinned staging buffers for ASYNCHRONOUS uploads (sentence start, prefill, work lists): a buffer is reused only after the
    // event recorded behind its last copy has completed (normally long ago), so no entry point has to synchronise the stream
    struct PinSlot { void* p = nullptr; size_t cap = 0; cudaEvent_t ev = nullptr; bool used = false; } pins[8];
    int pin_next = 0; PinSlot* pin_cur = nullptr;
    void* pin_acquire(size_t bytes) {
        PinSlot& ps = pins[pin_next]; pin_next = (pin_next + 1) % 8;
        if (!ps.ev) PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&ps.ev, cudaEventDisableTiming));
        if (ps.used) PTTS_CUDA_CHECK(cudaEventSynchronize(ps.ev));
        if (ps.cap < bytes) { if (ps.p) cudaFreeHost(ps.p); PTTS_CUDA_CHECK(cudaMallocHost(&ps.p, std::max<size_t>(bytes, 4096))); ps.cap = std::max<size_t>(bytes, 4096); }
        pin_cur = &ps; return ps.p;
    }
    void pin_release(cudaStream_t st) { PTTS_CUDA_CHECK(cudaEventRecord(pin_cur->ev, st)); pin_cur->used = true; }
    template <typename T> void grow(T*& ptr, size_t& cap, size_t need) {     // device scratch that only ever grows (old buffer stays in `allocs`)
        if (need <= cap) return;
        cap = std::max(need, cap * 2); ptr = dalloc<T>(cap, false);
    }
    bool begin_used = false;
    int* begin_meta = nullptr; float* begin_temp = nullptr; size_t begin_cap = 0;   // device copy of b200_begin_sentences' per-sentence metadata
    int* end_slots = nullptr; size_t end_slots_cap = 0;                             // device copy of b200_end_sentences' slot list
    // b200_submit / b200_collect: up to three frames in flight, a ring of four pinned staging sets
    struct Pending { float* noise = nullptr; float* pcm = nullptr; int* produced = nullptr; size_t cap = 0; int slot0 = 0, n = 0; bool busy = false;
                     cudaEvent_t done_main = nullptr, done_mimi = nullptr; } pend[4];
    unsigned long long submit_t = 0, collect_t = 0;
    TcPlanCache* tc = nullptr;
    // optional per-segment device timing (bench.py roofline leg): event pairs recorded on the engine stream
    bool profiling = false;
    struct Seg { int cat; cudaEvent_t a, b; };
    std::vector<Seg> segs; std::vector<cudaEvent_t> ev_pool; size_t ev_used = 0;
    cudaEvent_t next_event() {
        if (ev_used == ev_pool.size()) { cudaEvent_t ev; PTTS_CUDA_CHECK(cudaEventCreate(&ev)); ev_pool.push_back(ev); }
        return ev_pool[ev_used++];
    }
    int seg_begin(int cat, cudaStream_t st = nullptr) {
        if (!profiling) return -1;
        Seg sg; sg.cat = cat; sg.a = next_event(); sg.b = next_event();
        PTTS_CUDA_CHECK(cudaEventRecord(sg.a, st ? st : stream));
        segs.push_back(sg); return (int)segs.size() - 1;
    }
    void seg_end(int id, cudaStream_t st = nullptr) { if (id >= 0) PTTS_CUDA_CHECK(cudaEventRecord(segs[id].b, st ? st : stream)); }

    template <typename T> T* dalloc(size_t n, bool zero = true) {
        void* p = nullptr;
        PTTS_CUDA_CHECK(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
        if (zero) PTTS_CUDA_CHECK(cudaMemsetAsync(p, 0, std::max<size_t>(n, 1) * sizeof(T), stream));
        allocs.push_back(p);
        return (T*)p;
    }
    template <typename T> T* upload(const std::vector<T>& v) {
        T* p = dalloc<T>(v.size(), false);
        PTTS_CUDA_CHECK(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
        return p;
    }
    const HostTensor* find(const std::string& k, bool required = true) {
        auto it = host.find(k);
        if (it == host.end()) {
            if (required) { fprintf(stderr, "ptts_b200: error: missing tensor %s\n", k.c_str()); exit(1); }
            return nullptr;
        }
        return &it->second;
    }
    float* up_f32(const std::string& k, bool required = true) {
        auto* t = find(k, required);
        return t ? upload(t->f) : nullptr;
    }
    static std::vector<__nv_bfloat16> to_bf16(const std::vector<float>& v) {
        std::vector<__nv_bfloat16> o(v.size());
        for (size_t i = 0; i < v.size(); i++) o[i] = __float2bfloat16_rn(v[i]);
        return o;
    }
    LinW up_lin(const std::string& p, int out, int in) {
        auto* w = find(p + ".weight");
        if ((int64_t)w->f.size() != (int64_t)out * in) { fprintf(stderr, "ptts_b200: error: bad shape for %s\n", p.c_str()); exit(1); }
        LinW L; L.out = out; L.in = in;
        const auto wb = to_bf16(w->f);
        L.w = upload(wb);
        if (in % 64 == 0) L.wk = upload(tc_kblock_major(wb, out, in));
        L.b = up_f32(p + ".bias", false);
        return L;
    }
    // causal conv (torch [co][ci][k]) -> f16 [co][k*ci]  (loader policy: ggml_conv_1d weights F16, src/loader.h:209)
    // ci_pad > ci zero-pads the input-channel axis (the activation buffer is padded likewise) so that K % 64 == 0.
    ConvW up_conv(const std::string& p, int co, int ci, int k, int ci_pad = 0) {
        auto* w = find(p + ".conv.weight");
        const int cp = ci_pad > ci ? ci_pad : ci;
        std::vector<__half> o((size_t)co * k * cp, __float2half_rn(0.f));
        for (int a = 0; a < co; a++) for (int b = 0; b < ci; b++) for (int c = 0; c < k; c++)
            o[((size_t)a * k + c) * cp + b] = __float2half_rn(w->f[((size_t)a * ci + b) * k + c]);
        ConvW C; C.N = co; C.K = k * cp; C.w = upload(o); C.b = up_f32(p + ".conv.bias", false);
        if (C.K % 64 == 0) C.wk = upload(tc_kblock_major(o, C.N, C.K));
        return C;
    }
    // transposed conv K = 2s (torch [ci][co][k]) as a 2-tap GEMM over [prev row | current row]:
    //   out[t*s + j][co] = x[t-1] . W[:, co, j+s] + x[t] . W[:, co, j]     (see DESIGN.md "transposed convs")
    // row width Cc = ci (plain f16 activations) or 2*ci (hi | lo split).
    ConvW up_convt(const std::string& p, int ci, int co, int k, int s, int Cc) {
        auto* w = find(p + ".convtr.weight");
        const int N = s * co, Kw = 2 * Cc;
        std::vector<__half> o((size_t)N * Kw);
        for (int j = 0; j < s; j++) for (int c = 0; c < co; c++) for (int kk = 0; kk < Kw; kk++) {
            const bool cur = kk >= Cc; const int cin = (kk % Cc) % ci; const int tap = cur ? j : j + s;
            o[((size_t)(j * co + c)) * Kw + kk] = __float2half_rn(w->f[((size_t)cin * co + c) * k + tap]);
        }
        ConvW C; C.N = N; C.K = Kw; C.w = upload(o);
        if (Kw % 64 == 0) C.wk = upload(tc_kblock_major(o, N, Kw));
        auto* b = find(p + ".convtr.bias", false);
        if (b) { std::vector<float> bb(N); for (int j = 0; j < s; j++) for (int c = 0; c < co; c++) bb[j * co + c] = b->f[c]; C.b = upload(bb); }
        return C;
    }

    // ---------------------------------------------------------------------------------------------
    // Returns true when the LayerNorm described by `ln` was fused into the GEMM's split-K reduction.
    template <typename T>
    bool gemm(const T* A, RowMap amap, int a_rps, const T* W, const T* Wk, int R, int N, int K, const Epi& epi, const LnFuse* ln = nullptr) {
        if (R <= 0) return false;
        if (cfg.gemm_path == 0 && Wk && tc_gemm_supported<T>(R, N, K, amap, a_rps, epi)) {
            bool done = false;
            launches += tc_gemm_launch<T>(tc, A, amap, a_rps, Wk, R, N, K, epi, stream, ln, &done);
            return done;
        }
        if (R <= 8) {
            const int warps = (N + 1) / 2, blocks = (warps + 7) / 8;
            launch_k(pdl_active, gemv_small_kernel<T, 8>, dim3(blocks), dim3(256), (size_t)(0), stream, A, amap, a_rps, W, R, N, K, epi);
        } else {
            dim3 grid((N + 63) / 64, (R + 63) / 64);
            launch_k(pdl_active, gemm_ffma_kernel<T>, dim3(grid), dim3(256), (size_t)(0), stream, A, amap, a_rps, W, R, N, K, epi);
        }
        launches++;
        return false;
    }
    static RowMap rows(long long ld) { RowMap m; m.row_stride = ld; return m; }
    static RowMap smap(long long slot_stride, long long row_stride, long long base) { RowMap m; m.slot_stride = slot_stride; m.row_stride = row_stride; m.base = base; return m; }
    bool lin(const __nv_bfloat16* A, const LinW& L, int R, Epi epi, const LnFuse* ln = nullptr) {
        if (!epi.bias) epi.bias = L.b;
        return gemm<__nv_bfloat16>(A, rows(L.in), 1 << 30, L.w, L.wk, R, L.out, L.in, epi, ln);
    }

    // FlowLM transformer over R rows held in `h` (reference modules/transformer.h:253-278,363-374).
    // Batch 1-2 decode: LayerNorm fused into the GEMV that consumes it (gemv_ln_kernel); x = f32 rows [R][L.in].
    bool ln_in_gemv(int R) const { return R <= 2 && cfg.gemm_path == 0; }
    void lin_ln(const float* x, const LnArgs& ln, const LinW& L, int R, Epi epi) {
        if (!epi.bias) epi.bias = L.b;
        const int blocks = (L.out / 2 + 7) / 8;
        if (L.in == D_MODEL) launch_k(pdl_active, gemv_ln_kernel<D_MODEL>, dim3(blocks), dim3(256), (size_t)0, stream, x, ln, (const __nv_bfloat16*)L.w, R, L.out, epi);
        else launch_k(pdl_active, gemv_ln_kernel<D_FLOW>, dim3(blocks), dim3(256), (size_t)0, stream, x, ln, (const __nv_bfloat16*)L.w, R, L.out, epi);
        launches++;
    }

    // ---- FlowLM transformer over R rows held in `h` (reference modules/transformer.h:253-278,363-374), in two pieces per layer so that the
    //      decode step can be cut into segments at the end of every attention kernel (run_step) ----
    // ---- tap points (parity localisation; the reference's GraphContext::debug, src/context.h:526-547, printed tensor sums) ----
    // b200_debug_taps(1): steps run eagerly on one stream and the FlowLM residual stream / attention output of every layer are copied
    // aside; the Mimi-side taps are persistent buffers that can be read after any step (b200_debug_tap).
    bool taps_on = false; float* tap_h = nullptr; __nv_bfloat16* tap_att = nullptr; float* tap_up = nullptr; int tap_slot0 = 0, tap_n = 0;
    void tap_flow_layer(int l, int R) {
        if (!taps_on || actx.prefill) return;
        PTTS_CUDA_CHECK(cudaMemcpyAsync(tap_h + (size_t)l * cfg.max_slots * D_MODEL, h, (size_t)R * D_MODEL * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    }
    void tap_flow_attn(int l, int R) {
        if (!taps_on || actx.prefill) return;
        PTTS_CUDA_CHECK(cudaMemcpyAsync(tap_att + (size_t)l * cfg.max_slots * D_MODEL, att_bf, (size_t)R * D_MODEL * sizeof(__nv_bfloat16), cudaMemcpyDeviceToDevice, stream));
    }

    // Decode rows of the range [slot0, slot0+n): row r = slot slot0+r. With a shared voice prefix, (re)builds the work list of
    // attn_tile_kernel (plan_prefix_tiles) on the host when the range or the slot -> voice assignment changed. Stream-ordered upload.
    void prepare_decode(int slot0, int n) {
        actx = AttnCtx{}; actx.row_slot = row_slot; actx.row_pos = row_pos; actx.cs = cs;
        if (!cfg.prefix_share || cfg.kv_f32 || n < tile_min_rows) { dec_grid_items = 0; dec_key_n = -1; return; }
        if (dec_key_slot0 == slot0 && dec_key_n == n && dec_key_version == pfx_version) return;
        dec_key_slot0 = slot0; dec_key_n = n; dec_key_version = pfx_version;
        std::vector<AtItem> items; std::vector<int> rows;
        const int splits = plan_prefix_tiles(h_pfx_slot.data() + slot0, h_pfx_len.data() + slot0, n, tc ? tc->num_sms : 148, items, rows);
        if (splits == 0) { dec_grid_items = 0; return; }
        if ((int)items.size() > dec_items_cap) { fprintf(stderr, "ptts_b200: internal error: %zu prefix tiles exceed the work-list capacity %d\n", items.size(), dec_items_cap); abort(); }
        dec_grid_items = ((int)items.size() + 7) / 8 * 8;
        const size_t bytes = 4 * sizeof(int) + rows.size() * sizeof(int) + items.size() * sizeof(AtItem);
        char* pb = (char*)pin_acquire(bytes + 64);
        int* meta = (int*)pb; meta[0] = (int)items.size(); meta[1] = splits; meta[2] = 0; meta[3] = 0;
        int* prow = meta + 4; memcpy(prow, rows.data(), rows.size() * sizeof(int));
        char* pit = (char*)(prow + rows.size()); memcpy(pit, items.data(), items.size() * sizeof(AtItem));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(dec_meta, meta, 4 * sizeof(int), cudaMemcpyHostToDevice, stream));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(dec_rows, prow, rows.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(dec_items, pit, items.size() * sizeof(AtItem), cudaMemcpyHostToDevice, stream));
        pin_release(stream);
    }

    // Number of KV splits of the streaming attention kernel for R rows. The CTA total should come close to whole waves of the resident
    // CTAs (bf16: two 96 KB CTAs per SM) with at least ~2 CTAs per SM in flight (R = 256 rows streaming ~1.5k keys each: 3 splits =
    // 5.19 waves, the last wave streams on 28 SMs; 4 splits = 6.92 waves, measured 1.557 -> 1.467 ms per step for the six launches).
    // When the shared prefix is reduced by attn_tile_kernel the streamed part is only the utterance's own rows (a few hundred keys):
    // two CTAs per SM are enough, more splits would only add per-CTA prologue/merge cost.
    int af_splits(int R, bool short_stream) const {
        if (af_splits_override > 0) return std::min(af_splits_override, AF_MAX_SPLITS);
        const int sms = tc ? tc->num_sms : 148;
        if (short_stream) return std::max(1, std::min(AF_MAX_SPLITS, (sms + R - 1) / R));   // ~one CTA per SM: the tile kernel runs beside it (measured 1.095 -> 1.084 ms at R = 256)
        int splits = 1; double best = -1.0;
        for (int sp = 1; sp <= AF_MAX_SPLITS; sp++) {
            const long long ctas = (long long)R * sp;
            if (ctas < 2LL * sms && sp < AF_MAX_SPLITS) continue;
            const double waves = (double)ctas / sms, eff = waves / std::ceil(waves);
            if (eff > best + 1e-9) { best = eff; splits = sp; }
            if (ctas >= 8LL * sms) break;
        }
        return splits;
    }
    template <typename... A> void launch_tiles(int prec, bool pdl, dim3 grid, cudaStream_t st, A... a) {
        if (prec >= 2) launch_k(pdl, attn_tile_kernel<2>, grid, dim3(128), (size_t)0, st, a...);
        else if (prec == 1) launch_k(pdl, attn_tile_kernel<1>, grid, dim3(128), (size_t)0, st, a...);
        else launch_k(pdl, attn_tile_kernel<0>, grid, dim3(128), (size_t)0, st, a...);
    }
    // prefill chunk c (its rows start at row r0 of the `total` rows staged in pf_int; items from chunk_item0) becomes the attention context
    void prefill_chunk(int c, int r0, int total, const std::vector<int>& chunk_item0) {
        actx = AttnCtx{};
        actx.row_slot = pf_int + r0; actx.row_pos = pf_int + total + r0; actx.cs = cs; actx.prefill = true;
        actx.items = pf_items + chunk_item0[c]; actx.meta = pf_meta + 4 * c; actx.n_items = chunk_item0[c + 1] - chunk_item0[c];
    }
    bool use_prefix_tiles(int R) const { return cfg.prefix_share && !cfg.kv_f32 && !actx.prefill && R >= tile_min_rows && dec_grid_items > 0; }

    // in_proj (+RoPE, KV append) and attention of layer l. Expects norm1 of layer l in n_bf; rows are described by `actx`.
    void flow_attn_part(int l, int R) { flow_qkv(l, R); flow_attn(l, R); }
    Epi qkv_epi(int l) const {
        Epi e; e.mode = EPI_FLOW_QKV; e.row_slot = actx.row_slot; e.row_pos = actx.row_pos; e.cs = actx.cs; e.kv_f32 = cfg.kv_f32;
        e.kv_slot_stride = kv_slot_stride; e.q_out_f32 = q;
        if (cfg.kv_f32) { e.kcache = (float*)kc + l * kv_layer_stride; e.vcache = (float*)vc + l * kv_layer_stride; }
        else { e.kcache = (__nv_bfloat16*)kc + l * kv_layer_stride; e.vcache = (__nv_bfloat16*)vc + l * kv_layer_stride; }
        return e;
    }
    // in_proj of layer l: q -> `q` (f32), K/V rows appended to the cache at (row_slot, row_pos)
    void flow_qkv(int l, int R) {
        auto& L = fl[l];
        const Epi e = qkv_epi(l);
        if (l > 0 && ln_in_gemv(R)) { LnArgs a; a.w = L.n1w; a.b = L.n1b; a.eps = 1e-5f; lin_ln(h, a, L.in_proj, R, e); }   // layer 0: flow_in_kernel wrote n_bf
        else lin(n_bf, L.in_proj, R, e);
    }
    // attention of layer l over the rows of `actx` (q in `q`, keys in the cache) -> att_bf: picks the kernels (prefill tiles, shared-prefix
    // tiles beside the streaming kernel, streaming alone) and the merge, and launches them
    void flow_attn(int l, int R) {
        const Epi e = qkv_epi(l);
        int sg = -1;
        const bool pdl_saved = pdl_active;
        set_pdl(pdl_small);                                  // the KV-streaming kernel fills the machine: no early dependents around it
        if (actx.prefill && !cfg.kv_f32) {
            // T > 1 rows with the causal mask (reference transformer.h:157-169): one tensor-core tile per 64 rows of a slot and head, K/V read
            // once per tile instead of once per row
            if (actx.n_items > 0)
                launch_tiles(prefill_prec, pdl_active, dim3(actx.n_items, N_HEADS), stream, (const float*)q, (const __nv_bfloat16*)e.kcache,
                             (const __nv_bfloat16*)e.vcache, kv_slot_stride, actx.items, actx.meta, (const int*)nullptr, actx.row_pos, af_ml, af_acc, att_bf, (const int*)nullptr, (int*)nullptr, 0);
            launches++;
        } else {
            const bool tiles = use_prefix_tiles(R);
            const bool fork = tiles && fork_tiles;      // tile kernel (tensor cores, prefix from L2) beside the streaming kernel (HBM), merged afterwards
            const bool counted = fork && counted_merge;  // both kernels count per (row, head); the last arriver merges: no merge launch
            const int splits = af_splits(R, tiles);
            AfKeys keys; keys.pfx_slot = pfx_slot; keys.pfx_len = pfx_len; keys.tiles_meta = tiles ? dec_meta : nullptr; keys.defer_merge = fork ? (counted ? 2 : 1) : 0;
            keys.merge_cnt2 = af_cnt2;
            if (tiles) {   // shared voice prefix x all rows of the voice -> workspace partials
                cudaStream_t ts = stream;
                if (fork) {
                    PTTS_CUDA_CHECK(cudaEventRecord(ev_fork, stream));
                    PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream_t, ev_fork, 0));
                    ts = stream_t;
                }
                const int sgt = seg_begin(6, ts);
                launch_tiles(tile_prec, fork ? false : pdl_active, dim3(dec_grid_items, N_HEADS), ts, (const float*)q, (const __nv_bfloat16*)e.kcache,
                             (const __nv_bfloat16*)e.vcache, kv_slot_stride, (const AtItem*)dec_items, (const int*)dec_meta, (const int*)dec_rows, actx.row_pos, af_ml, af_acc, att_bf,
                             actx.row_slot, counted ? af_cnt2 : (int*)nullptr, splits);
                launches++;
                seg_end(sgt, ts);
                if (fork) PTTS_CUDA_CHECK(cudaEventRecord(ev_join, stream_t));
            }
            sg = seg_begin(0);
            if (cfg.kv_f32)
                launch_k(pdl_active, attn_flow_split_kernel<float>, dim3(splits, R), dim3(288), (size_t)(AfCfg<float>::SMEM), stream, (const float*)q, (const float*)e.kcache, (const float*)e.vcache,
                         kv_slot_stride, actx.row_slot, actx.row_pos, keys, splits, af_ml, af_acc, att_bf, af_cnt);
            else
                launch_k(pdl_active, attn_flow_split_kernel<__nv_bfloat16>, dim3(splits, R), dim3(288), (size_t)(AfCfg<__nv_bfloat16>::SMEM), stream, (const float*)q, (const __nv_bfloat16*)e.kcache,
                         (const __nv_bfloat16*)e.vcache, kv_slot_stride, actx.row_slot, actx.row_pos, keys, splits, af_ml, af_acc, att_bf, af_cnt);
            launches++;
            if (fork) {
                seg_end(sg); sg = -1;
                PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_join, 0));
                if (!counted) launch_k(false, attn_merge_kernel, dim3(R), dim3(256), (size_t)0, stream, actx.row_slot, (const int*)pfx_len, (const int*)dec_meta, splits, (const float*)af_ml, (const float*)af_acc, att_bf);
                if (!counted) launches++;
            }
        }
        set_pdl(pdl_saved);
        seg_end(sg);
        tap_flow_attn(l, R);
    }
    // out_proj (+residual, norm2), linear1 (+GELU), linear2 (+residual) of layer l; leaves norm1 of layer l+1 in n_bf.
    void flow_chain_part(int l, int R) {
        const int BIG = 1 << 30;
        auto& L = fl[l];
        Epi eo; eo.resid = h; eo.resid_map = rows(D_MODEL); eo.out = h; eo.out_map = rows(D_MODEL);
        LnFuse f2; f2.w = L.n2w; f2.b = L.n2b; f2.eps = 1e-5f; f2.out = n_bf;
        const bool fuse = ln_in_gemv(R);
        if (!lin(att_bf, L.out_proj, R, eo, &f2) && !fuse) {
            launch_k(pdl_l(), layernorm_kernel<D_MODEL>, dim3(R), dim3(D_MODEL / 4), (size_t)(0), stream, h, rows(D_MODEL), BIG, R, 1e-5f, L.n2w, L.n2b, nullptr, nullptr, 0, n_bf, nullptr); launches++;
        }
        Epi e1; e1.out2 = ff_bf; e1.out2_map = rows(D_FF); e1.out2_type = OUT2_BF16; e1.act = ACT_GELU;
        if (fuse) { LnArgs a; a.w = L.n2w; a.b = L.n2b; a.eps = 1e-5f; lin_ln(h, a, L.lin1, R, e1); }
        else lin(n_bf, L.lin1, R, e1);
        Epi e2; e2.resid = h; e2.resid_map = rows(D_MODEL); e2.out = h; e2.out_map = rows(D_MODEL);
        if (l + 1 < N_LAYERS) {
            LnFuse f1; f1.w = fl[l + 1].n1w; f1.b = fl[l + 1].n1b; f1.eps = 1e-5f; f1.out = n_bf;
            if (!lin(ff_bf, L.lin2, R, e2, &f1) && !fuse) {    // fused: the next in_proj normalises h itself (flow_attn_part)
                launch_k(pdl_l(), layernorm_kernel<D_MODEL>, dim3(R), dim3(D_MODEL / 4), (size_t)(0), stream, h, rows(D_MODEL), BIG, R, 1e-5f, fl[l + 1].n1w, fl[l + 1].n1b, nullptr, nullptr, 0, n_bf, nullptr); launches++;
            }
        } else {
            lin(ff_bf, L.lin2, R, e2);
        }
        tap_flow_layer(l, R);
    }
    void flow_forward(int R, bool ln1_done = false) {              // ln1_done: layer 0's norm1 already in n_bf (decode: flow_in_kernel)
        const int BIG = 1 << 30;
        if (!ln1_done) { launch_k(pdl_l(), layernorm_kernel<D_MODEL>, dim3(R), dim3(D_MODEL / 4), (size_t)(0), stream, h, rows(D_MODEL), BIG, R, 1e-5f, fl[0].n1w, fl[0].n1b, nullptr, nullptr, 0, n_bf, nullptr); launches++; }
        for (int l = 0; l < N_LAYERS; l++) { flow_attn_part(l, R); flow_chain_part(l, R); }
    }

    bool fused_head_allowed = getenv("PTTS_B200_FUSED_HEAD") ? atoi(getenv("PTTS_B200_FUSED_HEAD")) != 0 : true;   // tuning hook
    int fused_head_min_rows = getenv("PTTS_B200_FUSED_HEAD_MIN") ? atoi(getenv("PTTS_B200_FUSED_HEAD_MIN")) : 3;
    bool use_fused_head(int R) const { return fused_head_allowed && cfg.gemm_path == 0 && !taps_on && R >= fused_head_min_rows; }
    // out_norm + EOS + 1-step LSD head over R rows of `h` (reference models/flow_lm.h:114-142, modules/mlp.h:233-251).
    void flow_head(int R) {
        const int BIG = 1 << 30;
        launch_k(pdl_l(), head_pre_kernel, dim3(R), dim3(256), (size_t)(0), stream, h, R, onw, onb, w_eos, b_eos, c_bf, eos);
        // y = t_combined + cond_embed(c); sy = silu(y)
        Epi ec; ec.resid = t_combined; ec.resid_map = RowMap{}; ec.out2 = sy_bf; ec.out2_map = rows(D_FLOW); ec.out2_type = OUT2_BF16; ec.act = ACT_SILU;
        lin(c_bf, cond_embed, R, ec);
        // all seven adaLN projections of silu(y) in one GEMM: [6 x (shift|scale|gate)] + [shift|scale]
        Epi em; em.out = mod; em.out_map = rows(ada_all.out);
        lin(sy_bf, ada_all, R, em);
        if (use_fused_head(R)) {
            // six residual blocks + final layer in one cluster kernel (head_fused.cuh): activations stay in (distributed) shared memory
            HfParams hp{};
            hp.R = R; hp.xh = xh; hp.mod = mod; hp.mod_ld = ada_all.out;
            for (int r = 0; r < N_RES; r++) hp.rb[r] = {rb[r].lnw, rb[r].lnb, rb[r].mlp0.w, rb[r].mlp0.b, rb[r].mlp2.w, rb[r].mlp2.b};
            hp.fnw = fnw; hp.fnb = fnb; hp.wf = final_lin.w; hp.bf = final_lin.b; hp.noise = noise_f32; hp.latent = latent;
            launch_k(pdl_active, head_res_cluster_kernel, dim3((R + HF_ROWS - 1) / HF_ROWS * HF_CLUSTER), dim3(HF_THREADS), HF_SMEM_BYTES, stream, hp);
            launches += 2;                                   // + head_pre_kernel
            return;
        }
        for (int r = 0; r < N_RES; r++) {
            const float* m = mod + r * 3 * D_FLOW;
            Epi e0; e0.out2 = h1_bf; e0.out2_map = rows(D_FLOW); e0.out2_type = OUT2_BF16; e0.act = ACT_SILU;
            if (ln_in_gemv(R)) { LnArgs a; a.w = rb[r].lnw; a.b = rb[r].lnb; a.eps = 1e-6f; a.shift = m; a.scale = m + D_FLOW; a.mod_ld = ada_all.out; lin_ln(xh, a, rb[r].mlp0, R, e0); }
            else {
                launch_k(pdl_l(), layernorm_kernel<D_FLOW>, dim3(R), dim3(D_FLOW / 4), (size_t)(0), stream, xh, rows(D_FLOW), BIG, R, 1e-6f, rb[r].lnw, rb[r].lnb, m, m + D_FLOW, ada_all.out, hn_bf, nullptr);
                launches++;
                lin(hn_bf, rb[r].mlp0, R, e0);
            }
            Epi e2; e2.rowmul = m + 2 * D_FLOW; e2.rowmul_ld = ada_all.out; e2.resid = xh; e2.resid_map = rows(D_FLOW); e2.out = xh; e2.out_map = rows(D_FLOW);
            lin(h1_bf, rb[r].mlp2, R, e2);
        }
        const float* m = mod + N_RES * 3 * D_FLOW;
        Epi ef; ef.resid = noise_f32; ef.resid_map = rows(LDIM); ef.out = latent; ef.out_map = rows(LDIM);
        if (ln_in_gemv(R)) { LnArgs a; a.w = fnw; a.b = fnb; a.eps = 1e-6f; a.shift = m; a.scale = m + D_FLOW; a.mod_ld = ada_all.out; lin_ln(xh, a, final_lin, R, ef); }
        else {
            launch_k(pdl_l(), layernorm_kernel<D_FLOW>, dim3(R), dim3(D_FLOW / 4), (size_t)(0), stream, xh, rows(D_FLOW), BIG, R, 1e-6f, fnw, fnb, m, m + D_FLOW, ada_all.out, hn_bf, nullptr);
            launches++;
            lin(hn_bf, final_lin, R, ef);
        }
        launches += 1;
    }

    // Mimi front end (latent -> 16 transformer input rows, written to `xbuf`), reference models/mimi.h:77-83 + modules/conv.h:283-331.
    void mimi_front(int slot0, int n, float* xbuf) {
        launch_k(pdl_l(), mimi_front_kernel, dim3(n), dim3(M_DIM), (size_t)(0), stream, slot0, lat_f32, emb_std, emb_mean, wq, wup, bup, e_prev, xbuf);
        launches++;
    }
    // Mimi decoder body for slots [slot0, slot0+n) from the front end's rows in `xbuf` (reference models/mimi.h:85-104).
    // chunk < 0: everything; otherwise one of N_MCHUNK pieces of roughly equal duration (run_step interleaves them with the FlowLM segments)
    static constexpr int N_MCHUNK = 6;
    void mimi_ln(const float* x, int R, const float* w, const float* b) {      // LayerNorm(eps 0) of the Mimi transformer rows -> mn_bf
        const int BIG = 1 << 30;
        if (R >= 512) launch_k(pdl_l(), layernorm_rows_kernel<M_DIM>, dim3((R + 7) / 8), dim3(256), (size_t)0, stream, x, R, 0.0f, w, b, mn_bf);
        else launch_k(pdl_l(), layernorm_kernel<M_DIM>, dim3(R), dim3(M_DIM / 4), (size_t)(0), stream, x, rows(M_DIM), BIG, R, 0.0f, w, b, nullptr, nullptr, 0, mn_bf, nullptr);
    }
    void mimi(int slot0, int n, float* xbuf, int chunk = -1) {
        const int BIG = 1 << 30, R = n * M_T;
        auto on = [&](int c) { return chunk < 0 || chunk == c; };
        if (on(0)) {
            launch_k(pdl_l(), prepare_mimi_kernel, dim3((n * M_T * 32 + 255) / 256), dim3(256), (size_t)(0), stream, slot0, n, (const int*)mimi_off, (const float*)freq_mimi, mrow_slot, mrow_pos, mcs);
            launches++;
        }
        float* x = xbuf + (long long)slot0 * M_T * M_DIM;
        const int s_mtf = chunk < 0 ? seg_begin(3) : -1;
        for (int l = 0; l < M_LAYERS; l++) {
            auto& L = ml[l];
            // layer 0: [LN1 in_proj attn out_proj] = chunk 0, [LN2 lin1 lin2] = chunk 1; layer 1: [LN1 in_proj] = chunk 1, the rest = chunk 2
            const int c_qkv = l == 0 ? 0 : 1, c_att = l == 0 ? 0 : 2, c_mlp = l == 0 ? 1 : 2;
            Epi e; e.mode = EPI_MIMI_QKV; e.row_slot = mrow_slot; e.row_pos = mrow_pos; e.cs = mcs; e.kv_slot_stride = mkv_slot_stride;
            e.kcache = mkc + l * mkv_layer_stride; e.vcache = mvc + l * mkv_layer_stride; e.q_out_bf16 = mq_bf;
            if (on(c_qkv)) {
                mimi_ln(x, R, L.n1w, L.n1b);
                launches++;
                lin(mn_bf, L.in_proj, R, e);
            }
            if (on(c_att)) {
                if (cfg.gemm_path == 0) launch_k(pdl_active, attn_mimi_mma4_kernel, dim3(n * M_HEADS), dim3(128), (size_t)0, stream, (const __nv_bfloat16*)mq_bf, (const __nv_bfloat16*)e.kcache,
                                                 (const __nv_bfloat16*)e.vcache, mkv_slot_stride, slot0, (const int*)mimi_off, cfg.mimi_mask_mode, matt_bf);
                else launch_k(pdl_active, attn_mimi_kernel, dim3(n, M_HEADS), dim3(256), (size_t)(AM_SMEM), stream, mq_bf, (const __nv_bfloat16*)e.kcache, (const __nv_bfloat16*)e.vcache, mkv_slot_stride, slot0, mimi_off, cfg.mimi_mask_mode, matt_bf);
                launches++;
                Epi eo; eo.colscale = L.ls1; eo.resid = x; eo.resid_map = rows(M_DIM); eo.out = x; eo.out_map = rows(M_DIM);
                lin(matt_bf, L.out_proj, R, eo);
            }
            if (on(c_mlp)) {
                mimi_ln(x, R, L.n2w, L.n2b);
                launches++;
                Epi e1; e1.out2 = mff_bf; e1.out2_map = rows(M_FF); e1.out2_type = OUT2_BF16; e1.act = ACT_GELU;
                lin(mn_bf, L.lin1, R, e1);
                Epi e2; e2.colscale = L.ls2; e2.resid = x; e2.resid_map = rows(M_DIM);
                if (l + 1 < M_LAYERS) { e2.out = x; e2.out_map = rows(M_DIM); }
                else {
                    // last layer: the only consumer is SEANet's first conv, so write its f16 input rows (after the 6 carried rows) directly
                    e2.rps = M_T; e2.resid_map = smap((long long)M_T * M_DIM, M_DIM, 0);
                    e2.out2 = buf0 + slot0 * 22LL * 512; e2.out2_map = smap(22LL * 512, 512, 6 * 512); e2.out2_type = OUT2_F16;
                }
                lin(mff_bf, L.lin2, R, e2);
            }
        }
        seg_end(s_mtf);
        const int s_sea = chunk < 0 ? seg_begin(4) : -1;
        // SEANet (reference modules/seanet.h:187-211); every conv is a GEMM over overlapping channel-last rows.
        const int T0 = 16, T1 = 96, T2 = 480, T3 = 1920;
        const long long s0 = 22LL * 512, s2 = 17LL * C2, s3a = 98LL * 256, s3b = 96LL * 128, s5 = 97LL * C5, s6a = 482LL * 128, s6b = 480LL * 64,
                        s8 = 481LL * C8, s9a = 1922LL * 64, s9b = 1920LL * 64, s11 = 1922LL * 64;
        const int o2t = cfg.convt_split ? OUT2_F16_SPLIT : OUT2_F16;
        if (on(3)) { Epi e; e.rps = T0; e.bias = c0.b; e.act = ACT_ELU; e.out2 = buf2 + slot0 * s2; e.out2_map = smap(s2, C2, C2); e.out2_type = o2t; e.split_off = 512;
          gemm<__half>(buf0 + slot0 * s0, smap(s0, 512, 0), T0, c0.w, c0.wk, n * T0, c0.N, c0.K, e); }
        if (on(3)) { Epi e; e.rps = T0; e.bias = t2.b; e.out = y3 + slot0 * 96LL * 256; e.out_map = smap(96LL * 256, 1536, 0);
          e.act = ACT_ELU; e.out2 = buf3a + slot0 * s3a; e.out2_map = smap(s3a, 1536, 2 * 256); e.out2_type = OUT2_F16;
          gemm<__half>(buf2 + slot0 * s2, smap(s2, C2, 0), T0, t2.w, t2.wk, n * T0, t2.N, t2.K, e); }
        if (on(3)) { Epi e; e.rps = T1; e.bias = r3a.b; e.act = ACT_ELU; e.out2 = buf3b + slot0 * s3b; e.out2_map = smap(s3b, 128, 0); e.out2_type = OUT2_F16;
          gemm<__half>(buf3a + slot0 * s3a, smap(s3a, 256, 0), T1, r3a.w, r3a.wk, n * T1, r3a.N, r3a.K, e); }
        if (on(3)) { Epi e; e.rps = T1; e.bias = r3b.b; e.resid = y3 + slot0 * 96LL * 256; e.resid_map = smap(96LL * 256, 256, 0);
          e.act = ACT_ELU; e.out2 = buf5 + slot0 * s5; e.out2_map = smap(s5, C5, C5); e.out2_type = o2t; e.split_off = 256;
          gemm<__half>(buf3b + slot0 * s3b, smap(s3b, 128, 0), T1, r3b.w, r3b.wk, n * T1, r3b.N, r3b.K, e); }
        if (on(4)) { Epi e; e.rps = T1; e.bias = t5.b; e.out = y6 + slot0 * 480LL * 128; e.out_map = smap(480LL * 128, 640, 0);
          e.act = ACT_ELU; e.out2 = buf6a + slot0 * s6a; e.out2_map = smap(s6a, 640, 2 * 128); e.out2_type = OUT2_F16;
          gemm<__half>(buf5 + slot0 * s5, smap(s5, C5, 0), T1, t5.w, t5.wk, n * T1, t5.N, t5.K, e); }
        if (on(4) && use_fused_res6()) {
            // resnet block 6 in one streaming kernel (seanet_res.cuh): no 64-channel intermediate, the result lands in the next transposed conv's input rows
            SrParams sp{};
            sp.a1 = buf6a; sp.a1_slot_stride = s6a; sp.y = y6; sp.y_slot_stride = 480LL * 128; sp.out = buf8; sp.out_slot_stride = s8; sp.out_row0 = 1;
            sp.w3 = r6a.w; sp.b3 = r6a.b; sp.w1 = r6b.w; sp.w1_ld = r6b.K; sp.b1 = r6b.b; sp.slot0 = slot0; sp.n_slots = n; sp.T = T2;
            const long long items = (long long)n * (T2 / SR_ROWS);
            launch_k(pdl_active, seanet_res_kernel, dim3((unsigned)std::min<long long>(tc ? tc->num_sms : 148, (items + SR_WARPS - 1) / SR_WARPS)), dim3(SR_THREADS), SR_SMEM_BYTES, stream, sp);
            launches++;
        } else if (on(4)) {
        { Epi e; e.rps = T2; e.bias = r6a.b; e.act = ACT_ELU; e.out2 = buf6b + slot0 * s6b; e.out2_map = smap(s6b, 64, 0); e.out2_type = OUT2_F16;
          gemm<__half>(buf6a + slot0 * s6a, smap(s6a, 128, 0), T2, r6a.w, r6a.wk, n * T2, r6a.N, r6a.K, e); }
        { Epi e; e.rps = T2; e.bias = r6b.b; e.resid = y6 + slot0 * 480LL * 128; e.resid_map = smap(480LL * 128, 128, 0);
          e.act = ACT_ELU; e.out2 = buf8 + slot0 * s8; e.out2_map = smap(s8, C8, C8); e.out2_type = o2t; e.split_off = 128;
          gemm<__half>(buf6b + slot0 * s6b, smap(s6b, 64, 0), T2, r6b.w, r6b.wk, n * T2, r6b.N, r6b.K, e); }
        }
        if (on(5)) { Epi e; e.rps = T2; e.bias = t8.b; e.out = y9 + slot0 * 1920LL * 64; e.out_map = smap(1920LL * 64, 256, 0);
          e.act = ACT_ELU; e.out2 = buf9a + slot0 * s9a; e.out2_map = smap(s9a, 256, 2 * 64); e.out2_type = OUT2_F16;
          gemm<__half>(buf8 + slot0 * s8, smap(s8, C8, 0), T2, t8.w, t8.wk, n * T2, t8.N, t8.K, e); }
        if (on(5) && use_fused_tail()) {
            // resnet block 9 + output conv in one streaming kernel (seanet_tail.cuh): no padded intermediate, no a3 tensor
            StParams sp{};
            sp.a1 = buf9a; sp.a1_slot_stride = s9a; sp.y = y9; sp.y_slot_stride = 1920LL * 64; sp.d = dtail; sp.d_slot_stride = 1922LL * ST_DROW;
            sp.w3 = r9a.w; sp.b3 = r9a.b; sp.w1 = r9b.w; sp.w1_ld = r9b.K; sp.b1 = r9b.b; sp.w11 = c11.w; sp.slot0 = slot0; sp.n_slots = n; sp.T = T3;
            const long long items = (long long)n * (T3 / ST_ROWS);
            sp.ipw = tail_ipw;
            const int sms = tc ? tc->num_sms : 148;
            const int grid = tail_ipw > 0 ? (int)((items + ST_WARPS * tail_ipw - 1) / (ST_WARPS * tail_ipw)) : (int)std::min<long long>((long long)tail_ctas_per_sm * sms, (items + ST_WARPS - 1) / ST_WARPS);
            launch_k(pdl_active, seanet_tail_kernel, dim3(grid), dim3(ST_THREADS), ST_SMEM_BYTES, stream, sp);
            launch_k(pdl_l(), pcm_combine_kernel, dim3((unsigned)(((long long)n * T3 + 255) / 256)), dim3(256), (size_t)0, stream, (const float*)dtail, 1922LL * ST_DROW, slot0, n, T3,
                     (const float*)c11.b, pcm_out);
            launch_k(pdl_l(), shift_states_kernel, dim3(n, shifts.n), dim3(128), (size_t)(0), stream, shifts, slot0, mimi_off);
            launches += 3;
        } else if (on(5)) {
        { Epi e; e.rps = T3; e.bias = r9a.b; e.act = ACT_ELU; e.out2 = buf9b + slot0 * s9b; e.out2_map = smap(s9b, 64, 0); e.out2_type = OUT2_F16;
          gemm<__half>(buf9a + slot0 * s9a, smap(s9a, 64, 0), T3, r9a.w, r9a.wk, n * T3, r9a.N, r9a.K, e); }
        { Epi e; e.rps = T3; e.bias = r9b.b; e.resid = y9 + slot0 * 1920LL * 64; e.resid_map = smap(1920LL * 64, 64, 0);
          e.act = ACT_ELU; e.out2 = buf11 + slot0 * s11; e.out2_map = smap(s11, 64, 2 * 64); e.out2_type = OUT2_F16;
          gemm<__half>(buf9b + slot0 * s9b, smap(s9b, 64, 0), T3, r9b.w, r9b.wk, n * T3, r9b.N, r9b.K, e); }
            const int Rr = n * T3;
            launch_k(pdl_l(), conv_n1_kernel, dim3((Rr * 4 + 255) / 256), dim3(256), (size_t)(0), stream, buf11 + slot0 * s11, smap(s11, 64, 0), T3, c11.w, c11.b, Rr, c11.K, pcm_out + (long long)slot0 * FRAME);
            launch_k(pdl_l(), shift_states_kernel, dim3(n, shifts.n), dim3(128), (size_t)(0), stream, shifts, slot0, mimi_off);
            launches += 2;
        }
        seg_end(s_sea);
    }

    // ---- batch 1-2: the FlowLM step + head as ONE cooperative kernel (persistent.cuh) instead of ~75 dependent launches ----
    unsigned int* pf_barrier = nullptr;
    bool persistent_allowed = getenv("PTTS_B200_PERSISTENT") ? atoi(getenv("PTTS_B200_PERSISTENT")) != 0 : true;
    bool use_persistent(int n) const {
        return persistent_allowed && n <= PF_RMAX && !cfg.kv_f32 && cfg.gemm_path == 0 && !taps_on && !profiling && cfg.kv_capacity <= 8 * PF_MAX_KEYS;
    }
    void flow_persistent(int slot0, int n, bool injected, float* xbuf) {
        PfParams p{};
        const int sms = tc ? tc->num_sms : 148;
        p.slot0 = slot0; p.R = n;
        p.n_splits = std::min(16, std::max(std::max(1, sms / (n * N_HEADS)), (cfg.kv_capacity + PF_MAX_KEYS - 1) / PF_MAX_KEYS));   // <= 16: merge scratch of the kernel
        p.lat_in = lat_in_bf16; p.cur_len = cur_len; p.active = active; p.freq = freq_flow;
        p.kc = (__nv_bfloat16*)kc; p.vc = (__nv_bfloat16*)vc; p.kv_slot_stride = kv_slot_stride; p.kv_layer_stride = kv_layer_stride;
        p.pfx_slot = pfx_slot; p.pfx_len = pfx_len;
        p.input_linear_t = input_linear_t; p.input_linear_b = input_linear.b;
        for (int l = 0; l < N_LAYERS; l++) {
            p.L[l].in_proj = {fl[l].in_proj.w, fl[l].in_proj.b}; p.L[l].out_proj = {fl[l].out_proj.w, fl[l].out_proj.b};
            p.L[l].lin1 = {fl[l].lin1.w, fl[l].lin1.b}; p.L[l].lin2 = {fl[l].lin2.w, fl[l].lin2.b};
            p.L[l].n1w = fl[l].n1w; p.L[l].n1b = fl[l].n1b; p.L[l].n2w = fl[l].n2w; p.L[l].n2b = fl[l].n2b;
        }
        p.onw = onw; p.onb = onb; p.w_eos = w_eos; p.b_eos = b_eos;
        p.cond = {cond_embed.w, cond_embed.b}; p.ada = {ada_all.w, ada_all.b}; p.fin = {final_lin.w, final_lin.b}; p.ada_out = ada_all.out; p.t_combined = t_combined;
        for (int r = 0; r < N_RES; r++) { p.rb[r].lnw = rb[r].lnw; p.rb[r].lnb = rb[r].lnb; p.rb[r].m0 = {rb[r].mlp0.w, rb[r].mlp0.b}; p.rb[r].m2 = {rb[r].mlp2.w, rb[r].mlp2.b}; }
        p.fnw = fnw; p.fnb = fnb; p.input_proj_t = input_proj_t; p.input_proj_b = input_proj.b;
        p.injected = injected ? noise_src : nullptr; p.seed = d_seed; p.temp = temp; p.gen_step = gen_step; p.rng_id = rng_id;
        p.h = h; p.q = q; p.ws_ml = af_ml; p.ws_acc = af_acc; p.mod = mod; p.xh = xh; p.noise_f32 = noise_f32; p.latent = latent; p.eos = eos;
        p.ff_bf = ff_bf; p.sy_bf = sy_bf; p.h1_bf = h1_bf; p.barrier = pf_barrier;
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3(sms); lc.blockDim = dim3(PF_THREADS); lc.dynamicSmemBytes = PF_SMEM_BYTES; lc.stream = stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
        lc.attrs = at; lc.numAttrs = 1;
        PTTS_CUDA_CHECK(cudaLaunchKernelEx(&lc, flow_persistent_kernel, p));
        launches++;
        launch_k(false, step_front_kernel, dim3(n), dim3(M_DIM), (size_t)(0), stream, slot0, n, (const float*)eos, (const float*)latent, cur_len, gen_step, eos_step, (const int*)max_gen,
                 (const int*)fae, active, lat_in_bf16, lat_f32, produced, eos_out, (const float*)emb_std, (const float*)emb_mean, (const __half*)wq, (const float*)wup, (const float*)bup, e_prev, xbuf);
        launches++;
    }

    // One generation step for slots [slot0, slot0+n) (reference _stream_sentence_step, src/pocket_tts.cpp:446-492).
    // FlowLM step + head + stop rule + Mimi front end (everything that consumes / produces the latent hand-off), cut into N_LAYERS + 1
    // segments: segment l < 6 ends with the attention kernel of layer l, segment 6 is the rest. seg < 0 enqueues all of them.
    static constexpr int N_SEG = N_LAYERS + 1;
    void flow_part(int slot0, int n, bool injected, float* xbuf, int seg = -1) {
        if (seg < 0 && use_persistent(n)) { flow_persistent(slot0, n, injected, xbuf); return; }
        set_pdl(pdl_small || pdl_chain);
        const int s_flow = (seg < 0) ? seg_begin(1) : -1;
        for (int sg = 0; sg < N_SEG; sg++) {
            if (seg >= 0 && sg != seg) continue;
            if (sg == 0) {
                launch_k(pdl_l(), flow_in_kernel, dim3(n), dim3(256), (size_t)0, stream, slot0, n, (const __nv_bfloat16*)lat_in_bf16, (const __nv_bfloat16*)input_linear_t,
                         (const float*)input_linear.b, (const float*)fl[0].n1w, (const float*)fl[0].n1b, h, n_bf, (const int*)cur_len, (const int*)active, (const float*)freq_flow, row_slot, row_pos, cs);
                launches++;
            } else {
                flow_chain_part(sg - 1, n);
            }
            if (sg < N_LAYERS) flow_attn_part(sg, n);
        }
        if (seg >= 0 && seg != N_SEG - 1) return;
        seg_end(s_flow);
        const int s_head = seg_begin(2);
        launch_k(pdl_l(), noise_inproj_kernel, dim3(n), dim3(128), (size_t)(0), stream, slot0, n, (const float*)(injected ? noise_src : nullptr), (const unsigned long long*)d_seed,
                 (const float*)temp, (const int*)gen_step, (const unsigned int*)rng_id, noise_f32, (const __nv_bfloat16*)input_proj_t, (const float*)input_proj.b, xh);
        flow_head(n);
        launches += 1;
        seg_end(s_head);
        set_pdl(pdl_small);
        // stop rule + latent hand-off + Mimi front end (writes the 16 transformer input rows of every slot to xbuf)
        launch_k(pdl_l(), step_front_kernel, dim3(n), dim3(M_DIM), (size_t)(0), stream, slot0, n, (const float*)eos, (const float*)latent, cur_len, gen_step, eos_step, (const int*)max_gen,
                 (const int*)fae, active, lat_in_bf16, lat_f32, produced, eos_out, (const float*)emb_std, (const float*)emb_mean, (const __half*)wq, (const float*)wup, (const float*)bup, e_prev, xbuf);
        launches++;
    }
    void step_enqueue(int slot0, int n, bool injected) {       // single-stream form (eager / profiling)
        const int s_all = seg_begin(5);
        flow_part(slot0, n, injected, mx);
        if (taps_on)   // the Mimi transformer updates its input rows in place: keep the upsampler output aside
            PTTS_CUDA_CHECK(cudaMemcpyAsync(tap_up + (size_t)slot0 * M_T * M_DIM, mx + (size_t)slot0 * M_T * M_DIM, (size_t)n * M_T * M_DIM * sizeof(float), cudaMemcpyDeviceToDevice, stream));
        mimi(slot0, n, mx);
        seg_end(s_all);
    }

    // kind 0 = full generation step (one stream), 1 = Mimi-only decode, 2 = FlowLM segment `part` -> mx2[par], 3 = Mimi chunk `part`
    // from mx2[par]. Runs on the CURRENT `stream` member (the pipeline swaps in stream_m for kind 3).
    static constexpr int ALL_PARTS = 15;     // `part` value meaning every segment / chunk in one graph
    void run_graphed(int kind, int slot0, int n, bool injected, int par = 0, int part = 0) {
        // PDL overlaps each kernel's prologue (barrier init, TMEM allocation, weight prefetch) with its predecessor's tail: a win while
        // the step is launch/latency bound (measured +2..7 % at batch 16-128), a loss once the kernels fill the machine (-10 % at 256).
        // cfg.pdl: 0 never, 1 up to 128 utterances, 2 always, 3 = FlowLM graph always / Mimi graph up to 128, 4 = Mimi graph always / FlowLM up to 128 (experiments)
        const bool side = kind == 3 || kind == 1;
        pdl_small = cfg.pdl == 2 || (cfg.pdl >= 1 && n <= 128) || (cfg.pdl == 3 && !side) || (cfg.pdl == 4 && side);
        pdl_chain = cfg.pdl == 2 || (cfg.pdl == 3 && !side) || (cfg.pdl == 4 && side);
        set_pdl(pdl_small);
        pdl_light = pdl_light_allowed && cfg.pdl >= 1 && !pdl_small; tc->pdl_light = pdl_light;
        // TMA-store epilogue for the large Mimi GEMMs only when no second stream runs beside them (see EPI_CLASSES in gemm_tc.cuh)
        tc->tma_epilogue = tma_epilogue_allowed && (kind == 0 || kind == 1);
        auto body = [&]() {
            if (kind == 0) step_enqueue(slot0, n, injected);
            else if (kind == 1) { mimi_front(slot0, n, mx); mimi(slot0, n, mx); }
            else if (kind == 2) flow_part(slot0, n, injected, mx2[par], part == ALL_PARTS ? -1 : part);
            else mimi(slot0, n, mx2[par], part == ALL_PARTS ? -1 : part);
        };
        if (!cfg.cuda_graphs || profiling || taps_on) { body(); return; }
        const auto gkey = std::make_tuple((kind * 2 + par) * 16 + part, slot0, n, (injected ? 1 : 0) | (pcm_out != pcm ? 2 : 0) | (noise_src != noise_inj ? 4 : 0), (kind == 0 || kind == 2) ? dec_grid_items : 0);
        if (!graphs.count(gkey)) { graphs[gkey].last_use = ++graph_clock; evict_graphs(); }
        GraphEntry& g = graphs[gkey];
        g.last_use = ++graph_clock;
        if (g.exec) { PTTS_CUDA_CHECK(cudaGraphLaunch(g.exec, stream)); launches += g.nlaunch; return; }
        if (g.seen++ == 0) { body(); return; }              // eager once: function attributes set, tensor maps encoded
        PTTS_CUDA_CHECK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        const long long l0 = launches;
        body();
        g.nlaunch = launches - l0; launches = l0;
        cudaGraph_t graph = nullptr;
        PTTS_CUDA_CHECK(cudaStreamEndCapture(stream, &graph));
        PTTS_CUDA_CHECK(cudaGraphInstantiate(&g.exec, graph, 0));
        PTTS_CUDA_CHECK(cudaGraphDestroy(graph));
        PTTS_CUDA_CHECK(cudaGraphLaunch(g.exec, stream)); launches += g.nlaunch;
    }

    // ---- two-stream pipeline -------------------------------------------------------------------------------------------------------
    // FlowLM(t) runs on the main stream as N_SEG graphs, each ending with an attention kernel (HBM saturated, every SM busy). After
    // segment l the main stream records an event and the Mimi stream, gated by it, runs chunk l of the PREVIOUS frame's Mimi decode:
    // the tensor/ALU-bound Mimi work lands in the windows where the main stream runs its latency-bound chain of decode-sized GEMMs
    // instead of competing with the KV stream for HBM. A frame whose Mimi decode has not been enqueued yet is `pending`; it is
    // decoded by the next run_step, or right away by flush_pending() (synchronous b200_step, b200_join, b200_sync, b200_collect).
    struct PendingFrame { bool valid = false; int slot0 = 0, n = 0, par = 0; long long tag = -1; } pending;   // tag = b200_submit index or -1
    cudaEvent_t ev_seg[8] = {};

    void mimi_chunk_on_side(const PendingFrame& f, int chunk) {
        std::swap(stream, stream_m); tc->cur_ws = 1;          // the Mimi stream has its own split-K workspace
        if (f.tag >= 0) {
            pcm_out = pcm_alt[f.par];
            if ((chunk == ALL_PARTS || chunk == 0) && ev_copy_valid[f.par]) PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_copy[f.par], 0));   // frame t-2's copy read this buffer
        }
        run_graphed(3, f.slot0, f.n, false, f.par, chunk);
        pcm_out = pcm;
        std::swap(stream, stream_m); tc->cur_ws = 0;
    }
    void finish_mimi_frame(const PendingFrame& f) {
        PTTS_CUDA_CHECK(cudaEventRecord(ev_mimi[f.par], stream_m));
        ev_mimi_valid[f.par] = true; mimi_pending = true; last_mimi_par = f.par;
        if (f.tag >= 0) {   // b200_submit frame: its PCM copy runs on the copy stream behind its Mimi decode (join_mimi covers it through ev_copy)
            auto& pd = pend[f.tag & 3];
            PTTS_CUDA_CHECK(cudaEventRecord(ev_dec[f.par], stream_m));
            PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream_c, ev_dec[f.par], 0));
            PTTS_CUDA_CHECK(cudaMemcpyAsync(pd.pcm, pcm_alt[f.par] + (size_t)f.slot0 * FRAME, (size_t)f.n * FRAME * sizeof(float), cudaMemcpyDeviceToHost, stream_c));
            PTTS_CUDA_CHECK(cudaEventRecord(pd.done_mimi, stream_c));
            PTTS_CUDA_CHECK(cudaEventRecord(ev_copy[f.par], stream_c));
            ev_copy_valid[f.par] = true; last_copy_par = f.par;
        }
    }
    // Enqueue the whole Mimi decode of the pending frame now (no interleaving partner).
    void flush_pending() {
        if (!pending.valid) return;
        const PendingFrame f = pending; pending.valid = false;
        if (debug_skip_mimi) return;
        PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream_m, ev_main[f.par], 0));
        tc->coreside = tc->coreside_allowed;                  // same graphs (same launch shapes) as the interleaved form
        if (one_graph_per_stream(f.n)) mimi_chunk_on_side(f, ALL_PARTS);
        else for (int c = 0; c < N_MCHUNK; c++) mimi_chunk_on_side(f, c);
        tc->coreside = false;
        finish_mimi_frame(f);
    }
    // Main stream waits for everything enqueued on the Mimi stream (before any non-pipelined use of Mimi state / PCM on the main stream).
    cudaEvent_t ev_begin = nullptr, ev_reset = nullptr; bool reset_pending = false;   // sentence-start Mimi reset enqueued on the Mimi stream
    void join_mimi() {
        flush_pending();
        if (reset_pending) { PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_reset, 0)); reset_pending = false; }
        if (!mimi_pending) return;
        if (ev_mimi_valid[last_mimi_par]) PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_mimi[last_mimi_par], 0));
        if (last_copy_par >= 0) { PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_copy[last_copy_par], 0)); last_copy_par = -1; }
        mimi_pending = false;
    }

    // One generation step for slots [slot0, slot0+n).
    // Below this many utterances the step runs as ONE FlowLM graph + ONE Mimi graph enqueued right away; above, as 7 + 6 graphs with the Mimi
    // chunks gated behind the attention kernels. Round 1 measured the gated form ahead at batch >= 32; with the fused head / SEANet tail
    // (fewer, longer kernels) the single-graph form wins everywhere (batch 32: 0.551 -> 0.536 ms, 128: 0.715 -> 0.695, 192: 0.857 -> 0.794,
    // 256: 0.983 -> 0.933), so the default is "always"; the gated form stays selectable.
    int immediate_below = getenv("PTTS_B200_IMMEDIATE_BELOW") ? atoi(getenv("PTTS_B200_IMMEDIATE_BELOW")) : (1 << 30);   // tuning hook
    bool one_graph_per_stream(int n) const { return (n >= 4 && n < immediate_below) || use_persistent(n); }
    bool last_step_piped = false;        // the last run_step left its Mimi decode (and PCM copy, for b200_submit frames) to the Mimi stream
    void run_step(int slot0, int n, bool injected, long long tag = -1) {
        last_step_piped = false;
        prepare_decode(slot0, n);
        tap_slot0 = slot0; tap_n = n;
        if (!cfg.overlap || !cfg.cuda_graphs || profiling || taps_on) { join_mimi(); run_graphed(0, slot0, n, injected); return; }
        last_step_piped = true;
        const int par = (int)(pipe_t & 1);
        struct CoresideScope { TcPlanCache* c; CoresideScope(TcPlanCache* c_) : c(c_) { c->coreside = c->coreside_allowed; } ~CoresideScope() { c->coreside = false; } } cs_scope(tc);
        PendingFrame prev = pending; pending.valid = false;
        if (prev.valid && (prev.slot0 != slot0 || prev.n != n)) { pending = prev; flush_pending(); prev.valid = false; }   // different slot range: no interleave
        if (debug_skip_mimi) prev.valid = false;
        if (prev.valid) PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream_m, ev_main[prev.par], 0));
        if (one_graph_per_stream(n)) {
            // 4..31 utterances: one graph for the whole FlowLM part and one for the whole Mimi decode, enqueued immediately (measured:
            // batch 8 0.545 -> 0.533 ms, batch 16 0.604 -> 0.577 ms; at batch 1-3 the 7 + 6 short graphs are faster, 0.40 vs 0.46 ms)
            if (ev_mimi_valid[par]) PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_mimi[par], 0));
            run_graphed(2, slot0, n, injected, par, ALL_PARTS);
            PTTS_CUDA_CHECK(cudaEventRecord(ev_main[par], stream));
            pending.valid = true; pending.slot0 = slot0; pending.n = n; pending.par = par; pending.tag = tag;
            pipe_t++;
            flush_pending();
            return;
        }
        for (int sg = 0; sg < N_SEG; sg++) {
            // only the last segment (step_front_kernel) writes the hand-off rows mx2[par]: wait there, not at the start of the step, for
            // frame t-2's Mimi decode (long finished in steady state; waiting up front would put its tail on the critical path)
            if (sg == N_SEG - 1 && ev_mimi_valid[par]) PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_mimi[par], 0));
            run_graphed(2, slot0, n, injected, par, sg);
            if (prev.valid && sg < N_MCHUNK) {
                PTTS_CUDA_CHECK(cudaEventRecord(ev_seg[sg], stream));
                PTTS_CUDA_CHECK(cudaStreamWaitEvent(stream_m, ev_seg[sg], 0));
                mimi_chunk_on_side(prev, sg);
            }
        }
        if (prev.valid) finish_mimi_frame(prev);
        PTTS_CUDA_CHECK(cudaEventRecord(ev_main[par], stream));
        pending.valid = true; pending.slot0 = slot0; pending.n = n; pending.par = par; pending.tag = tag;
        pipe_t++;
        // Small batches are launch-latency bound, not HBM bound: there is nothing to gain from placing the Mimi chunks behind the next
        // step's attention kernels, and holding the frame back would add a whole FlowLM step to its latency. Decode it right away on
        // the Mimi stream; it still overlaps the next FlowLM step (streaming API look-ahead, b200_submit).
        if (n < immediate_below) flush_pending();
    }

    void ensure_pinned(size_t nf, size_t ni) {
        if (nf > pin_f_n) { if (pin_f) cudaFreeHost(pin_f); PTTS_CUDA_CHECK(cudaMallocHost(&pin_f, nf * sizeof(float))); pin_f_n = nf; }
        if (ni > pin_i_n) { if (pin_i) cudaFreeHost(pin_i); PTTS_CUDA_CHECK(cudaMallocHost(&pin_i, ni * sizeof(int))); pin_i_n = ni; }
    }

    // ---- voice-cloning encoder (DESIGN.md §4.6): PCM -> audio_prompt rows [T][1024] on the main stream ----
    bool has_enc = false;
    ConvW ec0, er1a, er1b, es3, er4a, er4b, es6, er7a, er7b, es9, ec11, eds;
    struct { LinW in_proj, out_proj, lin1, lin2; float *n1w, *n1b, *n2w, *n2b, *ls1, *ls2; } el[M_LAYERS];
    LinW spk;
    // Scratch of the last clone, grown to the longest prompt so far (one allocation; its own buffers, so that a Mimi decode running on the
    // other stream beside it shares nothing with it). The zero rows in front of the conv inputs are causal padding and are never written.
    struct EncBufs {
        int T = 0;
        float *pcm, *y0, *y1, *y2, *xs, *xt, *lat, *prompt; float2* cs;
        __half *a0, *b0, *c0, *a1, *b1, *c1, *a2, *b2, *c2, *d3, *ds;
        __nv_bfloat16 *ln, *q, *k, *v, *att, *ff, *lat_bf;
    } eb;
    int enc_T = 0;                       // rows of the last clone (debug taps)
    // Pinned staging of the clone's PCM, sized with the scratch. Not the shared pinned ring: a 10 s prompt is ~1 MB, and growing a ring
    // slot to that size (cudaFreeHost + cudaMallocHost) on most clones stalls the serving pipeline.
    float* enc_pin = nullptr; size_t enc_pin_cap = 0; cudaEvent_t enc_pin_ev = nullptr; bool enc_pin_used = false;
    void enc_reserve(int T) {
        if (T <= eb.T) return;
        const int Tc = std::min(std::max(T, 2 * eb.T), cfg.kv_capacity);   // no clone is longer than kv_capacity rows
        const long long L0 = (long long)ENC_HOP * Tc, L1 = L0 / 4, L2 = L1 / 5, L3 = L2 / 6;
        size_t off = 0;
        std::vector<std::pair<void**, size_t>> parts;
        auto part = [&](auto*& p, size_t bytes) { parts.push_back({(void**)&p, off}); off += (bytes + 255) / 256 * 256; };
        part(eb.pcm, (6 + L0) * 4); part(eb.y0, L0 * 64 * 4); part(eb.a0, (2 + L0) * 64 * 2); part(eb.b0, L0 * 64 * 2); part(eb.c0, (4 + L0) * 64 * 2);
        part(eb.y1, L1 * 128 * 4); part(eb.a1, (2 + L1) * 128 * 2); part(eb.b1, L1 * 64 * 2); part(eb.c1, (5 + L1) * 128 * 2);
        part(eb.y2, L2 * 256 * 4); part(eb.a2, (2 + L2) * 256 * 2); part(eb.b2, L2 * 128 * 2); part(eb.c2, (6 + L2) * 256 * 2);
        part(eb.d3, (2 + L3) * 512 * 2); part(eb.xs, L3 * 512 * 4); part(eb.xt, L3 * 512 * 4); part(eb.cs, L3 * 32 * 8);
        part(eb.ln, L3 * 512 * 2); part(eb.q, L3 * 512 * 2); part(eb.k, L3 * 512 * 2); part(eb.v, L3 * 512 * 2); part(eb.att, L3 * 512 * 2);
        part(eb.ff, L3 * M_FF * 2); part(eb.ds, (16 + L3) * 512 * 2); part(eb.lat, (long long)Tc * 512 * 4); part(eb.lat_bf, (long long)Tc * 512 * 2);
        part(eb.prompt, (long long)Tc * D_MODEL * 4);
        char* base = dalloc<char>(off, true);    // zeroed: padding rows and the padded channels of b0 stay zero for every later clone
        for (auto& pp : parts) *pp.first = base + pp.second;
        eb.T = Tc;
    }
    // Encodes pcm (already in eb.pcm behind 6 zero samples, zero-padded to 1920 T) into eb.prompt [T][1024]. Main stream, no host wait.
    void encode(int T) {
        const int BIG = 1 << 30;
        const long long L0 = (long long)ENC_HOP * T, L1 = L0 / 4, L2 = L1 / 5, L3 = L2 / 6;
        set_pdl(false);
        tc->tma_epilogue = false;                                  // the Mimi stream may be running beside the encoder
        launch_k(false, enc_front_kernel, dim3((unsigned)((L0 * 64 + 255) / 256)), dim3(256), (size_t)0, stream, (const float*)eb.pcm, (const __half*)ec0.w,
                 (const float*)ec0.b, (int)L0, eb.y0, eb.a0 + 2 * 64);
        launches++;
        // residual block: x + conv1(ELU(conv3(ELU(x)))), then ELU -> the f16 input rows of the next strided conv (behind `pad` zero rows)
        auto resblock = [&](ConvW& ca, ConvW& cb, long long L, int C, __half* a, __half* b, int ldb, float* y, __half* c, int pad) {
            { Epi e; e.rps = (int)L; e.bias = ca.b; e.act = ACT_ELU; e.out2 = b; e.out2_map = rows(ldb); e.out2_type = OUT2_F16;
              gemm<__half>(a, smap((L + 2) * C, C, 0), (int)L, ca.w, ca.wk, (int)L, ca.N, ca.K, e); }
            { Epi e; e.bias = cb.b; e.resid = y; e.resid_map = rows(C); e.act = ACT_ELU; e.out2 = c + (long long)pad * C; e.out2_map = rows(C); e.out2_type = OUT2_F16;
              gemm<__half>(b, rows(ldb), BIG, cb.w, cb.wk, (int)L, cb.N, cb.K, e); }
        };
        // conv k = 2r, stride r over [L][C] = 2-tap window over rows of r*C channels (one zero row-group in front): Lo = L / r rows out
        auto strided = [&](ConvW& cw, const __half* in, long long Lo, int rC, float* y, __half* out2, int out_pad) {
            Epi e; e.rps = (int)Lo; e.bias = cw.b; e.act = ACT_ELU; e.out2 = out2 + (long long)out_pad * cw.N; e.out2_map = rows(cw.N); e.out2_type = OUT2_F16;
            if (y) { e.out = y; e.out_map = rows(cw.N); }
            gemm<__half>(in, smap((Lo + 1) * rC, rC, 0), (int)Lo, cw.w, cw.wk, (int)Lo, cw.N, cw.K, e);
        };
        resblock(er1a, er1b, L0, 64, eb.a0, eb.b0, 64, eb.y0, eb.c0, 4);
        strided(es3, eb.c0, L1, 4 * 64, eb.y1, eb.a1, 2);
        resblock(er4a, er4b, L1, 128, eb.a1, eb.b1, 64, eb.y1, eb.c1, 5);
        strided(es6, eb.c1, L2, 5 * 128, eb.y2, eb.a2, 2);
        resblock(er7a, er7b, L2, 256, eb.a2, eb.b2, 128, eb.y2, eb.c2, 6);
        strided(es9, eb.c2, L3, 6 * 256, nullptr, eb.d3, 2);
        { Epi e; e.rps = (int)L3; e.bias = ec11.b; e.out = eb.xs; e.out_map = rows(512);
          gemm<__half>(eb.d3, smap((L3 + 2) * 512, 512, 0), (int)L3, ec11.w, ec11.wk, (int)L3, ec11.N, ec11.K, e); }
        // encoder transformer over the 16 T rows (positions 0 .. 16T-1), layer math of the Mimi decoder's, plain causal window
        const int R = (int)L3;
        launch_k(false, enc_rope_kernel, dim3((R * 32 + 255) / 256), dim3(256), (size_t)0, stream, (const float*)freq_mimi, eb.cs, R);
        launches++;
        auto ln = [&](const float* x, const float* w, const float* b) {
            if (R >= 512) launch_k(false, layernorm_rows_kernel<M_DIM>, dim3((R + 7) / 8), dim3(256), (size_t)0, stream, x, R, 0.0f, w, b, eb.ln);
            else launch_k(false, layernorm_kernel<M_DIM>, dim3(R), dim3(M_DIM / 4), (size_t)0, stream, x, rows(M_DIM), BIG, R, 0.0f, w, b, nullptr, nullptr, 0, eb.ln, nullptr);
            launches++;
        };
        for (int l = 0; l < M_LAYERS; l++) {
            auto& L = el[l];
            const float* xin = l == 0 ? eb.xs : eb.xt;
            ln(xin, L.n1w, L.n1b);
            Epi eq; eq.mode = EPI_MIMI_QKV; eq.kv_linear = 1; eq.cs = eb.cs; eq.kcache = eb.k; eq.vcache = eb.v; eq.q_out_bf16 = eb.q;
            lin(eb.ln, L.in_proj, R, eq);
            launch_k(false, attn_window_kernel, dim3((R + AW_Q - 1) / AW_Q, M_HEADS), dim3(AW_WARPS * 32), AW_SMEM, stream, (const __nv_bfloat16*)eb.q,
                     (const __nv_bfloat16*)eb.k, (const __nv_bfloat16*)eb.v, R, eb.att);
            launches++;
            Epi eo; eo.colscale = L.ls1; eo.resid = xin; eo.resid_map = rows(M_DIM); eo.out = eb.xt; eo.out_map = rows(M_DIM);
            lin(eb.att, L.out_proj, R, eo);
            ln(eb.xt, L.n2w, L.n2b);
            Epi e1; e1.out2 = eb.ff; e1.out2_map = rows(M_FF); e1.out2_type = OUT2_BF16; e1.act = ACT_GELU;
            lin(eb.ln, L.lin1, R, e1);
            Epi e2; e2.colscale = L.ls2; e2.resid = eb.xt; e2.resid_map = rows(M_DIM); e2.out = eb.xt; e2.out_map = rows(M_DIM);
            lin(eb.ff, L.lin2, R, e2);
        }
        // downsample k32 s16 (replicate padding) as a 2-tap window over rows of 16 x 512, then the speaker projection
        launch_k(false, enc_ds_pad_kernel, dim3((unsigned)(((long long)(R + 16) * M_DIM + 255) / 256)), dim3(256), (size_t)0, stream, (const float*)eb.xt, R, eb.ds);
        { Epi e; e.rps = T; e.bias = eds.b; e.out = eb.lat; e.out_map = rows(512);
          gemm<__half>(eb.ds, smap((long long)(T + 1) * 16 * 512, 16 * 512, 0), T, eds.w, eds.wk, T, eds.N, eds.K, e); }
        launch_k(false, enc_to_bf16_kernel, dim3((unsigned)(((long long)T * 512 + 255) / 256)), dim3(256), (size_t)0, stream, (const float*)eb.lat, (long long)T * 512, eb.lat_bf);
        launches += 2;
        { Epi e; e.out = eb.prompt; e.out_map = rows(D_MODEL); lin(eb.lat_bf, spk, T, e); }
        enc_T = T;
    }
};

namespace {

__global__ void set_meta_kernel(int slot, int cur, int mg, int f, float t, const float* bos, int* cur_len, int* gen_step, int* eos_step,
                                int* max_gen, int* fae, int* active, float* temp, __nv_bfloat16* lat_in_bf16, float* lat_f32) {
    pdl_prologue();
    const int i = threadIdx.x;
    if (i == 0) { cur_len[slot] = cur; gen_step[slot] = 0; eos_step[slot] = -1; max_gen[slot] = mg; fae[slot] = f; active[slot] = mg > 0 ? 1 : 0; temp[slot] = t; }
    if (i < LDIM) { lat_f32[slot * LDIM + i] = bos[i]; lat_in_bf16[slot * LDIM + i] = __float2bfloat16_rn(bos[i]); }
}

// Batched sentence start (b200_begin_sentences; reference _stream_sentence_init src/pocket_tts.cpp:416-444, copy_states models/flow_lm.h:70-78,
// init(mimi_states) models/mimi.h:71-75): one launch each for all n sentences instead of three launches per sentence.
// meta = [slot | src voice slot | prefix rows | cur_len | max_gen | frames_after_eos | shared prefix rows (0 = private copy) | RNG stream id] x n (ints), temps[n].
// FlowLM-side state (main stream): stop-rule counters, BOS latent, upsampler carry, prefix assignment.
__global__ void begin_meta_kernel(int n, const int* __restrict__ meta, const float* __restrict__ temps, const float* bos, int* cur_len, int* gen_step, int* eos_step,
                                  int* max_gen, int* fae, int* active, float* temp, __nv_bfloat16* lat_in_bf16, float* lat_f32,
                                  int* __restrict__ pfx_slot, int* __restrict__ pfx_len, float* __restrict__ e_prev, unsigned int* __restrict__ rng_id) {
    const int j = blockIdx.x, i = threadIdx.x;
    if (j >= n) return;
    const int slot = meta[j], cur = meta[3 * n + j], mg = meta[4 * n + j], f = meta[5 * n + j];
    if (i == 0) {
        cur_len[slot] = cur; gen_step[slot] = 0; eos_step[slot] = -1; max_gen[slot] = mg; fae[slot] = f; active[slot] = mg > 0 ? 1 : 0; temp[slot] = temps[j];
        pfx_slot[slot] = meta[n + j]; pfx_len[slot] = meta[6 * n + j]; rng_id[slot] = (unsigned int)meta[7 * n + j];
    }
    if (i < LDIM) { lat_f32[slot * LDIM + i] = bos[i]; lat_in_bf16[slot * LDIM + i] = __float2bfloat16_rn(bos[i]); }
    for (int c = i; c < M_DIM; c += blockDim.x) e_prev[(long long)slot * M_DIM + c] = 0.f;
}
// b200_end_sentences: the listed slots become dead rows from the next step on (main stream, so steps enqueued earlier still see them live).
__global__ void end_slots_kernel(int n, const int* __restrict__ slots, int* __restrict__ active) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) active[slots[i]] = 0;
}
__global__ void begin_copy_prefix_kernel(int n, const int* __restrict__ meta, char* kc, char* vc, long long slot_bytes, long long layer_bytes, long long row_bytes) {
    const int j = blockIdx.z;
    const int dst_slot = meta[j], src_slot = meta[n + j];
    const long long n16 = (long long)meta[2 * n + j] * row_bytes / 16;
    char* base = (blockIdx.y & 1) ? vc : kc;
    const int layer = blockIdx.y >> 1;
    const uint4* src = reinterpret_cast<const uint4*>(base + layer * layer_bytes + src_slot * slot_bytes);
    uint4* dst = reinterpret_cast<uint4*>(base + layer * layer_bytes + dst_slot * slot_bytes);
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n16; i += 4 * stride) {              // four independent 16-byte loads in flight per thread
        const uint4 a = src[i], b = src[i + stride], c = src[i + 2 * stride], d = src[i + 3 * stride];
        dst[i] = a; dst[i + stride] = b; dst[i + 2 * stride] = c; dst[i + 3 * stride] = d;
    }
    for (; i < n16; i += stride) dst[i] = src[i];
}
// Mimi-side state (Mimi stream, behind every decode already enqueued there): carried conv rows, ring offset.
__global__ void begin_reset_kernel(int n, const int* __restrict__ meta, ShiftAll sa, int* __restrict__ mimi_off) {
    const int slot = meta[blockIdx.x];
    const ShiftDesc d = sa.d[blockIdx.y];
    __half* base = d.buf + (long long)slot * d.slot_stride;
    for (int i = threadIdx.x; i < d.S * d.C; i += blockDim.x) base[i] = __float2half_rn(0.f);
    if (blockIdx.y == 0 && threadIdx.x == 0) mimi_off[slot] = 0;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

void b200_default_config(b200_config* c) {
    memset(c, 0, sizeof(*c));
    c->device = 0; c->max_slots = 1; c->max_voices = 8; c->kv_capacity = 2048; c->kv_f32 = 0; c->mimi_mask_mode = 0;
    c->convt_split = 0; c->gemm_path = 0; c->max_prefill_rows = 4096; c->cuda_graphs = 1; c->pdl = 1; c->overlap = 1; c->prefix_share = 1;
}

int b200_engine_create(const b200_config* cfg, b200_engine** out) {
    if (!cfg || !out || cfg->max_slots < 1 || cfg->kv_capacity < 16 || cfg->kv_capacity > 12288) return B200_EINVAL;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        fprintf(stderr, "ptts_b200: error: no CUDA device (this engine has no CPU fallback)\n");
        return B200_ESTATE;
    }
    auto* e = new b200_engine; e->cfg = *cfg;
    if (e->cfg.max_prefill_rows <= 0) e->cfg.max_prefill_rows = 4096;
    if (e->cfg.max_voices < 1) e->cfg.max_voices = 1;
    PTTS_CUDA_CHECK(cudaSetDevice(cfg->device));
    {   // the FlowLM chain is the critical path of a frame: it gets the higher priority, the Mimi decode fills the gaps
        int lo = 0, hi = 0;
        PTTS_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        PTTS_CUDA_CHECK(cudaStreamCreateWithPriority(&e->stream, cudaStreamNonBlocking, hi));
        PTTS_CUDA_CHECK(cudaStreamCreateWithPriority(&e->stream_m, cudaStreamNonBlocking, lo));
        PTTS_CUDA_CHECK(cudaStreamCreateWithPriority(&e->stream_t, cudaStreamNonBlocking, hi));
        PTTS_CUDA_CHECK(cudaStreamCreateWithPriority(&e->stream_c, cudaStreamNonBlocking, lo));
        PTTS_CUDA_CHECK(cudaStreamCreateWithPriority(&e->stream_n, cudaStreamNonBlocking, hi));
        PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
        PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
        for (int i = 0; i < 2; i++) {
            PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_main[i], cudaEventDisableTiming));
            PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_mimi[i], cudaEventDisableTiming));
            PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_dec[i], cudaEventDisableTiming));
            PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_copy[i], cudaEventDisableTiming));
            PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_noise[i], cudaEventDisableTiming));
        }
        for (auto& ev : e->ev_seg) PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_begin, cudaEventDisableTiming));
        PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_reset, cudaEventDisableTiming));
    }
    e->total_slots = cfg->max_slots + e->cfg.max_voices;
    e->max_rows = std::max(cfg->max_slots, e->cfg.max_prefill_rows);
    e->voice_len.assign(e->cfg.max_voices, 0);
    e->h_cur_len.assign(cfg->max_slots, 0);
    e->h_pfx_slot.assign(e->total_slots, 0); e->h_pfx_len.assign(e->total_slots, 0);
    e->tc = tc_plan_cache_create();
    *out = e;
    return B200_OK;
}

void b200_engine_destroy(b200_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    cudaStreamSynchronize(e->stream);
    cudaStreamSynchronize(e->stream_m); cudaStreamSynchronize(e->stream_c);
    cudaStreamSynchronize(e->stream_t);
    for (auto& kv : e->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    for (void* p : e->allocs) cudaFree(p);
    for (auto& pd : e->pend) {
        if (pd.noise) cudaFreeHost(pd.noise); if (pd.pcm) cudaFreeHost(pd.pcm); if (pd.produced) cudaFreeHost(pd.produced);
        if (pd.done_main) cudaEventDestroy(pd.done_main); if (pd.done_mimi) cudaEventDestroy(pd.done_mimi);
    }
    if (e->pin_f) cudaFreeHost(e->pin_f);
    if (e->pin_i) cudaFreeHost(e->pin_i);
    for (auto& ps : e->pins) { if (ps.p) cudaFreeHost(ps.p); if (ps.ev) cudaEventDestroy(ps.ev); }
    if (e->ev_begin) cudaEventDestroy(e->ev_begin); if (e->ev_reset) cudaEventDestroy(e->ev_reset);
    if (e->enc_pin) cudaFreeHost(e->enc_pin); if (e->enc_pin_ev) cudaEventDestroy(e->enc_pin_ev);
    tc_plan_cache_destroy(e->tc);
    for (int i = 0; i < 2; i++) { cudaEventDestroy(e->ev_main[i]); cudaEventDestroy(e->ev_mimi[i]); cudaEventDestroy(e->ev_dec[i]); cudaEventDestroy(e->ev_copy[i]); cudaEventDestroy(e->ev_noise[i]); }
    for (auto& ev : e->ev_seg) cudaEventDestroy(ev);
    cudaEventDestroy(e->ev_fork); cudaEventDestroy(e->ev_join);
    cudaStreamDestroy(e->stream); cudaStreamDestroy(e->stream_m); cudaStreamDestroy(e->stream_t); cudaStreamDestroy(e->stream_c); cudaStreamDestroy(e->stream_n);
    delete e;
}

int b200_upload_tensor(b200_engine* e, const char* key, const void* data, int dtype, const int64_t* shape, int ndim) {
    if (!e || !key || !data || e->finalized) return B200_EINVAL;
    HostTensor t; t.dtype = dtype; size_t n = 1;
    for (int i = 0; i < ndim; i++) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
    t.f.resize(n);
    if (dtype == B200_DT_F32) memcpy(t.f.data(), data, n * 4);
    else if (dtype == B200_DT_BF16) { const uint16_t* s = (const uint16_t*)data; for (size_t i = 0; i < n; i++) { uint32_t u = (uint32_t)s[i] << 16; memcpy(&t.f[i], &u, 4); } }
    else if (dtype == B200_DT_F16) { const __half* s = (const __half*)data; for (size_t i = 0; i < n; i++) t.f[i] = __half2float(s[i]); }
    else return B200_EINVAL;
    e->host[key] = std::move(t);
    return B200_OK;
}

int b200_finalize_weights(b200_engine* e) {
    if (!e || e->finalized) return B200_ESTATE;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    const auto& cfg = e->cfg;
    // ---------------- weights ----------------
    auto* emb = e->find("flow_lm.conditioner.embed.weight");
    e->n_embed = (int)emb->shape[0];
    e->embed = e->upload(b200_engine::to_bf16(emb->f));
    e->emb_std = e->up_f32("flow_lm.emb_std"); e->emb_mean = e->up_f32("flow_lm.emb_mean");
    e->h_bos = e->find("flow_lm.bos_emb")->f; e->d_bos = e->upload(e->h_bos);
    e->input_linear = e->up_lin("flow_lm.input_linear", D_MODEL, LDIM);
    auto transposed = [&](const std::string& key, int out, int in) {
        const auto& w = e->find(key)->f;
        std::vector<float> t((size_t)out * in);
        for (int o = 0; o < out; o++) for (int k = 0; k < in; k++) t[(size_t)k * out + o] = w[(size_t)o * in + k];
        return e->upload(b200_engine::to_bf16(t));
    };
    e->input_linear_t = transposed("flow_lm.input_linear.weight", D_MODEL, LDIM);
    e->onw = e->up_f32("flow_lm.out_norm.weight"); e->onb = e->up_f32("flow_lm.out_norm.bias", false);
    e->w_eos = e->upload(b200_engine::to_bf16(e->find("flow_lm.out_eos.weight")->f));
    e->b_eos = e->up_f32("flow_lm.out_eos.bias", false);
    for (int l = 0; l < N_LAYERS; l++) {
        const std::string p = "flow_lm.transformer.layers." + std::to_string(l) + ".";
        auto& L = e->fl[l];
        L.in_proj = e->up_lin(p + "self_attn.in_proj", 3 * D_MODEL, D_MODEL); L.out_proj = e->up_lin(p + "self_attn.out_proj", D_MODEL, D_MODEL);
        L.lin1 = e->up_lin(p + "linear1", D_FF, D_MODEL); L.lin2 = e->up_lin(p + "linear2", D_MODEL, D_FF);
        L.n1w = e->up_f32(p + "norm1.weight"); L.n1b = e->up_f32(p + "norm1.bias", false);
        L.n2w = e->up_f32(p + "norm2.weight"); L.n2b = e->up_f32(p + "norm2.bias", false);
    }
    const std::string f = "flow_lm.flow_net.";
    e->input_proj = e->up_lin(f + "input_proj", D_FLOW, LDIM);
    e->input_proj_t = transposed(f + "input_proj.weight", D_FLOW, LDIM);
    e->cond_embed = e->up_lin(f + "cond_embed", D_FLOW, D_MODEL);
    {   // seven adaLN projections of the same silu(y) fused into one [10240][512] weight
        std::vector<float> w, b; bool has_b = true;
        for (int r = 0; r <= N_RES; r++) {
            const std::string p = r < N_RES ? f + "res_blocks." + std::to_string(r) + ".adaLN_modulation.1" : f + "final_layer.adaLN_modulation.1";
            auto* tw = e->find(p + ".weight"); w.insert(w.end(), tw->f.begin(), tw->f.end());
            auto* tb = e->find(p + ".bias", false);
            if (tb) b.insert(b.end(), tb->f.begin(), tb->f.end()); else { has_b = false; b.resize(w.size() / D_FLOW, 0.f); }
        }
        (void)has_b;
        e->ada_all.out = (int)(w.size() / D_FLOW); e->ada_all.in = D_FLOW;
        const auto wb = b200_engine::to_bf16(w);
        e->ada_all.w = e->upload(wb); e->ada_all.wk = e->upload(tc_kblock_major(wb, e->ada_all.out, D_FLOW)); e->ada_all.b = e->upload(b);
    }
    for (int r = 0; r < N_RES; r++) {
        const std::string p = f + "res_blocks." + std::to_string(r) + ".";
        e->rb[r].lnw = e->up_f32(p + "in_ln.weight", false); e->rb[r].lnb = e->up_f32(p + "in_ln.bias", false);
        e->rb[r].mlp0 = e->up_lin(p + "mlp.0", D_FLOW, D_FLOW); e->rb[r].mlp2 = e->up_lin(p + "mlp.2", D_FLOW, D_FLOW);
    }
    e->final_lin = e->up_lin(f + "final_layer.linear", LDIM, D_FLOW);
    e->fnw = e->up_f32(f + "final_layer.norm_final.weight", false); e->fnb = e->up_f32(f + "final_layer.norm_final.bias", false);
    {   // constant timestep embedding t_combined = (TE1(t=1) + TE0(s=0)) / 2 (reference modules/mlp.h:92-106,18-37,241-245)
        std::vector<float> tc(D_FLOW, 0.f);
        const float tval[2] = {0.0f, 1.0f};
        for (int idx = 0; idx < 2; idx++) {
            const std::string p = f + "time_embed." + std::to_string(idx) + ".";
            auto *w0 = e->find(p + "mlp.0.weight"), *b0 = e->find(p + "mlp.0.bias", false), *w2 = e->find(p + "mlp.2.weight"), *b2 = e->find(p + "mlp.2.bias", false);
            auto *alpha = e->find(p + "mlp.3.alpha"), *freqs = e->find(p + "freqs");
            float emb2[256], h1[D_FLOW], u[D_FLOW];
            for (int i = 0; i < 128; i++) { const float a = freqs->f[i] * tval[idx]; emb2[i] = h_bf16r(cosf(a)); emb2[128 + i] = h_bf16r(sinf(a)); }
            for (int o = 0; o < D_FLOW; o++) { float acc = 0.f; for (int i = 0; i < 256; i++) acc += h_bf16r(w0->f[(size_t)o * 256 + i]) * emb2[i]; h1[o] = h_bf16r(h_silu(acc + (b0 ? b0->f[o] : 0.f))); }
            for (int o = 0; o < D_FLOW; o++) { float acc = 0.f; for (int i = 0; i < D_FLOW; i++) acc += h_bf16r(w2->f[(size_t)o * D_FLOW + i]) * h1[i]; u[o] = acc + (b2 ? b2->f[o] : 0.f); }
            double s = 0; for (int i = 0; i < D_FLOW; i++) s += u[i];
            const float mean = (float)(s / D_FLOW);
            double ss = 0; for (int i = 0; i < D_FLOW; i++) { const float d = u[i] - mean; ss += (double)(d * d); }
            const float sd = sqrtf((float)ss * (1.f / (D_FLOW - 1)) + 1e-5f);
            for (int i = 0; i < D_FLOW; i++) tc[i] += alpha->f[i] * (u[i] / sd);
        }
        for (auto& v : tc) v *= 0.5f;
        e->t_combined = e->upload(tc);
    }
    // Mimi
    {
        auto* q = e->find("mimi.quantizer.output_proj.weight");
        // both stored transposed ([tap or input][channel]) so that lane = channel reads coalesced lines (mimi_front_kernel)
        std::vector<__half> qh(q->f.size());
        for (int c = 0; c < M_DIM; c++) for (int i = 0; i < LDIM; i++) qh[(size_t)i * M_DIM + c] = __float2half_rn(q->f[(size_t)c * LDIM + i]);
        e->wq = e->upload(qh);
        auto* up = e->find("mimi.upsample.convtr.convtr.weight");
        std::vector<float> ut(up->f.size());
        for (int c = 0; c < M_DIM; c++) for (int k = 0; k < 32; k++) ut[(size_t)k * M_DIM + c] = up->f[(size_t)c * 32 + k];
        e->wup = e->upload(ut); e->bup = e->up_f32("mimi.upsample.convtr.convtr.bias", false);
    }
    for (int l = 0; l < M_LAYERS; l++) {
        const std::string p = "mimi.decoder_transformer.transformer.layers." + std::to_string(l) + ".";
        auto& L = e->ml[l];
        L.in_proj = e->up_lin(p + "self_attn.in_proj", 3 * M_DIM, M_DIM); L.out_proj = e->up_lin(p + "self_attn.out_proj", M_DIM, M_DIM);
        L.lin1 = e->up_lin(p + "linear1", M_FF, M_DIM); L.lin2 = e->up_lin(p + "linear2", M_DIM, M_FF);
        L.n1w = e->up_f32(p + "norm1.weight"); L.n1b = e->up_f32(p + "norm1.bias", false);
        L.n2w = e->up_f32(p + "norm2.weight"); L.n2b = e->up_f32(p + "norm2.bias", false);
        L.ls1 = e->up_f32(p + "layer_scale_1.scale"); L.ls2 = e->up_f32(p + "layer_scale_2.scale");
    }
    e->C2 = cfg.convt_split ? 1024 : 512; e->C5 = cfg.convt_split ? 512 : 256; e->C8 = cfg.convt_split ? 256 : 128;
    const std::string d = "mimi.decoder.model.";
    e->c0 = e->up_conv(d + "0", 512, 512, 7);
    e->t2 = e->up_convt(d + "2", 512, 256, 12, 6, e->C2);
    e->r3a = e->up_conv(d + "3.block.1", 128, 256, 3); e->r3b = e->up_conv(d + "3.block.3", 256, 128, 1);
    e->t5 = e->up_convt(d + "5", 256, 128, 10, 5, e->C5);
    e->r6a = e->up_conv(d + "6.block.1", 64, 128, 3); e->r6b = e->up_conv(d + "6.block.3", 128, 64, 1);
    e->t8 = e->up_convt(d + "8", 128, 64, 8, 4, e->C8);
    e->r9a = e->up_conv(d + "9.block.1", 32, 64, 3); e->r9b = e->up_conv(d + "9.block.3", 64, 32, 1, 64);
    e->c11 = e->up_conv(d + "11", 1, 64, 3);
    {
        std::vector<float> ff(32), fm(32);
        for (int i = 0; i < 32; i++) {
            ff[i] = expf((float)i * (-logf(10000.0f) / 32));        // FlowLM: ggml_scale then ggml_exp (rope.h:36-38)
            fm[i] = (float)expf(-logf(10000.0f) * i / 32);          // Mimi: ggml_timestep_embedding (rope.h:8-20)
        }
        e->freq_flow = e->upload(ff); e->freq_mimi = e->upload(fm);
    }
    {   // voice-cloning encoder: all or nothing. Its key names live in this one table (a checkpoint with other names is a one-line change).
        const std::string se = "mimi.encoder.model.", te = "mimi.encoder_transformer.transformer.layers.";
        struct ConvKey { ConvW* dst; std::string key; int co, ci, k, ci_pad; };
        const ConvKey convs[] = {
            {&e->ec0, se + "0", 64, 1, 7, 0},          {&e->er1a, se + "1.block.1", 32, 64, 3, 0},  {&e->er1b, se + "1.block.3", 64, 32, 1, 64},
            {&e->es3, se + "3", 128, 64, 8, 0},        {&e->er4a, se + "4.block.1", 64, 128, 3, 0}, {&e->er4b, se + "4.block.3", 128, 64, 1, 0},
            {&e->es6, se + "6", 256, 128, 10, 0},      {&e->er7a, se + "7.block.1", 128, 256, 3, 0}, {&e->er7b, se + "7.block.3", 256, 128, 1, 0},
            {&e->es9, se + "9", 512, 256, 12, 0},      {&e->ec11, se + "11", 512, 512, 3, 0},       {&e->eds, "mimi.downsample.conv", 512, 512, 32, 0}};
        const char* layer_keys[] = {"self_attn.in_proj.weight", "self_attn.out_proj.weight", "linear1.weight", "linear2.weight", "norm1.weight", "norm2.weight",
                                    "layer_scale_1.scale", "layer_scale_2.scale"};
        const std::string spk_key = "flow_lm.speaker_proj_weight";
        if (e->find(se + "0.conv.weight", false)) {
            std::vector<std::string> need;
            for (const auto& c : convs) need.push_back(c.key + ".conv.weight");
            for (int l = 0; l < M_LAYERS; l++) for (const char* k : layer_keys) need.push_back(te + std::to_string(l) + "." + k);
            need.push_back(spk_key);
            for (const auto& k : need) if (!e->find(k, false)) { fprintf(stderr, "ptts_b200: error: incomplete encoder weights, missing tensor %s\n", k.c_str()); return B200_EINVAL; }
            for (const auto& c : convs) {
                const auto* w = e->find(c.key + ".conv.weight");
                if ((int64_t)w->f.size() != (int64_t)c.co * c.ci * c.k) { fprintf(stderr, "ptts_b200: error: bad shape for %s.conv.weight\n", c.key.c_str()); return B200_EINVAL; }
                *c.dst = e->up_conv(c.key, c.co, c.ci, c.k, c.ci_pad);
            }
            for (int l = 0; l < M_LAYERS; l++) {
                const std::string p = te + std::to_string(l) + ".";
                auto& L = e->el[l];
                L.in_proj = e->up_lin(p + "self_attn.in_proj", 3 * M_DIM, M_DIM); L.out_proj = e->up_lin(p + "self_attn.out_proj", M_DIM, M_DIM);
                L.lin1 = e->up_lin(p + "linear1", M_FF, M_DIM); L.lin2 = e->up_lin(p + "linear2", M_DIM, M_FF);
                L.n1w = e->up_f32(p + "norm1.weight"); L.n1b = e->up_f32(p + "norm1.bias", false);
                L.n2w = e->up_f32(p + "norm2.weight"); L.n2b = e->up_f32(p + "norm2.bias", false);
                L.ls1 = e->up_f32(p + "layer_scale_1.scale"); L.ls2 = e->up_f32(p + "layer_scale_2.scale");
            }
            {   // [1024][512] plain tensor (no .weight suffix), no bias
                const auto* w = e->find(spk_key);
                if ((int64_t)w->f.size() != (int64_t)D_MODEL * M_DIM) { fprintf(stderr, "ptts_b200: error: bad shape for %s\n", spk_key.c_str()); return B200_EINVAL; }
                const auto wb = b200_engine::to_bf16(w->f);
                e->spk.out = D_MODEL; e->spk.in = M_DIM; e->spk.w = e->upload(wb); e->spk.wk = e->upload(tc_kblock_major(wb, D_MODEL, M_DIM));
            }
            e->has_enc = true;
        }
    }
    e->host.clear();

    // ---------------- state + scratch ----------------
    const int S = cfg.max_slots, TS = e->total_slots, cap = cfg.kv_capacity, MR = e->max_rows;
    e->kv_slot_stride = (long long)cap * D_MODEL; e->kv_layer_stride = e->kv_slot_stride * TS;
    const size_t kv_elems = (size_t)e->kv_layer_stride * N_LAYERS;
    if (cfg.kv_f32) { e->kc = e->dalloc<float>(kv_elems); e->vc = e->dalloc<float>(kv_elems); }
    else { e->kc = e->dalloc<__nv_bfloat16>(kv_elems); e->vc = e->dalloc<__nv_bfloat16>(kv_elems); }
    e->mkv_slot_stride = (long long)M_CTX * M_DIM; e->mkv_layer_stride = e->mkv_slot_stride * S;
    e->mkc = e->dalloc<__nv_bfloat16>((size_t)e->mkv_layer_stride * M_LAYERS); e->mvc = e->dalloc<__nv_bfloat16>((size_t)e->mkv_layer_stride * M_LAYERS);
    e->cur_len = e->dalloc<int>(TS); e->mimi_off = e->dalloc<int>(S); e->gen_step = e->dalloc<int>(S); e->eos_step = e->dalloc<int>(S);
    e->max_gen = e->dalloc<int>(S); e->fae = e->dalloc<int>(S); e->active = e->dalloc<int>(S); e->temp = e->dalloc<float>(S);
    { std::vector<unsigned int> ids(S); for (int i = 0; i < S; i++) ids[i] = (unsigned int)i; e->rng_id = e->upload(ids); }
    e->lat_in_bf16 = e->dalloc<__nv_bfloat16>((size_t)S * LDIM); e->lat_f32 = e->dalloc<float>((size_t)S * LDIM);
    e->e_prev = e->dalloc<float>((size_t)S * M_DIM);
    e->h = e->dalloc<float>((size_t)MR * D_MODEL); e->q = e->dalloc<float>((size_t)MR * D_MODEL);
    e->n_bf = e->dalloc<__nv_bfloat16>((size_t)MR * D_MODEL); e->att_bf = e->dalloc<__nv_bfloat16>((size_t)MR * D_MODEL);
    e->ff_bf = e->dalloc<__nv_bfloat16>((size_t)MR * D_FF);
    e->af_ml = e->dalloc<float>((size_t)MR * AF_WS_STRIDE * 32); e->af_acc = e->dalloc<float>((size_t)MR * AF_WS_STRIDE * D_MODEL); e->af_cnt = e->dalloc<int>(MR); e->af_cnt2 = e->dalloc<int>((size_t)MR * N_HEADS);
    e->pfx_slot = e->dalloc<int>(TS); e->pfx_len = e->dalloc<int>(TS);
    e->dec_items_cap = prefix_tiles_capacity(S, e->cfg.max_voices);
    e->dec_items = e->dalloc<AtItem>(e->dec_items_cap); e->dec_meta = e->dalloc<int>(4); e->dec_rows = e->dalloc<int>(S);
    e->pf_barrier = e->dalloc<unsigned int>(4);
    e->tap_up = e->dalloc<float>((size_t)S * M_T * M_DIM);
    e->tap_h = e->dalloc<float>((size_t)N_LAYERS * S * D_MODEL); e->tap_att = e->dalloc<__nv_bfloat16>((size_t)N_LAYERS * S * D_MODEL);
    e->row_slot = e->dalloc<int>(MR); e->row_pos = e->dalloc<int>(MR); e->tok = e->dalloc<int>(MR); e->cs = e->dalloc<float2>((size_t)MR * 32);
    e->c_bf = e->dalloc<__nv_bfloat16>((size_t)S * D_MODEL); e->sy_bf = e->dalloc<__nv_bfloat16>((size_t)S * D_FLOW);
    e->hn_bf = e->dalloc<__nv_bfloat16>((size_t)S * D_FLOW); e->h1_bf = e->dalloc<__nv_bfloat16>((size_t)S * D_FLOW);
    e->eos = e->dalloc<float>(S); e->eos_out = e->dalloc<float>(S); e->mod = e->dalloc<float>((size_t)S * e->ada_all.out); e->xh = e->dalloc<float>((size_t)S * D_FLOW);
    e->noise_f32 = e->dalloc<float>((size_t)S * LDIM); e->noise_inj = e->dalloc<float>((size_t)S * LDIM); e->noise_src = e->noise_inj;
    for (int i = 0; i < 2; i++) e->noise_alt[i] = e->dalloc<float>((size_t)S * LDIM); e->latent = e->dalloc<float>((size_t)S * LDIM);
    e->produced = e->dalloc<int>(S);
    e->d_seed = e->dalloc<unsigned long long>(1);
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->d_seed, &e->seed, sizeof(uint64_t), cudaMemcpyHostToDevice, e->stream));
    const size_t MRm = (size_t)S * M_T;
    e->mx = e->dalloc<float>(MRm * M_DIM); e->mx2[0] = e->dalloc<float>(MRm * M_DIM); e->mx2[1] = e->dalloc<float>(MRm * M_DIM); e->mn_bf = e->dalloc<__nv_bfloat16>(MRm * M_DIM); e->mq_bf = e->dalloc<__nv_bfloat16>(MRm * M_DIM);
    e->matt_bf = e->dalloc<__nv_bfloat16>(MRm * M_DIM); e->mff_bf = e->dalloc<__nv_bfloat16>(MRm * M_FF);
    e->mrow_slot = e->dalloc<int>(MRm); e->mrow_pos = e->dalloc<int>(MRm); e->mcs = e->dalloc<float2>(MRm * 32);
    e->buf0 = e->dalloc<__half>((size_t)S * 22 * 512); e->buf2 = e->dalloc<__half>((size_t)S * 17 * e->C2);
    e->buf3a = e->dalloc<__half>((size_t)S * 98 * 256); e->buf3b = e->dalloc<__half>((size_t)S * 96 * 128);
    e->buf5 = e->dalloc<__half>((size_t)S * 97 * e->C5); e->buf6a = e->dalloc<__half>((size_t)S * 482 * 128);
    e->buf6b = e->dalloc<__half>((size_t)S * 480 * 64); e->buf8 = e->dalloc<__half>((size_t)S * 481 * e->C8);
    e->buf9a = e->dalloc<__half>((size_t)S * 1922 * 64); e->buf9b = e->dalloc<__half>((size_t)S * 1920 * 64);   // 32 channels zero-padded to 64 (K % 64 == 0 for the tensor-core path)
    e->buf11 = e->dalloc<__half>((size_t)S * 1922 * 64);
    e->y3 = e->dalloc<float>((size_t)S * 96 * 256); e->y6 = e->dalloc<float>((size_t)S * 480 * 128); e->y9 = e->dalloc<float>((size_t)S * 1920 * 64);
    e->pcm = e->dalloc<float>((size_t)S * FRAME); e->pcm_out = e->pcm;
    for (int i = 0; i < 2; i++) e->pcm_alt[i] = e->dalloc<float>((size_t)S * FRAME);
    e->shifts.n = 9;
    e->shifts.d[0] = {e->buf0, 22LL * 512, 6, 16, 512};
    e->shifts.d[1] = {e->buf2, 17LL * e->C2, 1, 16, e->C2};
    e->shifts.d[2] = {e->buf3a, 98LL * 256, 2, 96, 256};
    e->shifts.d[3] = {e->buf5, 97LL * e->C5, 1, 96, e->C5};
    e->shifts.d[4] = {e->buf6a, 482LL * 128, 2, 480, 128};
    e->shifts.d[5] = {e->buf8, 481LL * e->C8, 1, 480, e->C8};
    e->shifts.d[6] = {e->buf9a, 1922LL * 64, 2, 1920, 64};
    e->shifts.d[7] = {e->buf11, 1922LL * 64, 2, 1920, 64};
    e->dtail = e->dalloc<float>((size_t)S * 1922 * ST_DROW);
    e->shifts.d[8] = {(__half*)e->dtail, 1922LL * ST_DROW * 2, 2, 1920, ST_DROW * 2};   // f32 rows seen as 16-bit pairs: plain row copies / zeroing
    // Keep the shared-memory carve-out identical for every kernel of the step: mixed carve-outs force an SM reconfiguration
    // between consecutive launches, which shows up as microseconds of idle time on the ~100 small kernels of a frame.
    {
        const void* ks[] = {(const void*)prepare_mimi_kernel, (const void*)rope_table_kernel, (const void*)gemm_ffma_kernel<__nv_bfloat16>, (const void*)gemm_ffma_kernel<__half>,
                            (const void*)gemv_small_kernel<__nv_bfloat16, 8>, (const void*)gemv_small_kernel<__half, 8>, (const void*)gemv_ln_kernel<D_MODEL>, (const void*)gemv_ln_kernel<D_FLOW>, (const void*)layernorm_kernel<D_MODEL>,
                            (const void*)layernorm_kernel<D_FLOW>, 
                            (const void*)splitk_reduce_kernel, (const void*)splitk_reduce_ln_kernel<1024>, (const void*)splitk_reduce_ln_kernel<512>,
                            (const void*)attn_flow_split_kernel<__nv_bfloat16>, (const void*)attn_flow_split_kernel<float>, (const void*)attn_tile_kernel<2>, (const void*)attn_tile_kernel<1>, (const void*)attn_tile_kernel<0>, (const void*)attn_merge_kernel, (const void*)flow_persistent_kernel, (const void*)noise_inproj_kernel, (const void*)flow_in_kernel, (const void*)head_pre_kernel,
                            (const void*)step_front_kernel, (const void*)mimi_front_kernel, (const void*)attn_mimi_kernel, (const void*)attn_mimi_mma4_kernel,
                            (const void*)conv_n1_kernel, (const void*)shift_states_kernel};
        for (const void* k : ks) PTTS_CUDA_CHECK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(attn_mimi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AM_SMEM));
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(attn_flow_split_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, AfCfg<__nv_bfloat16>::SMEM));
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(attn_flow_split_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, AfCfg<float>::SMEM));
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(flow_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PF_SMEM_BYTES));
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(head_res_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HF_SMEM_BYTES));
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(seanet_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ST_SMEM_BYTES));
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(seanet_res_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SR_SMEM_BYTES));
    PTTS_CUDA_CHECK(cudaFuncSetAttribute(attn_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AW_SMEM));
    e->actx.row_slot = e->row_slot; e->actx.row_pos = e->row_pos; e->actx.cs = e->cs;
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    e->finalized = true;
    return B200_OK;
}

// ---- ragged FlowLM prefill (reference _run_flow_lm with T > 1, src/pocket_tts.cpp:40-98): rows = (slot, position, token | voice row), slot-major
//      with ascending positions. Everything is staged once (pinned ring -> device) and enqueued without a host synchronisation; the rows are
//      processed in chunks of max_prefill_rows (a later chunk of a sentence attends to the cache rows the earlier chunk appended). ----
// x_host / x_dev: the rows' input vectors [total][1024] on the host (staged through the pinned ring) or already on the device.
static void prefill_rows(b200_engine* e, const std::vector<int>& slots, const std::vector<int>& pos, const std::vector<int>* tokens, const float* x_host,
                         const float* x_dev = nullptr) {
    NvtxRange nvtx_range("ptts.prefill_rows");
    const int total = (int)slots.size(), MRp = e->cfg.max_prefill_rows;
    if (total == 0) return;
    const int nchunks = (total + MRp - 1) / MRp;
    // tensor-core tile work list (bf16 cache): one item per run of <= 64 consecutive positions of one slot inside a chunk
    std::vector<AtItem> items; std::vector<int> chunk_item0(nchunks + 1, 0);
    if (!e->cfg.kv_f32) plan_prefill_items(slots.data(), pos.data(), total, MRp, e->h_pfx_slot.data(), e->h_pfx_len.data(), items, chunk_item0);
    e->grow(e->pf_int, e->pf_int_cap, (size_t)3 * total);
    e->grow(e->pf_items, e->pf_items_cap, items.size() + 1);
    e->grow(e->pf_meta, e->pf_meta_cap, (size_t)4 * nchunks);
    if (x_host) e->grow(e->pf_x, e->pf_x_cap, (size_t)total * D_MODEL);
    const size_t b_int = (size_t)3 * total * sizeof(int), b_meta = (size_t)4 * nchunks * sizeof(int), b_items = items.size() * sizeof(AtItem);
    const size_t b_x = x_host ? (size_t)total * D_MODEL * sizeof(float) : 0;
    char* pb = (char*)e->pin_acquire(b_int + b_meta + b_items + b_x + 256);
    int* pi = (int*)pb;
    for (int i = 0; i < total; i++) { pi[i] = slots[i]; pi[total + i] = pos[i]; pi[2 * total + i] = tokens ? (*tokens)[i] : 0; }
    int* pm = pi + 3 * total;
    for (int c = 0; c < nchunks; c++) { pm[4 * c] = chunk_item0[c + 1] - chunk_item0[c]; pm[4 * c + 1] = 0; pm[4 * c + 2] = 0; pm[4 * c + 3] = 0; }
    char* pit = (char*)(pm + 4 * nchunks);
    if (b_items) memcpy(pit, items.data(), b_items);
    char* px = pit + ((b_items + 15) / 16) * 16;
    if (x_host) memcpy(px, x_host, b_x);
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_int, pi, b_int, cudaMemcpyHostToDevice, e->stream));
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_meta, pm, b_meta, cudaMemcpyHostToDevice, e->stream));
    if (b_items) PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_items, pit, b_items, cudaMemcpyHostToDevice, e->stream));
    if (x_host) PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_x, px, b_x, cudaMemcpyHostToDevice, e->stream));
    e->pin_release(e->stream);
    e->set_pdl(false);
    e->tc->tma_epilogue = false;                                  // the Mimi stream may be running beside the prefill
    const b200_engine::AttnCtx saved = e->actx;
    for (int c = 0; c < nchunks; c++) {
        const int r0 = c * MRp, R = std::min(MRp, total - r0);
        e->prefill_chunk(c, r0, total, chunk_item0);
        if (tokens) {
            launch_k(false, embed_gather_kernel, dim3(R), dim3(256), (size_t)(0), e->stream, e->embed, (const int*)(e->pf_int + 2 * total + r0), e->h, R);
            e->launches++;
        } else {
            PTTS_CUDA_CHECK(cudaMemcpyAsync(e->h, (x_dev ? x_dev : e->pf_x) + (size_t)r0 * D_MODEL, (size_t)R * D_MODEL * sizeof(float), cudaMemcpyDeviceToDevice, e->stream));
        }
        launch_k(false, rope_table_kernel, dim3((R * 32 + 255) / 256), dim3(256), (size_t)(0), e->stream, e->actx.row_pos, e->freq_flow, e->cs, R);
        e->launches++;
        e->flow_forward(R);
    }
    e->actx = saved;
}

int b200_voice_create(b200_engine* e, const float* audio_prompt, int T) {
    NvtxRange nvtx_range("ptts.voice_create");
    if (!e || !e->finalized || T < 0 || (T > 0 && !audio_prompt)) return B200_EINVAL;
    if (e->n_voices >= e->cfg.max_voices) return B200_ECAPACITY;
    if (T > e->cfg.kv_capacity) return B200_ECAPACITY;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    const int v = e->n_voices++;
    const int slot = e->cfg.max_slots + v;
    std::vector<int> slots(T, slot), pos(T);
    for (int i = 0; i < T; i++) pos[i] = i;
    if (T > 0) prefill_rows(e, slots, pos, nullptr, audio_prompt);
    e->voice_len[v] = T;
    return v;
}

int b200_has_encoder(b200_engine* e) { return e && e->finalized && e->has_enc ? 1 : 0; }

// Voice cloning: uploads the PCM through the pinned ring and enqueues the encoder on the main stream (no host wait). Returns T.
static int enc_enqueue(b200_engine* e, const float* pcm, long long n) {
    if (!e || !e->finalized || !pcm || n < 1) return B200_EINVAL;
    if (!e->has_enc) return B200_ENOTFOUND;
    const long long T = (n + ENC_HOP - 1) / ENC_HOP;
    if (T > e->cfg.kv_capacity) return B200_ECAPACITY;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->enc_reserve((int)T);
    const long long L0 = T * ENC_HOP;
    if (!e->enc_pin_ev) PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&e->enc_pin_ev, cudaEventDisableTiming));
    if (e->enc_pin_used) PTTS_CUDA_CHECK(cudaEventSynchronize(e->enc_pin_ev));   // the previous clone's upload (long done in steady state)
    if (e->enc_pin_cap < (size_t)n) {
        if (e->enc_pin) PTTS_CUDA_CHECK(cudaFreeHost(e->enc_pin));
        e->enc_pin_cap = (size_t)e->eb.T * ENC_HOP;
        PTTS_CUDA_CHECK(cudaMallocHost(&e->enc_pin, e->enc_pin_cap * sizeof(float)));
    }
    memcpy(e->enc_pin, pcm, (size_t)n * sizeof(float));
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->eb.pcm + 6, e->enc_pin, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    PTTS_CUDA_CHECK(cudaEventRecord(e->enc_pin_ev, e->stream));
    e->enc_pin_used = true;
    if (L0 > n) PTTS_CUDA_CHECK(cudaMemsetAsync(e->eb.pcm + 6 + n, 0, (size_t)(L0 - n) * sizeof(float), e->stream));
    e->encode((int)T);
    return (int)T;
}

int b200_voice_embed_audio(b200_engine* e, const float* pcm, long long n, float* out) {
    NvtxRange nvtx_range("ptts.voice_embed_audio");
    const int T = enc_enqueue(e, pcm, n);
    if (T < 0 || !out) return T;
    PTTS_CUDA_CHECK(cudaMemcpyAsync(out, e->eb.prompt, (size_t)T * D_MODEL * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    return T;
}

int b200_voice_create_from_audio(b200_engine* e, const float* pcm, long long n) {
    NvtxRange nvtx_range("ptts.voice_create_from_audio");
    if (e && e->finalized && e->has_enc && pcm && n >= 1 && e->n_voices >= e->cfg.max_voices) return B200_ECAPACITY;
    const int T = enc_enqueue(e, pcm, n);
    if (T < 0) return T;
    const int v = e->n_voices++;
    const int slot = e->cfg.max_slots + v;
    std::vector<int> slots(T, slot), pos(T);
    for (int i = 0; i < T; i++) pos[i] = i;
    prefill_rows(e, slots, pos, nullptr, nullptr, e->eb.prompt);
    e->voice_len[v] = T;
    return v;
}

int b200_begin_sentences(b200_engine* e, int n, const int32_t* slots, const int32_t* voices, const int32_t* tokens,
                         const int32_t* tok_off, const int32_t* max_gen_len, const int32_t* frames_after_eos, const float* temp) {
    return b200_begin_sentences_ex(e, n, slots, voices, tokens, tok_off, max_gen_len, frames_after_eos, temp, nullptr);
}

int b200_begin_sentences_ex(b200_engine* e, int n, const int32_t* slots, const int32_t* voices, const int32_t* tokens, const int32_t* tok_off,
                            const int32_t* max_gen_len, const int32_t* frames_after_eos, const float* temp, const uint32_t* rng_stream) {
    NvtxRange nvtx_range("ptts.begin_sentences");
    if (!e || !e->finalized || n < 0) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    std::vector<int> rs, rp, rt;
    for (int i = 0; i < n; i++) {
        const int slot = slots[i], v = voices[i];
        if (slot < 0 || slot >= e->cfg.max_slots || v < 0 || v >= e->n_voices) return B200_EINVAL;
        const int nt = tok_off[i + 1] - tok_off[i];
        const int start = e->voice_len[v];
        if (nt < 0 || start + nt >= e->cfg.kv_capacity) return B200_ECAPACITY;
        for (int t = 0; t < nt; t++) {
            const int id = tokens[tok_off[i] + t];
            if (id < 0 || id >= e->n_embed) return B200_EINVAL;
            rs.push_back(slot); rp.push_back(start + t); rt.push_back(id);
        }
    }
    if (n == 0) return B200_OK;
    // A frame of these slots whose Mimi decode is still waiting for an interleaving partner must be decoded BEFORE the Mimi-state reset
    // below (it belongs to the previous sentence). Nothing here waits on the host: uploads go through the pinned ring.
    e->flush_pending();
    // the previous call's Mimi-side reset reads the device copy of ITS metadata, which the upload below overwrites
    if (e->begin_used) PTTS_CUDA_CHECK(cudaStreamWaitEvent(e->stream, e->ev_reset, 0));
    e->begin_used = true;
    const size_t elt = e->cfg.kv_f32 ? 4 : 2;
    // per-sentence metadata in one upload: [slot | src voice slot | prefix rows | cur_len | max_gen | frames_after_eos | shared rows] x n, then temps
    int* pm = (int*)e->pin_acquire((size_t)9 * n * sizeof(int));
    float* pt = (float*)(pm + 8 * n);
    int max_copy = 0;
    for (int i = 0; i < n; i++) {
        const int slot = slots[i], v = voices[i];
        const int nt = tok_off[i + 1] - tok_off[i];
        const int start = e->voice_len[v];
        // KV capacity guard (the reference has none: 1000 rows, no bounds check, src/pocket_tts.cpp:367): clamp the cap so that the last
        // appended row is capacity-1; finished slots are dead rows on the device and never append (flow_in_kernel).
        int mg = max_gen_len[i];
        const int room = e->cfg.kv_capacity - (start + nt);
        if (mg > room) mg = room;
        const int shared = e->cfg.prefix_share ? start : 0;
        pm[i] = slot; pm[n + i] = e->cfg.max_slots + v; pm[2 * n + i] = start; pm[3 * n + i] = start + nt;
        pm[4 * n + i] = mg; pm[5 * n + i] = frames_after_eos[i]; pm[6 * n + i] = shared; pm[7 * n + i] = (int)(rng_stream ? rng_stream[i] : (uint32_t)slot);
        pt[i] = temp[i];
        e->h_cur_len[slot] = start + nt;
        if (e->h_pfx_slot[slot] != e->cfg.max_slots + v || e->h_pfx_len[slot] != shared) { e->h_pfx_slot[slot] = e->cfg.max_slots + v; e->h_pfx_len[slot] = shared; e->pfx_version++; }
        if (!e->cfg.prefix_share) max_copy = std::max(max_copy, start);
    }
    if ((size_t)n > e->begin_cap) {
        e->begin_meta = e->dalloc<int>((size_t)8 * n, false); e->begin_temp = e->dalloc<float>((size_t)n, false); e->begin_cap = n;
    }
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->begin_meta, pm, (size_t)8 * n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->begin_temp, pt, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    e->pin_release(e->stream);
    if (max_copy > 0)   // reference semantics (prefix_share = 0): private copy of the voice-conditioned prefix, models/flow_lm.h:70-78
        launch_k(false, begin_copy_prefix_kernel, dim3(8, 2 * N_LAYERS, n), dim3(256), (size_t)0, e->stream, n, (const int*)e->begin_meta, (char*)e->kc, (char*)e->vc,
                 (long long)(e->kv_slot_stride * elt), (long long)(e->kv_layer_stride * elt), (long long)(D_MODEL * elt));
    launch_k(false, begin_meta_kernel, dim3(n), dim3(128), (size_t)0, e->stream, n, (const int*)e->begin_meta, (const float*)e->begin_temp, (const float*)e->d_bos, e->cur_len,
             e->gen_step, e->eos_step, e->max_gen, e->fae, e->active, e->temp, e->lat_in_bf16, e->lat_f32, e->pfx_slot, e->pfx_len, e->e_prev, e->rng_id);
    // Mimi-side reset on the Mimi stream: behind every Mimi decode already enqueued there, ahead of the new sentences' first decode. The
    // main stream only waits for it when it touches Mimi state itself (join_mimi: synchronous b200_step, Mimi-only calls).
    PTTS_CUDA_CHECK(cudaEventRecord(e->ev_begin, e->stream));
    PTTS_CUDA_CHECK(cudaStreamWaitEvent(e->stream_m, e->ev_begin, 0));
    launch_k(false, begin_reset_kernel, dim3(n, e->shifts.n), dim3(256), (size_t)0, e->stream_m, n, (const int*)e->begin_meta, e->shifts, e->mimi_off);
    PTTS_CUDA_CHECK(cudaEventRecord(e->ev_reset, e->stream_m));
    e->reset_pending = true;
    e->launches += 3;
    if (!rs.empty()) prefill_rows(e, rs, rp, &rt, nullptr);
    return B200_OK;
}

// Retires slots: the next step sees them as dead rows (flow_in_kernel: no KV append, no attention; step_front_kernel: produced = 0, position
// kept), exactly like a slot whose sentence reached EOS. The slot list goes through the pinned ring, so the call never waits on the host.
int b200_end_sentences(b200_engine* e, int n, const int32_t* slots) {
    NvtxRange nvtx_range("ptts.end_sentences");
    if (!e || !e->finalized || n < 0 || (n > 0 && !slots)) return B200_EINVAL;
    for (int i = 0; i < n; i++) if (slots[i] < 0 || slots[i] >= e->cfg.max_slots) return B200_EINVAL;
    if (n == 0) return B200_OK;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->grow(e->end_slots, e->end_slots_cap, (size_t)n);
    int* ps = (int*)e->pin_acquire((size_t)n * sizeof(int));
    memcpy(ps, slots, (size_t)n * sizeof(int));
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->end_slots, ps, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
    e->pin_release(e->stream);
    launch_k(false, end_slots_kernel, dim3((n + 127) / 128), dim3(128), (size_t)0, e->stream, n, (const int*)e->end_slots, e->active);
    e->launches++;
    return B200_OK;
}

int b200_voice_len(b200_engine* e, int voice) { return (!e || voice < 0 || voice >= e->n_voices) ? B200_EINVAL : e->voice_len[voice]; }
int b200_kv_capacity(b200_engine* e) { return e ? e->cfg.kv_capacity : B200_EINVAL; }
int b200_max_slots(b200_engine* e) { return e ? e->cfg.max_slots : B200_EINVAL; }

int b200_begin_sentence(b200_engine* e, int slot, int voice, const int32_t* tokens, int n_tokens, int max_gen_len, int frames_after_eos, float temp) {
    const int32_t off[2] = {0, n_tokens};
    return b200_begin_sentences(e, 1, &slot, &voice, tokens, off, &max_gen_len, &frames_after_eos, &temp);
}

int b200_step_enqueue(b200_engine* e, int slot0, int n, int use_injected_noise) {
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->run_step(slot0, n, use_injected_noise != 0);
    return B200_OK;
}

// `count` consecutive steps enqueued by one native call (no host-language overhead between them).
int b200_steps_enqueue(b200_engine* e, int slot0, int n, int count) {
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots || count < 0) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    for (int i = 0; i < count; i++) e->run_step(slot0, n, false);
    return B200_OK;
}

int b200_sync(b200_engine* e) {
    if (!e) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->flush_pending();                                      // a frame whose Mimi decode was waiting for an interleaving partner
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream_m));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream_c));
    PTTS_CUDA_CHECK(cudaGetLastError());
    return B200_OK;
}

// Makes the main stream wait for all Mimi-stream work enqueued so far (so that an event recorded on b200_stream() afterwards covers
// the complete frames, PCM included). Costs nothing when the pipeline is idle.
int b200_join(b200_engine* e) {
    if (!e) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->join_mimi();
    return B200_OK;
}

int b200_step(b200_engine* e, int slot0, int n, const float* noise, float* pcm, int32_t* produced, float* latents, float* eos_logit) {
    NvtxRange nvtx_range("ptts.step");
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots || !pcm || !produced) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->ensure_pinned((size_t)n * (FRAME + 2 * LDIM + 1), (size_t)std::max(n, 16) * 3);
    float* p_noise = e->pin_f; float* p_pcm = e->pin_f + (size_t)n * LDIM; float* p_lat = p_pcm + (size_t)n * FRAME; float* p_eos = p_lat + (size_t)n * LDIM;
    if (noise) {
        memcpy(p_noise, noise, (size_t)n * LDIM * sizeof(float));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(e->noise_inj, p_noise, (size_t)n * LDIM * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    }
    // synchronous API: this frame's PCM is returned by this call, so there is nothing to overlap - replay the whole step as ONE graph
    // on the main stream (13 graph launches + events per frame would only add host latency, which is what batch-1 streaming feels)
    e->join_mimi();
    e->prepare_decode(slot0, n);
    e->tap_slot0 = slot0; e->tap_n = n;
    e->run_graphed(0, slot0, n, noise != nullptr);
    PTTS_CUDA_CHECK(cudaMemcpyAsync(p_pcm, e->pcm + (size_t)slot0 * FRAME, (size_t)n * FRAME * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pin_i, e->produced, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    if (latents) PTTS_CUDA_CHECK(cudaMemcpyAsync(p_lat, e->latent, (size_t)n * LDIM * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    if (eos_logit) PTTS_CUDA_CHECK(cudaMemcpyAsync(p_eos, e->eos_out, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    memcpy(pcm, p_pcm, (size_t)n * FRAME * sizeof(float));
    for (int i = 0; i < n; i++) { produced[i] = e->pin_i[i]; }
    if (latents) memcpy(latents, p_lat, (size_t)n * LDIM * sizeof(float));
    if (eos_logit) memcpy(eos_logit, p_eos, (size_t)n * sizeof(float));
    return B200_OK;
}

// Pipelined form of b200_step for throughput serving: b200_submit(t) enqueues frame t (H2D noise, FlowLM part on the main stream, Mimi
// body on the Mimi stream, D2H of PCM / flags into pinned staging) and returns immediately; b200_collect() blocks until the OLDEST
// submitted frame is complete and copies it out. At most three frames may be in flight (submit returns B200_ESTATE otherwise): the Mimi
// decode of frame t is interleaved with the FlowLM step of frame t+1 (run_step), so a caller that keeps two submits ahead of its
// collects never leaves the GPU waiting for the host. Frames come back in submission order.
int b200_submit(b200_engine* e, int slot0, int n, const float* noise) {
    NvtxRange nvtx_range("ptts.submit");
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots) return B200_EINVAL;
    if (e->submit_t - e->collect_t >= 3) return B200_ESTATE;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    auto& pd = e->pend[e->submit_t & 3];
    if (pd.cap < (size_t)n) {
        if (pd.noise) cudaFreeHost(pd.noise); if (pd.pcm) cudaFreeHost(pd.pcm); if (pd.produced) cudaFreeHost(pd.produced);
        PTTS_CUDA_CHECK(cudaMallocHost(&pd.noise, (size_t)n * LDIM * sizeof(float)));
        PTTS_CUDA_CHECK(cudaMallocHost(&pd.pcm, (size_t)n * FRAME * sizeof(float)));
        PTTS_CUDA_CHECK(cudaMallocHost(&pd.produced, (size_t)n * sizeof(int)));
        pd.cap = n;
    }
    if (!pd.done_main) { PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&pd.done_main, cudaEventDisableTiming)); PTTS_CUDA_CHECK(cudaEventCreateWithFlags(&pd.done_mimi, cudaEventDisableTiming)); }
    if (noise) {
        memcpy(pd.noise, noise, (size_t)n * LDIM * sizeof(float));
        if (e->cfg.overlap && e->cfg.cuda_graphs && !e->profiling && !e->taps_on) {       // the step will be pipelined with parity pipe_t & 1 (run_step)
            const int par = (int)(e->pipe_t & 1);
            PTTS_CUDA_CHECK(cudaStreamWaitEvent(e->stream_n, e->ev_main[par], 0));         // frame t-2 has read this buffer
            PTTS_CUDA_CHECK(cudaMemcpyAsync(e->noise_alt[par], pd.noise, (size_t)n * LDIM * sizeof(float), cudaMemcpyHostToDevice, e->stream_n));
            PTTS_CUDA_CHECK(cudaEventRecord(e->ev_noise[par], e->stream_n));
            PTTS_CUDA_CHECK(cudaStreamWaitEvent(e->stream, e->ev_noise[par], 0));
            e->noise_src = e->noise_alt[par];
        } else {
            PTTS_CUDA_CHECK(cudaMemcpyAsync(e->noise_inj, pd.noise, (size_t)n * LDIM * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        }
    }
    e->run_step(slot0, n, noise != nullptr, (long long)e->submit_t);
    e->noise_src = e->noise_inj;
    PTTS_CUDA_CHECK(cudaMemcpyAsync(pd.produced, e->produced, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    PTTS_CUDA_CHECK(cudaEventRecord(pd.done_main, e->stream));
    if (!e->last_step_piped) {   // non-pipelined step (overlap off): the frame is already decoded on the main stream
        PTTS_CUDA_CHECK(cudaMemcpyAsync(pd.pcm, e->pcm + (size_t)slot0 * FRAME, (size_t)n * FRAME * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        PTTS_CUDA_CHECK(cudaEventRecord(pd.done_mimi, e->stream));
    }   // otherwise the PCM copy is enqueued behind the frame's Mimi decode (finish_mimi_frame), by the next submit or by collect
    pd.slot0 = slot0; pd.n = n; pd.busy = true; e->submit_t++;
    return B200_OK;
}

int b200_collect(b200_engine* e, float* pcm, int32_t* produced) {
    NvtxRange nvtx_range("ptts.collect");
    if (!e || !pcm || !produced) return B200_EINVAL;
    if (e->collect_t == e->submit_t) return B200_ESTATE;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    auto& pd = e->pend[e->collect_t & 3];
    if (e->pending.valid && e->pending.tag == (long long)e->collect_t) e->flush_pending();   // nobody submitted after it: decode it now
    PTTS_CUDA_CHECK(cudaEventSynchronize(pd.done_main));
    PTTS_CUDA_CHECK(cudaEventSynchronize(pd.done_mimi));
    memcpy(pcm, pd.pcm, (size_t)pd.n * FRAME * sizeof(float));
    memcpy(produced, pd.produced, (size_t)pd.n * sizeof(int));
    pd.busy = false; e->collect_t++;
    return pd.n;
}

int b200_mimi_reset(b200_engine* e, int slot0, int n) {
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->join_mimi();
    for (int s = slot0; s < slot0 + n; s++) launch_k(false, reset_slot_kernel, dim3(1, e->shifts.n), dim3(256), (size_t)(0), e->stream, e->shifts, s, e->e_prev, e->mimi_off);
    e->launches += n;
    return B200_OK;
}

int b200_mimi_decode_enqueue(b200_engine* e, int slot0, int n) {
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->join_mimi();
    e->run_graphed(1, slot0, n, false);
    return B200_OK;
}

int b200_mimi_decode(b200_engine* e, int slot0, int n, const float* latents, float* pcm) {
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots || !latents || !pcm) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->join_mimi();
    e->ensure_pinned((size_t)n * (FRAME + LDIM), 16);
    memcpy(e->pin_f, latents, (size_t)n * LDIM * sizeof(float));
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->lat_f32 + (size_t)slot0 * LDIM, e->pin_f, (size_t)n * LDIM * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    e->run_graphed(1, slot0, n, false);
    float* p_pcm = e->pin_f + (size_t)n * LDIM;
    PTTS_CUDA_CHECK(cudaMemcpyAsync(p_pcm, e->pcm + (size_t)slot0 * FRAME, (size_t)n * FRAME * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    memcpy(pcm, p_pcm, (size_t)n * FRAME * sizeof(float));
    return B200_OK;
}

void b200_set_seed(b200_engine* e, uint64_t seed) {
    if (!e || (e->seed == seed && e->d_seed)) return;
    e->seed = seed;
    if (e->d_seed) {   // device-resident so that captured graphs see later seeds
        PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
        PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
        PTTS_CUDA_CHECK(cudaMemcpy(e->d_seed, &e->seed, sizeof(uint64_t), cudaMemcpyHostToDevice));
    }
}

int b200_slot_position(b200_engine* e, int slot) {
    if (!e || slot < 0 || slot >= e->cfg.max_slots) return B200_EINVAL;
    int v = 0;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    PTTS_CUDA_CHECK(cudaMemcpy(&v, e->cur_len + slot, sizeof(int), cudaMemcpyDeviceToHost));
    return v;
}

int b200_debug_set_position(b200_engine* e, int slot0, int n, int pos, int max_gen_len) {
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots || pos < 0 || pos + max_gen_len > e->cfg.kv_capacity) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->join_mimi();
    const float* bos = e->d_bos;
    for (int s = slot0; s < slot0 + n; s++) {
        launch_k(false, reset_slot_kernel, dim3(1, e->shifts.n), dim3(256), (size_t)(0), e->stream, e->shifts, s, e->e_prev, e->mimi_off);
        launch_k(false, set_meta_kernel, dim3(1), dim3(32), (size_t)(0), e->stream, s, pos, max_gen_len, 1 << 28, 0.f, bos, e->cur_len, e->gen_step, e->eos_step, e->max_gen, e->fae, e->active,
                                                 e->temp, e->lat_in_bf16, e->lat_f32);
    }
    e->launches += 2 * n;
    return B200_OK;
}

// Unit-test hook for the GEMM family: C[n_slots*T][N] = windows(A)[.][taps*C] . W[N][taps*C]^T (+bias, optional ELU->f16 copy)
// A is [n_slots][rows_buf][C] (f32 on the host, rounded to bf16/f16 here). path: 0 = dispatcher (tcgen05 when supported),
// 1 = CUDA-core. Returns 1 if the tensor-core kernel was used, 0 if a CUDA-core kernel was, negative on error.
int b200_debug_gemm(b200_engine* e, int f16, const float* A, int n_slots, int rows_buf, int C, int T, int taps, const float* W, int N,
                    const float* bias, int path, float* out, float* out2_as_f32) {
    if (!e || !A || !W || !out || n_slots < 1 || T < 1 || rows_buf < T + taps - 1) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    const int R = n_slots * T, K = taps * C;
    const size_t na = (size_t)n_slots * rows_buf * C, nw = (size_t)N * K;
    void *dA, *dW; float *dO, *dB = nullptr; void* dO2;
    PTTS_CUDA_CHECK(cudaMalloc(&dA, na * 2)); PTTS_CUDA_CHECK(cudaMalloc(&dW, nw * 2));
    PTTS_CUDA_CHECK(cudaMalloc(&dO, (size_t)R * N * 4)); PTTS_CUDA_CHECK(cudaMalloc(&dO2, (size_t)R * N * 2));
    std::vector<uint16_t> ha(na), hw(nw);
    auto cvt = [&](float v) -> uint16_t { if (f16) { __half h = __float2half_rn(v); return *(uint16_t*)&h; } __nv_bfloat16 b = __float2bfloat16_rn(v); return *(uint16_t*)&b; };
    for (size_t i = 0; i < na; i++) ha[i] = cvt(A[i]);
    for (size_t i = 0; i < nw; i++) hw[i] = cvt(W[i]);
    PTTS_CUDA_CHECK(cudaMemcpy(dA, ha.data(), na * 2, cudaMemcpyHostToDevice));
    PTTS_CUDA_CHECK(cudaMemcpy(dW, hw.data(), nw * 2, cudaMemcpyHostToDevice));
    if (bias) { PTTS_CUDA_CHECK(cudaMalloc(&dB, N * 4)); PTTS_CUDA_CHECK(cudaMemcpy(dB, bias, N * 4, cudaMemcpyHostToDevice)); }
    Epi ep; ep.rps = T; ep.bias = dB; ep.out = dO; ep.out_map = b200_engine::smap((long long)T * N, N, 0);
    if (out2_as_f32) { ep.out2 = dO2; ep.out2_map = ep.out_map; ep.out2_type = f16 ? OUT2_F16 : OUT2_BF16; ep.act = ACT_ELU; }
    const RowMap am = (n_slots == 1 && taps == 1) ? b200_engine::rows(C) : b200_engine::smap((long long)rows_buf * C, C, 0);
    const int rps = (n_slots == 1 && taps == 1) ? (1 << 30) : T;
    const int saved = e->cfg.gemm_path; e->cfg.gemm_path = path;
    e->set_pdl(false);
    int used_tc = 0;
    void* dWk = nullptr;
    if (K % 64 == 0) {
        const std::vector<uint16_t> hk = tc_kblock_major(hw, N, K);
        PTTS_CUDA_CHECK(cudaMalloc(&dWk, nw * 2)); PTTS_CUDA_CHECK(cudaMemcpy(dWk, hk.data(), nw * 2, cudaMemcpyHostToDevice));
    }
    if (f16) { used_tc = (path == 0 && dWk && tc_gemm_supported<__half>(R, N, K, am, rps, ep)); e->gemm<__half>((const __half*)dA, am, rps, (const __half*)dW, (const __half*)dWk, R, N, K, ep); }
    else { used_tc = (path == 0 && dWk && tc_gemm_supported<__nv_bfloat16>(R, N, K, am, rps, ep)); e->gemm<__nv_bfloat16>((const __nv_bfloat16*)dA, am, rps, (const __nv_bfloat16*)dW, (const __nv_bfloat16*)dWk, R, N, K, ep); }
    e->cfg.gemm_path = saved;
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    PTTS_CUDA_CHECK(cudaGetLastError());
    PTTS_CUDA_CHECK(cudaMemcpy(out, dO, (size_t)R * N * 4, cudaMemcpyDeviceToHost));
    if (out2_as_f32) {
        std::vector<uint16_t> h2((size_t)R * N);
        PTTS_CUDA_CHECK(cudaMemcpy(h2.data(), dO2, h2.size() * 2, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < h2.size(); i++) out2_as_f32[i] = f16 ? __half2float(*(__half*)&h2[i]) : __bfloat162float(*(__nv_bfloat16*)&h2[i]);
    }
    cudaFree(dA); cudaFree(dW); cudaFree(dO); cudaFree(dO2); if (dB) cudaFree(dB); if (dWk) cudaFree(dWk);
    return used_tc;
}

// Parity helper: overwrite the backbone input (previous latent) of slots [slot0, slot0+n) — teacher forcing.
int b200_debug_set_latent(b200_engine* e, int slot0, int n, const float* latents) {
    if (!e || !e->finalized || slot0 < 0 || n < 1 || slot0 + n > e->cfg.max_slots || !latents) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    std::vector<__nv_bfloat16> b((size_t)n * LDIM);
    for (size_t i = 0; i < b.size(); i++) b[i] = __float2bfloat16_rn(latents[i]);
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    PTTS_CUDA_CHECK(cudaMemcpy(e->lat_f32 + (size_t)slot0 * LDIM, latents, (size_t)n * LDIM * sizeof(float), cudaMemcpyHostToDevice));
    PTTS_CUDA_CHECK(cudaMemcpy(e->lat_in_bf16 + (size_t)slot0 * LDIM, b.data(), b.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice));
    return B200_OK;
}

// Per-segment device timing. b200_profile(e,1) arms it; after b200_sync, b200_profile_read sums the recorded event
// pairs per category: 0 FlowLM attention streaming kernel, 1 FlowLM backbone, 2 head, 3 Mimi transformer, 4 SEANet, 5 whole step,
// 6 FlowLM shared-prefix tile kernel. out_ms[7], out_count[7]. Reading disarms and clears.
int b200_profile(b200_engine* e, int on) {
    if (!e) return B200_EINVAL;
    e->profiling = on != 0; e->segs.clear(); e->ev_used = 0;
    return B200_OK;
}
int b200_profile_read(b200_engine* e, float* out_ms, int* out_count) {
    if (!e || !out_ms || !out_count) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    for (int i = 0; i < 7; i++) { out_ms[i] = 0.f; out_count[i] = 0; }
    for (auto& sg : e->segs) {
        float ms = 0.f;
        PTTS_CUDA_CHECK(cudaEventElapsedTime(&ms, sg.a, sg.b));
        if (sg.cat >= 0 && sg.cat < 7) { out_ms[sg.cat] += ms; out_count[sg.cat]++; }
    }
    e->profiling = false; e->segs.clear(); e->ev_used = 0;
    return B200_OK;
}

// cudaProfilerStart/Stop, so that `ncu --profile-from-start off` captures only the bracketed region.
void b200_profiler_range(int start) { if (start) cudaProfilerStart(); else cudaProfilerStop(); }

void* b200_stream(b200_engine* e) { return e ? (void*)e->stream : nullptr; }

// Debug read of a named f32 device buffer (see b200_device_ptr) after a full synchronisation: out[n] = buffer[offset .. offset+n).
int b200_debug_read_f32(b200_engine* e, const char* name, long long offset, float* out, int n) {
    float* p = (float*)b200_device_ptr(e, name);
    if (!p || !out || n < 0 || offset < 0 || std::string(name) == "produced") return B200_EINVAL;
    b200_sync(e);
    PTTS_CUDA_CHECK(cudaMemcpy(out, p + offset, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    return B200_OK;
}

void* b200_device_ptr(b200_engine* e, const char* name) {
    if (!e || !name) return nullptr;
    const std::string s = name;
    if (s == "pcm") return e->pcm;
    if (s == "latent") return e->latent;
    if (s == "noise") return e->noise_inj;
    if (s == "produced") return e->produced;
    if (s == "eos") return e->eos_out;
    if (s == "lat_f32") return e->lat_f32;
    if (s == "noise_drawn") return e->noise_f32;
    return nullptr;
}

long long b200_launch_count(b200_engine* e) { return e ? e->launches : 0; }

// Logical cache rows [0, n_pos) of a slot: with a shared voice prefix the first rows come from the voice's resident copy.
int b200_read_kv(b200_engine* e, int slot, int layer, int which, int n_pos, float* out) {
    if (!e || !e->finalized || slot < 0 || slot >= e->total_slots || layer < 0 || layer >= N_LAYERS || n_pos < 0 || n_pos > e->cfg.kv_capacity) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    const int P = std::min(n_pos, e->h_pfx_len[slot]);
    for (int part = 0; part < 2; part++) {
        const int r0 = part == 0 ? 0 : P, r1 = part == 0 ? P : n_pos, src_slot = part == 0 ? e->h_pfx_slot[slot] : slot;
        if (r1 <= r0) continue;
        const size_t n = (size_t)(r1 - r0) * D_MODEL;
        const long long off = layer * e->kv_layer_stride + src_slot * e->kv_slot_stride + (long long)r0 * D_MODEL;
        float* dst = out + (size_t)r0 * D_MODEL;
        if (e->cfg.kv_f32) {
            PTTS_CUDA_CHECK(cudaMemcpy(dst, (const float*)(which ? e->vc : e->kc) + off, n * 4, cudaMemcpyDeviceToHost));
        } else {
            std::vector<uint16_t> tmp(n);
            PTTS_CUDA_CHECK(cudaMemcpy(tmp.data(), (const __nv_bfloat16*)(which ? e->vc : e->kc) + off, n * 2, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < n; i++) { uint32_t u = (uint32_t)tmp[i] << 16; memcpy(&dst[i], &u, 4); }
        }
    }
    return B200_OK;
}

// Test hook: physical cache rows [pos0, pos0 + n) of a slot (no prefix redirection), from f32 rows [n][1024] rounded to the cache type.
int b200_debug_write_kv(b200_engine* e, int slot, int layer, int which, int pos0, int n, const float* rows) {
    if (!e || !e->finalized || !rows || slot < 0 || slot >= e->total_slots || layer < 0 || layer >= N_LAYERS || pos0 < 0 || n < 0 ||
        pos0 + n > e->cfg.kv_capacity) return B200_EINVAL;
    b200_sync(e);                                              // also selects the engine's device
    const size_t cnt = (size_t)n * D_MODEL;
    const long long off = layer * e->kv_layer_stride + slot * e->kv_slot_stride + (long long)pos0 * D_MODEL;
    if (e->cfg.kv_f32) {
        PTTS_CUDA_CHECK(cudaMemcpyAsync((float*)(which ? e->vc : e->kc) + off, rows, cnt * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    } else {
        const std::vector<__nv_bfloat16> b = b200_engine::to_bf16(std::vector<float>(rows, rows + cnt));
        PTTS_CUDA_CHECK(cudaMemcpyAsync((__nv_bfloat16*)(which ? e->vc : e->kc) + off, b.data(), cnt * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice, e->stream));
    }
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

// Test hook: keys [0, pfx_len) of `slot` are rows of `pfx_slot` (what a sentence start of a voice sets up; 0 = private cache).
int b200_debug_set_prefix(b200_engine* e, int slot, int pfx_slot, int pfx_len) {
    if (!e || !e->finalized || slot < 0 || slot >= e->cfg.max_slots || pfx_slot < 0 || pfx_slot >= e->total_slots || pfx_len < 0 ||
        pfx_len > e->cfg.kv_capacity) return B200_EINVAL;
    b200_sync(e);                                              // also selects the engine's device
    e->h_pfx_slot[slot] = pfx_slot; e->h_pfx_len[slot] = pfx_len; e->pfx_version++;
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pfx_slot + slot, &pfx_slot, sizeof(int), cudaMemcpyHostToDevice, e->stream));
    PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pfx_len + slot, &pfx_len, sizeof(int), cudaMemcpyHostToDevice, e->stream));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    return B200_OK;
}

// Test hook: the FlowLM attention dispatch of one layer (flow_attn: the kernels, splits and merge a step or a prefill would pick) over
// caller-given rows and q, run eagerly, synchronised; out[n][1024] = att_bf widened to f32. Rows whose output is not written keep a NaN.
// Every upload is ordered on the engine stream: a plain cudaMemcpy / cudaMemset runs on the legacy stream, which the engine's
// non-blocking streams do not wait for.
int b200_debug_attention(b200_engine* e, int layer, int prefill, int slot0, int n, const int32_t* rows_slot, const int32_t* rows_pos,
                         const float* q, const b200_attn_opts* opts, float* out) {
    if (!e || !e->finalized || layer < 0 || layer >= N_LAYERS || n < 1 || !rows_pos || !q || !out) return B200_EINVAL;
    const int cap = e->cfg.kv_capacity;
    if (prefill) {
        if (!rows_slot) return B200_EINVAL;
        for (int r = 0; r < n; r++)
            if (rows_slot[r] < 0 || rows_slot[r] >= e->total_slots || rows_pos[r] < 0 || rows_pos[r] >= cap ||
                (r > 0 && (rows_slot[r] < rows_slot[r - 1] || (rows_slot[r] == rows_slot[r - 1] && rows_pos[r] <= rows_pos[r - 1])))) return B200_EINVAL;
    } else {
        if (slot0 < 0 || slot0 + n > e->cfg.max_slots) return B200_EINVAL;
        for (int r = 0; r < n; r++) if (rows_pos[r] >= cap) return B200_EINVAL;
        // prefix assignments set through b200_debug_set_prefix can form more distinct prefixes than the work list holds (it is sized for
        // max_voices of them): refuse those here, where prepare_decode would abort
        std::vector<AtItem> items; std::vector<int> rows;
        plan_prefix_tiles(e->h_pfx_slot.data() + slot0, e->h_pfx_len.data() + slot0, n, e->tc ? e->tc->num_sms : 148, items, rows);
        if ((int)items.size() > e->dec_items_cap) return B200_ECAPACITY;
    }
    b200_sync(e);                                              // also selects the engine's device
    const int s_splits = e->af_splits_override, s_tprec = e->tile_prec, s_pprec = e->prefill_prec, s_min = e->tile_min_rows;
    const bool s_fork = e->fork_tiles, s_counted = e->counted_merge, s_pdl_small = e->pdl_small, s_pdl = e->pdl_active;
    const int s_grid = e->dec_grid_items;
    const b200_engine::AttnCtx s_actx = e->actx;
    if (opts) {
        if (opts->stream_splits >= 0) e->af_splits_override = opts->stream_splits;
        if (opts->tile_prec >= 0) e->tile_prec = opts->tile_prec;
        if (opts->prefill_prec >= 0) e->prefill_prec = opts->prefill_prec;
        if (opts->fork_tiles >= 0) e->fork_tiles = opts->fork_tiles != 0;
        if (opts->counted_merge >= 0) e->counted_merge = opts->counted_merge != 0;
        if (opts->tile_min_rows >= 0) e->tile_min_rows = opts->tile_min_rows;
    }
    e->pdl_small = false; e->set_pdl(false);
    auto read_out = [&](float* dst, int R) {
        PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
        PTTS_CUDA_CHECK(cudaGetLastError());
        std::vector<uint16_t> tmp((size_t)R * D_MODEL);
        PTTS_CUDA_CHECK(cudaMemcpy(tmp.data(), e->att_bf, tmp.size() * 2, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < tmp.size(); i++) { const uint32_t u = (uint32_t)tmp[i] << 16; memcpy(&dst[i], &u, 4); }
    };
    int tiles = 0;
    if (!prefill) {
        std::vector<int> rs(n), rp(n);
        for (int r = 0; r < n; r++) { rs[r] = rows_pos[r] < 0 ? -1 : slot0 + r; rp[r] = std::max(0, (int)rows_pos[r]); }   // negative position: dead row
        PTTS_CUDA_CHECK(cudaMemcpyAsync(e->row_slot, rs.data(), n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(e->row_pos, rp.data(), n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(e->q, q, (size_t)n * D_MODEL * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        PTTS_CUDA_CHECK(cudaMemsetAsync(e->att_bf, 0xff, (size_t)n * D_MODEL * sizeof(__nv_bfloat16), e->stream));
        e->dec_key_n = -1;                                     // plan the prefix tiles for this call's rows and options
        e->prepare_decode(slot0, n);
        tiles = e->use_prefix_tiles(n) ? 1 : 0;
        e->flow_attn(layer, n);
        read_out(out, n);
    } else {
        const int MRp = e->cfg.max_prefill_rows, nchunks = (n + MRp - 1) / MRp;
        std::vector<AtItem> items; std::vector<int> chunk_item0(nchunks + 1, 0);
        if (!e->cfg.kv_f32) plan_prefill_items(rows_slot, rows_pos, n, MRp, e->h_pfx_slot.data(), e->h_pfx_len.data(), items, chunk_item0);
        e->grow(e->pf_int, e->pf_int_cap, (size_t)3 * n);
        e->grow(e->pf_items, e->pf_items_cap, items.size() + 1);
        e->grow(e->pf_meta, e->pf_meta_cap, (size_t)4 * nchunks);
        std::vector<int> meta((size_t)4 * nchunks, 0);
        for (int c = 0; c < nchunks; c++) meta[4 * c] = chunk_item0[c + 1] - chunk_item0[c];
        PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_int, rows_slot, n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_int + n, rows_pos, n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_meta, meta.data(), meta.size() * sizeof(int), cudaMemcpyHostToDevice, e->stream));
        if (!items.empty()) PTTS_CUDA_CHECK(cudaMemcpyAsync(e->pf_items, items.data(), items.size() * sizeof(AtItem), cudaMemcpyHostToDevice, e->stream));
        for (int c = 0; c < nchunks; c++) {
            const int r0 = c * MRp, R = std::min(MRp, n - r0);
            e->prefill_chunk(c, r0, n, chunk_item0);
            PTTS_CUDA_CHECK(cudaMemcpyAsync(e->q, q + (size_t)r0 * D_MODEL, (size_t)R * D_MODEL * sizeof(float), cudaMemcpyHostToDevice, e->stream));
            PTTS_CUDA_CHECK(cudaMemsetAsync(e->att_bf, 0xff, (size_t)R * D_MODEL * sizeof(__nv_bfloat16), e->stream));
            e->flow_attn(layer, R);
            read_out(out + (size_t)r0 * D_MODEL, R);
        }
        tiles = (int)items.size();
    }
    e->af_splits_override = s_splits; e->tile_prec = s_tprec; e->prefill_prec = s_pprec; e->tile_min_rows = s_min;
    e->fork_tiles = s_fork; e->counted_merge = s_counted; e->pdl_small = s_pdl_small; e->set_pdl(s_pdl);
    e->actx = s_actx; e->dec_grid_items = s_grid;
    e->dec_key_n = -1;                                         // the device work list is this call's: the next step plans and uploads its own
    return tiles;
}

// Tap points for localising a parity failure (the reference's GraphContext::debug, src/context.h:526-547). Names are the ones the CPU
// restatement under tests uses: "flow.layer<l>" = residual stream after FlowLM layer l [1024], "flow.attn<l>" = attention output of layer l [1024]
// (both need b200_debug_taps(e, 1) before the step), "mimi.upsample" [16][512], "mimi.transformer" [16][512], "seanet.conv0" [16][512],
// "seanet.convt2" [96][256], "seanet.res3" [96][256], "seanet.res6" [480][128], "seanet.res9" [1920][64] (state of the LAST step that
// covered `slot`; low-precision buffers are widened to f32). Returns the element count, or a negative error.
int b200_debug_taps(b200_engine* e, int on) {
    if (!e || !e->finalized) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->join_mimi();
    e->taps_on = on != 0;
    return B200_OK;
}
int b200_debug_tap(b200_engine* e, const char* name, int slot, float* out, int max_elems) {
    if (!e || !e->finalized || !name || slot < 0 || slot >= e->cfg.max_slots) return B200_EINVAL;
    PTTS_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    e->join_mimi();
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    const std::string s = name;
    if (s.rfind("enc.", 0) == 0 && e->enc_T == 0) return B200_ENOTFOUND;   // no clone yet
    auto give_f32 = [&](const float* src, size_t n) -> int {
        if (!out) return (int)n;
        if ((size_t)max_elems < n) return B200_EINVAL;
        PTTS_CUDA_CHECK(cudaMemcpy(out, src, n * sizeof(float), cudaMemcpyDeviceToHost));
        return (int)n;
    };
    // rows [row0, row0 + rows) x the first `cols` of `ld` columns of a 16-bit buffer
    auto give_16 = [&](const void* base, bool f16, long long slot_stride, int row0, int rows, int ld, int cols) -> int {
        const size_t n = (size_t)rows * cols;
        if (!out) return (int)n;
        if ((size_t)max_elems < n) return B200_EINVAL;
        std::vector<uint16_t> tmp((size_t)rows * ld);
        PTTS_CUDA_CHECK(cudaMemcpy(tmp.data(), (const uint16_t*)base + (size_t)slot * slot_stride + (size_t)row0 * ld, tmp.size() * 2, cudaMemcpyDeviceToHost));
        for (int r = 0; r < rows; r++) for (int c = 0; c < cols; c++) {
            const uint16_t u = tmp[(size_t)r * ld + c];
            out[(size_t)r * cols + c] = f16 ? __half2float(*(const __half*)&u) : __bfloat162float(*(const __nv_bfloat16*)&u);
        }
        return (int)n;
    };
    if (s.rfind("flow.layer", 0) == 0 || s.rfind("flow.attn", 0) == 0) {
        const bool att = s[5] == 'a';
        const int l = atoi(s.c_str() + (att ? 9 : 10)), r = slot - e->tap_slot0;
        if (l < 0 || l >= N_LAYERS || r < 0 || r >= e->tap_n) return B200_EINVAL;
        if (att) return give_16(e->tap_att + (size_t)l * e->cfg.max_slots * D_MODEL, false, 0, r, 1, D_MODEL, D_MODEL);
        return give_f32(e->tap_h + ((size_t)l * e->cfg.max_slots + r) * D_MODEL, D_MODEL);
    }
    if (s == "mimi.upsample") return give_f32(e->tap_up + (size_t)slot * M_T * M_DIM, (size_t)M_T * M_DIM);   // needs b200_debug_taps(e, 1)
    if (s == "mimi.transformer") return give_16(e->buf0, true, 22LL * 512, 6, 16, 512, 512);
    if (s == "seanet.conv0") return give_16(e->buf2, true, 17LL * e->C2, 1, 16, e->C2, 512);
    if (s == "seanet.convt2") return give_f32(e->y3 + (size_t)slot * 96 * 256, (size_t)96 * 256);
    if (s == "seanet.res3") return give_16(e->buf5, true, 97LL * e->C5, 1, 96, e->C5, 256);
    if (s == "seanet.res6") return give_16(e->buf8, true, 481LL * e->C8, 1, 480, e->C8, 128);
    if (s == "seanet.res9") return give_16(e->buf11, true, 1922LL * 64, 2, 1920, 64, 64);
    if (s == "enc.seanet") return give_f32(e->eb.xs, (size_t)e->enc_T * M_T * M_DIM);          // the last clone's buffers (slot ignored)
    if (s == "enc.transformer") return give_f32(e->eb.xt, (size_t)e->enc_T * M_T * M_DIM);
    if (s == "enc.downsample") return give_f32(e->eb.lat, (size_t)e->enc_T * M_DIM);
    return B200_ENOTFOUND;
}

// Host-only: the tile width / split-K plan the tensor-core GEMM dispatcher picks for a [R x K] . [N x K]^T product of one slot
// (no device needed; tests/test_cabi.py checks the invariants of the cost model).
int b200_debug_gemm_plan(int R, int N, int K, int num_sms, int want_ln, int* bn, int* splits) {
    if (R < 1 || N < 32 || N % 32 != 0 || K < 64 || K % 64 != 0 || num_sms < 1 || !bn || !splits) return B200_EINVAL;
    const TcPlan p = tc_plan((R + 127) / 128, R, N, K, num_sms, want_ln != 0);
    *bn = p.bn; *splits = p.splits;
    return B200_OK;
}

// Test hook: the encoder's window attention (attn_window_kernel) alone over q, k, v [R][512] f32 (rounded to bf16 here; q and k taken as
// already rotated); out [R][512] = the bf16 output as f32. Synchronises. Needs no encoder weights.
int b200_debug_window_attention(b200_engine* e, int R, const float* q, const float* k, const float* v, float* out) {
    if (!e || !e->finalized || R < 1 || !q || !k || !v || !out) return B200_EINVAL;
    b200_sync(e);                                              // also selects the engine's device
    const size_t n = (size_t)R * M_DIM;
    __nv_bfloat16* d = nullptr;
    PTTS_CUDA_CHECK(cudaMalloc(&d, 4 * n * sizeof(__nv_bfloat16)));
    const float* src[3] = {q, k, v};
    for (int i = 0; i < 3; i++) {
        const std::vector<__nv_bfloat16> b = b200_engine::to_bf16(std::vector<float>(src[i], src[i] + n));
        PTTS_CUDA_CHECK(cudaMemcpyAsync(d + i * n, b.data(), n * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice, e->stream));
        PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    }
    launch_k(false, attn_window_kernel, dim3((R + AW_Q - 1) / AW_Q, M_HEADS), dim3(AW_WARPS * 32), AW_SMEM, e->stream, (const __nv_bfloat16*)d,
             (const __nv_bfloat16*)(d + n), (const __nv_bfloat16*)(d + 2 * n), R, d + 3 * n);
    e->launches++;
    std::vector<uint16_t> tmp(n);
    PTTS_CUDA_CHECK(cudaMemcpyAsync(tmp.data(), d + 3 * n, n * sizeof(uint16_t), cudaMemcpyDeviceToHost, e->stream));
    PTTS_CUDA_CHECK(cudaStreamSynchronize(e->stream));
    PTTS_CUDA_CHECK(cudaFree(d));
    for (size_t i = 0; i < n; i++) { const uint32_t u = (uint32_t)tmp[i] << 16; memcpy(&out[i], &u, 4); }
    return B200_OK;
}

// Host-only: the attention work lists the engine builds (plan_prefix_tiles / plan_prefill_items), for tests without a device.
int b200_debug_attn_plan(int prefill, int n, const int32_t* row_slot, const int32_t* row_pos, const int32_t* pfx_slot, const int32_t* pfx_len,
                         int num_sms, int chunk_rows, int max_voices, int32_t* items_out, int cap, int32_t* aux_out, int* n_items) {
    if (n < 1 || !pfx_slot || !pfx_len || !items_out || !aux_out || !n_items || cap < 0) return B200_EINVAL;
    std::vector<AtItem> items; std::vector<int> aux;
    int ret;
    if (prefill) {
        if (!row_slot || !row_pos || chunk_rows < 1) return B200_EINVAL;
        plan_prefill_items(row_slot, row_pos, n, chunk_rows, pfx_slot, pfx_len, items, aux);
        ret = (int)aux.size() - 1;
    } else {
        if (num_sms < 1) return B200_EINVAL;
        ret = plan_prefix_tiles(pfx_slot, pfx_len, n, num_sms, items, aux);
        if ((int)items.size() > prefix_tiles_capacity(n, max_voices)) ret = B200_ECAPACITY;
    }
    *n_items = (int)items.size();
    if ((int)items.size() > cap) return B200_ECAPACITY;
    for (size_t i = 0; i < items.size(); i++) {
        const AtItem& it = items[i];
        const int v[9] = {it.row0, it.nrows, it.a_slot, it.a_k0, it.a_k1, it.b_slot, it.b_k0, it.b_k1, it.out_split};
        memcpy(items_out + 9 * i, v, sizeof(v));
    }
    memcpy(aux_out, aux.data(), aux.size() * sizeof(int));
    return ret;
}

const char* b200_build_info(void) { return "ptts_b200 sm_100a " __DATE__ " " __TIME__; }

}  // extern "C"
