// host_api.cpp — the reference's own streaming API (include/pocket_tts/pocket_tts.h:18-42 of
// Codes4Fun/pocket-tts.cpp) implemented on the B200 engine: same function names, signatures (mangled C++),
// argument meaning and error behaviour, so demos/pocket-tts.cpp links against libptts_b200.so unchanged.
// Host code is C++ and reaches CUDA only through the C ABI in include/ptts_b200.h.
#include "../../include/pocket_tts/pocket_tts.h"
#include "../../include/ptts_b200.h"
#include "host/safetensors.hpp"
#include "host/spm_unigram.hpp"
#include "host/batch_scheduler.hpp"

#include <cctype>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <string>
#include <vector>

using namespace ptts_host;

// ------------------------------------------------------------------------------------------------
// Text front end (reference src/pocket_tts/conditioners/text.h:52-94,181-251)
// ------------------------------------------------------------------------------------------------
namespace {

int count_words_impl(const std::string& text) {
    size_t i = 0; int words = 0;
    while (i < text.size() && isspace((unsigned char)text[i])) i++;
    while (i < text.size()) {
        words++;
        while (i < text.size() && !isspace((unsigned char)text[i])) i++;
        if (i == text.size()) return words;
        while (i < text.size() && isspace((unsigned char)text[i])) i++;
    }
    return words;
}

struct SentenceSplitter {
    std::string tail; std::deque<std::string> sentences;
    bool was_ws = true, was_eos = false, leading = true;
    void reset() { tail.clear(); sentences.clear(); was_ws = true; was_eos = false; leading = true; }
    static bool eos_char(char c) { return c == '.' || c == '!' || c == '?'; }
    void ingest(const std::string& chunk) {
        for (char c : chunk) {
            const bool is_eos = eos_char(c);
            if (!is_eos && was_eos) { sentences.push_back(tail); tail.clear(); was_ws = true; leading = true; }
            const bool ws = isspace((unsigned char)c) != 0;
            if (ws && !was_ws) tail += ' ';
            else if (!ws) {
                if (leading) { if (islower((unsigned char)c)) c = (char)toupper((unsigned char)c); leading = false; }
                tail += c;
            }
            was_ws = ws; was_eos = is_eos;
        }
    }
    void flush() {
        if (!tail.empty()) {
            if (isalnum((unsigned char)tail.back())) tail += '.';
            sentences.push_back(tail); tail.clear();
        }
        was_ws = true; was_eos = false; leading = true;
    }
};

unsigned int g_seed = 0x5eed5eedu;
bool g_seed_set = false;

const char* kVoices[] = {"alba", "azelma", "cosette", "eponine", "fantine", "javert", "jean", "marius"};

int env_int(const char* name, int dflt) { const char* v = getenv(name); return v && *v ? atoi(v) : dflt; }

bool ends_with(const std::string& s, const char* suffix) { const size_t n = strlen(suffix); return s.size() >= n && s.compare(s.size() - n, n, suffix) == 0; }

// RIFF/WAVE reader: PCM16 or float32 (format 1 / 3, or WAVE_FORMAT_EXTENSIBLE with either subformat), any channel count, mixed down
// to mono by averaging. Returns false for anything else, including a data chunk that runs past the end of the file.
bool read_wav(const std::string& path, std::vector<float>& out, int& sample_rate) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    std::vector<uint8_t> b;
    uint8_t buf[65536]; size_t got;
    while ((got = fread(buf, 1, sizeof buf, f)) > 0) b.insert(b.end(), buf, buf + got);
    fclose(f);
    auto u16 = [&](size_t o) { return (uint32_t)b[o] | ((uint32_t)b[o + 1] << 8); };
    auto u32 = [&](size_t o) { return u16(o) | (u16(o + 2) << 16); };
    if (b.size() < 12 || memcmp(b.data(), "RIFF", 4) != 0 || memcmp(b.data() + 8, "WAVE", 4) != 0) return false;
    int fmt = -1, channels = 0, bits = 0; bool have_fmt = false;
    for (size_t o = 12; o + 8 <= b.size();) {
        const uint32_t sz = u32(o + 4);
        const size_t body = o + 8;
        if ((uint64_t)body + sz > b.size()) return false;                        // truncated chunk
        if (memcmp(b.data() + o, "fmt ", 4) == 0) {
            if (sz < 16) return false;
            fmt = (int)u16(body); channels = (int)u16(body + 2); sample_rate = (int)u32(body + 4); bits = (int)u16(body + 14);
            if (fmt == 0xFFFE) { if (sz < 26) return false; fmt = (int)u16(body + 24); }   // extensible: the subformat GUID starts with the format tag
            have_fmt = true;
        } else if (memcmp(b.data() + o, "data", 4) == 0) {
            if (!have_fmt || channels < 1) return false;
            const bool pcm16 = fmt == 1 && bits == 16, f32 = fmt == 3 && bits == 32;
            if (!pcm16 && !f32) return false;
            const size_t frame_bytes = (size_t)channels * (bits / 8), n = sz / frame_bytes;
            out.assign(n, 0.f);
            for (size_t i = 0; i < n; i++) {
                double acc = 0;
                for (int c = 0; c < channels; c++) {
                    const size_t at = body + i * frame_bytes + (size_t)c * (bits / 8);
                    if (pcm16) acc += (int16_t)u16(at) / 32768.0;
                    else { float v; memcpy(&v, b.data() + at, 4); acc += v; }
                }
                out[i] = (float)(acc / channels);
            }
            return true;
        }
        o = body + sz + (sz & 1);                                                // chunks are padded to even sizes
    }
    return false;
}

// audio_prompt [1, T, 1024] F32, the layout of a voice file
bool write_voice_file(const std::string& path, const std::vector<float>& prompt) {
    const size_t T = prompt.size() / 1024;
    std::string h = "{\"audio_prompt\":{\"dtype\":\"F32\",\"shape\":[1," + std::to_string(T) + ",1024],\"data_offsets\":[0," + std::to_string(prompt.size() * 4) + "]}}";
    while (h.size() % 8) h += ' ';
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    const uint64_t hl = h.size();
    bool ok = fwrite(&hl, 8, 1, f) == 1 && fwrite(h.data(), 1, h.size(), f) == h.size() && fwrite(prompt.data(), 4, prompt.size(), f) == prompt.size();
    return fclose(f) == 0 && ok;
}

}  // namespace

struct ptts_context_t {
    b200_engine* engine = nullptr;
    std::string model_path;
    SpmUnigram tokenizer;
    std::map<std::string, int> voices;      // resolved voice file or registered name -> engine voice id
    std::map<std::string, std::vector<float>> cloned;   // voices created from audio: their audio_prompt rows [T][1024] (for export)
    std::vector<bool> slot_used;
    int n_streams = 0;
    bool lookahead = true;                  // PTTS_B200_LOOKAHEAD=0: strictly one step per receive
    unsigned int seed_pushed = 0; bool seed_valid = false;   // last seed handed to the engine (ptts_set_seed is process-global)
};

struct ptts_stream_t {
    ptts_context_t* ctx = nullptr;
    int slot = -1, voice = -1;
    float temp = 0.7f;
    SentenceSplitter sproc;
    int frames_after_eos = 0, max_gen_len = 0, generation_step = 0;
    int inflight = 0;                       // frames submitted to the engine but not collected yet (look-ahead pipeline)
    std::vector<float> scratch;             // sink for a look-ahead frame that turned out to lie past the end of the sentence
};

static int upload_checkpoint(b200_engine* eng, const std::string& file) {
    SafeTensors st;
    if (!st.open(file)) return -1;
    std::vector<uint8_t> raw;
    for (auto& kv : st.entries) {
        int dt;
        if (kv.second.dtype == "F32") dt = B200_DT_F32; else if (kv.second.dtype == "BF16") dt = B200_DT_BF16; else if (kv.second.dtype == "F16") dt = B200_DT_F16; else continue;
        if (!st.read(kv.second, raw)) return -1;
        if (b200_upload_tensor(eng, kv.first.c_str(), raw.data(), dt, kv.second.shape.data(), (int)kv.second.shape.size()) != B200_OK) return -1;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// The 10 reference API functions
// ------------------------------------------------------------------------------------------------
void ptts_set_seed(unsigned int seed) { g_seed = seed; g_seed_set = true; }   // reference src/pocket_tts.cpp:252-255
unsigned int ptts_get_seed() { return g_seed; }                                // :257-259

static ptts_context_t* init_with_config(const char* model_path, const b200_config& cfg) {
    auto* ctx = new ptts_context_t;
    ctx->model_path = model_path;
    if (b200_engine_create(&cfg, &ctx->engine) != B200_OK) { fprintf(stderr, "error: failed to create the B200 engine\n"); exit(1); }
    const std::string filename = ctx->model_path + "tts_b6369a24.safetensors";
    if (upload_checkpoint(ctx->engine, filename) != 0) { fprintf(stderr, "error: weights not found %s\n", filename.c_str()); exit(1); }
    if (b200_finalize_weights(ctx->engine) != B200_OK) { fprintf(stderr, "error: failed to load weights %s\n", filename.c_str()); exit(1); }
    if (!ctx->tokenizer.load(ctx->model_path + "tokenizer.model")) { fprintf(stderr, "error: tokenizer not found %stokenizer.model\n", model_path); exit(1); }
    ctx->slot_used.assign(cfg.max_slots, false);
    ctx->lookahead = env_int("PTTS_B200_LOOKAHEAD", 1) != 0 && cfg.overlap != 0;
    return ctx;
}

// reference src/pocket_tts.cpp:273-322. The ggml backends are ignored (this engine IS the backend).
ptts_context_t* ptts_init(ggml_backend*, ggml_backend*, const char* model_path) {
    b200_config cfg; b200_default_config(&cfg);
    cfg.device = env_int("PTTS_B200_DEVICE", 0);
    cfg.max_slots = env_int("PTTS_B200_MAX_STREAMS", 4);
    cfg.kv_capacity = env_int("PTTS_B200_KV_CAPACITY", 2048);
    cfg.kv_f32 = env_int("PTTS_B200_KV_F32", 0);
    cfg.mimi_mask_mode = env_int("PTTS_B200_MIMI_CAUSAL", 0);
    cfg.gemm_path = env_int("PTTS_B200_GEMM_PATH", 0);
    cfg.cuda_graphs = env_int("PTTS_B200_CUDA_GRAPHS", 1);
    cfg.pdl = env_int("PTTS_B200_PDL", 1);
    cfg.overlap = env_int("PTTS_B200_OVERLAP", 1);
    cfg.prefix_share = env_int("PTTS_B200_PREFIX_SHARE", 1);
    return init_with_config(model_path, cfg);
}

int ptts_get_sample_rate(ptts_context_t*) { return 24000; }   // reference :324-326
int ptts_get_frame_size(ptts_context_t*) { return 1920; }     // reference :328-330

// Clones a voice from mono 24 kHz PCM and registers it under `name`. The rows come back to the host once, so that the voice can be exported.
static int add_audio_voice(ptts_context_t* ctx, const std::string& name, const float* pcm, long long n) {
    const long long T = (n + 1919) / 1920;
    if (n < 1 || T > b200_kv_capacity(ctx->engine)) return n < 1 ? B200_EINVAL : B200_ECAPACITY;
    std::vector<float> prompt((size_t)T * 1024);
    const int t = b200_voice_embed_audio(ctx->engine, pcm, n, prompt.data());
    if (t < 0) return t;
    const int vid = b200_voice_create(ctx->engine, prompt.data(), t);
    if (vid < 0) return vid;
    ctx->voices[name] = vid;
    ctx->cloned[name] = std::move(prompt);
    return vid;
}

// Voice name or path -> engine voice id; the first use loads the file and prefills the prefix (reference src/pocket_tts.cpp:356-359,100-124).
// A path ending in ".wav" is a recording: it is cloned (add_audio_voice).
static int resolve_voice(ptts_context_t* ctx, const char* voice_c_str) {
    std::string voice = voice_c_str;
    for (const char* v : kVoices) if (voice == v) { voice = ctx->model_path + "embeddings/" + v + ".safetensors"; break; }
    int vid;
    auto it = ctx->voices.find(voice);
    if (it != ctx->voices.end()) vid = it->second;
    else if (ends_with(voice, ".wav")) {
        std::vector<float> pcm; int rate = 0;
        if (!read_wav(voice, pcm, rate)) { fprintf(stderr, "error: failed to open voice %s\n", voice.c_str()); exit(1); }
        if (rate != 24000) { fprintf(stderr, "error: voice %s: sample rate %d Hz, the encoder takes 24000 Hz\n", voice.c_str(), rate); exit(1); }
        vid = add_audio_voice(ctx, voice, pcm.data(), (long long)pcm.size());
        if (vid < 0) { fprintf(stderr, "error: failed to clone voice %s (%d)\n", voice.c_str(), vid); exit(1); }
    } else {
        SafeTensors st;
        if (!st.open(voice)) { fprintf(stderr, "error: failed to open voice %s\n", voice.c_str()); exit(1); }
        auto e = st.entries.find("audio_prompt");
        std::vector<uint8_t> raw;
        if (e == st.entries.end() || !st.read(e->second, raw)) { fprintf(stderr, "error: failed to open voice %s\n", voice.c_str()); exit(1); }
        size_t n = 1; for (auto d : e->second.shape) n *= (size_t)d;
        if (n == 0 || n % 1024 != 0) { fprintf(stderr, "error: voice %s: audio_prompt has %zu elements, not a multiple of 1024\n", voice.c_str(), n); exit(1); }
        std::vector<float> prompt(n);
        if (e->second.dtype == "F32") memcpy(prompt.data(), raw.data(), n * 4);
        else if (e->second.dtype == "BF16") { const uint16_t* s = (const uint16_t*)raw.data(); for (size_t i = 0; i < n; i++) { uint32_t u = (uint32_t)s[i] << 16; memcpy(&prompt[i], &u, 4); } }
        else { fprintf(stderr, "error: unsupported voice dtype %s\n", e->second.dtype.c_str()); exit(1); }
        vid = b200_voice_create(ctx->engine, prompt.data(), (int)(n / 1024));
        if (vid < 0) { fprintf(stderr, "error: failed to prefill voice %s (%d)\n", voice.c_str(), vid); exit(1); }
        ctx->voices[voice] = vid;
    }
    return vid;
}

// reference src/pocket_tts.cpp:351-394 (+ get_state_for_audio_prompt :100-124)
ptts_stream_t* ptts_stream_from_safetensors(ptts_context_t* ctx, const char* voice_c_str, float temp) {
    const int vid = resolve_voice(ctx, voice_c_str);
    int slot = -1;
    for (size_t i = 0; i < ctx->slot_used.size(); i++) if (!ctx->slot_used[i]) { slot = (int)i; break; }
    if (slot < 0) { fprintf(stderr, "error: no free stream slot (raise PTTS_B200_MAX_STREAMS)\n"); exit(1); }
    ctx->slot_used[slot] = true; ctx->n_streams++;
    auto* s = new ptts_stream_t;
    s->ctx = ctx; s->slot = slot; s->voice = vid; s->temp = temp;
    ptts_stream_reset(s);
    return s;
}

static void stream_drain(ptts_stream_t* s);
void ptts_stream_reset(ptts_stream_t* s) { stream_drain(s); s->max_gen_len = 0; s->generation_step = 0; s->sproc.reset(); }   // reference :396-400
void ptts_stream_flush(ptts_stream_t* s) { s->sproc.flush(); }                                                  // reference :402-404
void ptts_stream_send(ptts_stream_t* s, const char* chunk) {                                                   // reference :406-414
    if (chunk[0] == '\0') { ptts_stream_flush(s); return; }
    s->sproc.ingest(chunk);
}

// Collect and drop whatever this stream still has in flight (end of sentence, reset).
static void stream_drain(ptts_stream_t* s) {
    int32_t produced = 0;
    if (s->inflight > 0 && s->scratch.size() < 1920) s->scratch.resize(1920);
    while (s->inflight > 0) { b200_collect(s->ctx->engine, s->scratch.data(), &produced); s->inflight--; }
}

// reference _stream_sentence_step :446-492. With a single stream in the context the engine runs one frame AHEAD: the FlowLM step of
// frame t+1 is submitted before frame t is collected, so it overlaps frame t's Mimi decode (b200_submit / b200_collect). At batch 1
// both halves are launch-latency bound, so a frame costs max(FlowLM, Mimi) instead of their sum. A look-ahead step past the end of a
// sentence is harmless: an inactive slot keeps its FlowLM state, and the Mimi state is reset by the next sentence start anyway.
static bool stream_step(ptts_stream_t* s, float* samples) {
    if (s->generation_step >= s->max_gen_len) { fprintf(stderr, "warning: called with high gen step\n"); return false; }
    int32_t produced = 0;
    b200_engine* eng = s->ctx->engine;
    if (s->ctx->seed_pushed != g_seed || !s->ctx->seed_valid) { b200_set_seed(eng, g_seed); s->ctx->seed_pushed = g_seed; s->ctx->seed_valid = true; }
    if (!s->ctx->lookahead || s->ctx->n_streams != 1) {               // several streams share the engine's in-order frame queue: stay synchronous
        if (s->inflight > 0) {
            // This stream submitted look-ahead frames while it was alone in the context and a second stream has appeared since. The engine
            // has already advanced the slot for those frames (gen_step, latent feedback), so they ARE the next frames of this stream:
            // hand them out in order instead of dropping them (only a stream that was alone can own in-flight frames, so the engine's
            // in-order queue holds nothing else).
            if (b200_collect(eng, samples, &produced) < 0) { fprintf(stderr, "error: step failed\n"); exit(1); }
            s->inflight--;
        } else if (b200_step(eng, s->slot, 1, nullptr, samples, &produced, nullptr, nullptr) != B200_OK) { fprintf(stderr, "error: step failed\n"); exit(1); }
    } else {
        if (s->inflight == 0) { if (b200_submit(eng, s->slot, 1, nullptr) != B200_OK) { fprintf(stderr, "error: step failed\n"); exit(1); } s->inflight++; }
        if (s->generation_step + s->inflight < s->max_gen_len && s->inflight < 2) {
            if (b200_submit(eng, s->slot, 1, nullptr) != B200_OK) { fprintf(stderr, "error: step failed\n"); exit(1); }
            s->inflight++;
        }
        if (b200_collect(eng, samples, &produced) < 0) { fprintf(stderr, "error: step failed\n"); exit(1); }
        s->inflight--;
    }
    if (!produced) { s->generation_step = s->max_gen_len; stream_drain(s); return false; }
    s->generation_step++;
    return true;
}

bool ptts_stream_receive(ptts_stream_t* s, float* samples) {          // reference :494-519
    if (s->generation_step < s->max_gen_len) {
        if (stream_step(s, samples)) return true;
    }
    if (!s->sproc.sentences.empty()) {
        const std::string text = s->sproc.sentences.front();
        s->sproc.sentences.pop_front();
        const int words = count_words_impl(text);
        const int fae = (words <= 4 ? 3 : 1) + 2;
        const int max_gen_len = (int)((words + 2.0f) * 12.5f);          // _stream_sentence_init :429-430
        std::vector<int> ids = s->ctx->tokenizer.encode(text);
        std::vector<int32_t> ids32(ids.begin(), ids.end());
        stream_drain(s);
        const int rc = b200_begin_sentence(s->ctx->engine, s->slot, s->voice, ids32.data(), (int)ids32.size(), max_gen_len, fae, s->temp);
        if (rc != B200_OK) { fprintf(stderr, "error: sentence init failed (%d)\n", rc); exit(1); }
        s->frames_after_eos = fae; s->max_gen_len = max_gen_len; s->generation_step = 0;
        if (stream_step(s, samples)) return true;
    }
    return false;
}

// ------------------------------------------------------------------------------------------------
// extern "C" aliases for FFI users
// ------------------------------------------------------------------------------------------------
extern "C" {
void ptts_c_set_seed(unsigned int seed) { ptts_set_seed(seed); }
unsigned int ptts_c_get_seed(void) { return ptts_get_seed(); }
ptts_context_t* ptts_c_init(const char* model_path) { return ptts_init(nullptr, nullptr, model_path); }
ptts_context_t* ptts_c_init_ex(const char* model_path, const b200_config* cfg) { return init_with_config(model_path, *cfg); }
int ptts_c_voice(ptts_stream_t* s) { return s->voice; }
int ptts_c_slot(ptts_stream_t* s) { return s->slot; }
int ptts_c_get_sample_rate(ptts_context_t* c) { return ptts_get_sample_rate(c); }
int ptts_c_get_frame_size(ptts_context_t* c) { return ptts_get_frame_size(c); }
ptts_stream_t* ptts_c_stream_from_safetensors(ptts_context_t* c, const char* voice, float temp) { return ptts_stream_from_safetensors(c, voice, temp); }
void ptts_c_stream_reset(ptts_stream_t* s) { ptts_stream_reset(s); }
void ptts_c_stream_flush(ptts_stream_t* s) { ptts_stream_flush(s); }
void ptts_c_stream_send(ptts_stream_t* s, const char* chunk) { ptts_stream_send(s, chunk); }
int ptts_c_stream_receive(ptts_stream_t* s, float* samples) { return ptts_stream_receive(s, samples) ? 1 : 0; }
b200_engine* ptts_c_engine(ptts_context_t* c) { return c ? c->engine : nullptr; }
// The reference API has no destroy functions (contexts live for the process, src/pocket_tts.cpp:313,381); long-running hosts and
// tests that create several engines need one. Streams of the context must not be used afterwards.
void ptts_c_destroy(ptts_context_t* c) { if (c) { b200_engine_destroy(c->engine); delete c; } }
int ptts_c_tokenize(ptts_context_t* c, const char* text, int32_t* ids, int max_ids) {
    std::vector<int> v = c->tokenizer.encode(text);
    for (int i = 0; i < (int)v.size() && i < max_ids; i++) ids[i] = v[i];
    return (int)v.size();
}
int ptts_c_count_words(const char* text) { return count_words_impl(text); }
int ptts_c_voice_add_audio(ptts_context_t* c, const char* name, const float* pcm, long long n, int sample_rate) {
    if (!c || !name || !pcm || sample_rate != 24000 || c->voices.count(name)) return B200_EINVAL;
    for (const char* v : kVoices) if (strcmp(name, v) == 0) return B200_EINVAL;   // resolve_voice maps these to the model's voice files first
    if (!b200_has_encoder(c->engine)) return B200_ENOTFOUND;
    return add_audio_voice(c, name, pcm, n);
}
int ptts_c_voice_export(ptts_context_t* c, const char* name, const char* path) {
    if (!c || !name || !path) return B200_EINVAL;
    auto it = c->cloned.find(name);
    if (it == c->cloned.end()) return B200_ENOTFOUND;
    return write_voice_file(path, it->second) ? B200_OK : B200_EINVAL;
}
int ptts_c_wav_read(const char* path, float* pcm, long long max, int* sample_rate) {
    std::vector<float> v; int rate = 0;
    if (!path || !read_wav(path, v, rate)) return B200_EINVAL;
    if (pcm) memcpy(pcm, v.data(), (size_t)std::min<long long>(std::max<long long>(max, 0), (long long)v.size()) * sizeof(float));
    if (sample_rate) *sample_rate = rate;
    return (int)v.size();
}
int ptts_c_stream_pending(ptts_stream_t* s, int index, char* buf, int buflen) {
    const int n = (int)s->sproc.sentences.size();
    if (index >= 0 && index < n && buf && buflen > 0) {
        const std::string& t = s->sproc.sentences[index];
        const int m = std::min((int)t.size(), buflen - 1);
        memcpy(buf, t.data(), m); buf[m] = 0;
    }
    return n;
}

// ---- continuous batching (host/batch_scheduler.hpp): many utterances over the engine's slots, finished slots refilled ----
struct ptts_batch_t {
    ptts_context_t* ctx = nullptr;                // null for a scheduler driven through caller-supplied ops (tests)
    BatchScheduler* sched = nullptr;
};
static int batch_begin_engine(void* u, int n, const int32_t* sl, const int32_t* vo, const int32_t* toks, const int32_t* off, const int32_t* mg,
                              const int32_t* fae, const float* tp, const uint32_t* rs) {
    return b200_begin_sentences_ex((b200_engine*)u, n, sl, vo, toks, off, mg, fae, tp, rs);
}
static int batch_submit_engine(void* u, int slot0, int n) { return b200_submit((b200_engine*)u, slot0, n, nullptr); }
static int batch_collect_engine(void* u, float* pcm, int32_t* produced) { return b200_collect((b200_engine*)u, pcm, produced); }
static int batch_end_engine(void* u, int n, const int32_t* slots) { return b200_end_sentences((b200_engine*)u, n, slots); }

ptts_batch_t* ptts_c_batch_create(ptts_context_t* ctx, int n_slots) {
    if (!ctx) return nullptr;
    const int max_slots = b200_max_slots(ctx->engine);
    if (n_slots <= 0 || n_slots > max_slots) n_slots = max_slots;
    for (bool used : ctx->slot_used) if (used) { fprintf(stderr, "error: ptts_c_batch_create needs a context without open streams (slots are shared)\n"); return nullptr; }
    auto* b = new ptts_batch_t; b->ctx = ctx;
    BatchOps ops; ops.user = ctx->engine; ops.begin = batch_begin_engine; ops.submit = batch_submit_engine; ops.collect = batch_collect_engine;
    ops.end = batch_end_engine;
    b->sched = new BatchScheduler(ops, n_slots);
    if (ctx->seed_pushed != g_seed || !ctx->seed_valid) { b200_set_seed(ctx->engine, g_seed); ctx->seed_pushed = g_seed; ctx->seed_valid = true; }
    return b;
}
ptts_batch_t* ptts_c_batch_create_with_ops_ex(void* user, ptts_batch_begin_fn begin, ptts_batch_submit_fn submit, ptts_batch_collect_fn collect,
                                              ptts_batch_end_fn end, int n_slots, int frame_size) {
    if (!begin || !submit || !collect || n_slots < 1 || frame_size < 1) return nullptr;
    auto* b = new ptts_batch_t;
    BatchOps ops; ops.user = user; ops.begin = begin; ops.submit = submit; ops.collect = collect; ops.end = end;
    b->sched = new BatchScheduler(ops, n_slots, frame_size);
    return b;
}
ptts_batch_t* ptts_c_batch_create_with_ops(void* user, ptts_batch_begin_fn begin, ptts_batch_submit_fn submit, ptts_batch_collect_fn collect, int n_slots, int frame_size) {
    return ptts_c_batch_create_with_ops_ex(user, begin, submit, collect, nullptr, n_slots, frame_size);
}
void ptts_c_batch_destroy(ptts_batch_t* b) { if (b) { b->sched->drain(); delete b->sched; delete b; } }
int ptts_c_batch_configure(ptts_batch_t* b, int refill_min, int refill_every, int range_quantum, int keep_pcm) {
    if (!b) return B200_EINVAL;
    if (refill_min > 0) b->sched->refill_min = refill_min;
    if (refill_every > 0) b->sched->refill_every = refill_every;
    if (range_quantum > 0) b->sched->range_quantum = range_quantum;
    if (keep_pcm >= 0) b->sched->keep_pcm = keep_pcm != 0;
    return B200_OK;
}
// One utterance = text in the reference's streaming sense: split into sentences (str_processor, conditioners/text.h:181-251), each
// sentence is one job with the reference's cap and frames_after_eos (src/pocket_tts.cpp:429-430,504-506).
int ptts_c_batch_add(ptts_batch_t* b, const char* voice, const char* text, float temp) {
    if (!b || !b->ctx || !voice || !text) return B200_EINVAL;
    const int vid = resolve_voice(b->ctx, voice);
    auto& rv = b->sched->room_of_voice;
    if ((int)rv.size() <= vid) rv.resize(vid + 1, 1 << 30);
    rv[vid] = b200_kv_capacity(b->ctx->engine) - b200_voice_len(b->ctx->engine, vid);
    SentenceSplitter sp; sp.reset(); sp.ingest(text); sp.flush();
    const int utt = b->sched->add_utterance();
    int idx = 0;
    for (const std::string& sent : sp.sentences) {
        BatchScheduler::Job j; j.utt = utt; j.index = idx++; j.voice = vid; j.temp = temp;
        const int words = count_words_impl(sent);
        j.fae = (words <= 4 ? 3 : 1) + 2; j.max_gen = (int)((words + 2.0f) * 12.5f);
        std::vector<int> ids = b->ctx->tokenizer.encode(sent);
        j.ids.assign(ids.begin(), ids.end());
        b->sched->add_job(std::move(j));
    }
    return utt;
}
// One sentence given as token ids, appended to utterance `utt`.
static int batch_add_token_job(ptts_batch_t* b, int utt, int voice_id, const int32_t* ids, int n_ids, int max_gen_len, int frames_after_eos, float temp, uint32_t rng_stream) {
    if (n_ids < 0 || (n_ids > 0 && !ids)) return B200_EINVAL;
    if (b->ctx) {
        auto& rv = b->sched->room_of_voice;
        const int vl = b200_voice_len(b->ctx->engine, voice_id);
        if (vl < 0) return B200_EINVAL;
        if ((int)rv.size() <= voice_id) rv.resize(voice_id + 1, 1 << 30);
        rv[voice_id] = b200_kv_capacity(b->ctx->engine) - vl;
    }
    if (utt < 0) utt = b->sched->add_utterance();
    BatchScheduler::Job j; j.utt = utt; j.index = b->sched->sentences(utt); j.voice = voice_id; j.temp = temp; j.max_gen = max_gen_len; j.fae = frames_after_eos;
    j.rng_stream = rng_stream; j.ids.assign(ids, ids + n_ids);
    b->sched->add_job(std::move(j));
    return utt;
}
int ptts_c_batch_add_tokens(ptts_batch_t* b, int voice_id, const int32_t* ids, int n_ids, int max_gen_len, int frames_after_eos, float temp, uint32_t rng_stream) {
    if (!b) return B200_EINVAL;
    return batch_add_token_job(b, -1, voice_id, ids, n_ids, max_gen_len, frames_after_eos, temp, rng_stream);
}
int ptts_c_batch_append_tokens(ptts_batch_t* b, int utt, int voice_id, const int32_t* ids, int n_ids, int max_gen_len, int frames_after_eos, float temp,
                               uint32_t rng_stream) {
    if (!b || !b->sched->valid_utt(utt) || b->sched->status(utt, nullptr) == BatchScheduler::kCancelled) return B200_EINVAL;
    return batch_add_token_job(b, utt, voice_id, ids, n_ids, max_gen_len, frames_after_eos, temp, rng_stream);
}
long long ptts_c_batch_run(ptts_batch_t* b) { return b ? b->sched->run() : B200_EINVAL; }
long long ptts_c_batch_pump(ptts_batch_t* b, int max_steps) { return b && max_steps > 0 ? b->sched->pump(max_steps) : B200_EINVAL; }
int ptts_c_batch_frames(ptts_batch_t* b, int utt) {
    if (!b || !b->sched->valid_utt(utt)) return B200_EINVAL;
    return b->sched->frames(utt);
}
int ptts_c_batch_read(ptts_batch_t* b, int utt, float* pcm, int max_frames) {
    if (!b || !b->sched->valid_utt(utt) || !pcm) return B200_EINVAL;
    return b->sched->read(utt, pcm, max_frames);
}
int ptts_c_batch_pop(ptts_batch_t* b, int utt, float* pcm, int max_frames) {
    if (!b || !b->sched->valid_utt(utt) || !pcm) return B200_EINVAL;
    return b->sched->pop(utt, pcm, std::max(max_frames, 0));
}
int ptts_c_batch_cancel(ptts_batch_t* b, int utt) {
    if (!b || !b->sched->valid_utt(utt)) return B200_EINVAL;
    b->sched->cancel(utt);
    return B200_OK;
}
int ptts_c_batch_status(ptts_batch_t* b, int utt, int* ready_frames) {
    if (!b || !b->sched->valid_utt(utt)) return B200_EINVAL;
    return b->sched->status(utt, ready_frames);
}
void ptts_c_batch_stats(ptts_batch_t* b, ptts_batch_stats* out) {
    if (!b || !out) return;
    const BatchStats& s = b->sched->stats();
    out->steps = s.steps; out->frames = s.frames; out->slot_steps = s.slot_steps; out->sentences = s.sentences; out->refills = s.refills; out->wall_ms = s.wall_ms; out->begin_ms = s.begin_ms; out->submit_ms = s.submit_ms; out->collect_ms = s.collect_ms;
}

// Host-only helpers (no GPU needed): tokenizer / splitter objects for CPU-side tests and FFI users.
struct ptts_text_t { SpmUnigram tok; SentenceSplitter sp; };
B200_API ptts_text_t* ptts_c_text_create(const char* tokenizer_model) {
    auto* t = new ptts_text_t;
    if (!t->tok.load(tokenizer_model)) { delete t; return nullptr; }
    t->sp.reset();
    return t;
}
B200_API void ptts_c_text_destroy(ptts_text_t* t) { delete t; }
B200_API int ptts_c_text_encode(ptts_text_t* t, const char* text, int32_t* ids, int max_ids) {
    std::vector<int> v = t->tok.encode(text);
    for (int i = 0; i < (int)v.size() && i < max_ids; i++) ids[i] = v[i];
    return (int)v.size();
}
B200_API void ptts_c_text_send(ptts_text_t* t, const char* chunk) { if (chunk[0] == '\0') t->sp.flush(); else t->sp.ingest(chunk); }
B200_API void ptts_c_text_flush(ptts_text_t* t) { t->sp.flush(); }
B200_API void ptts_c_text_reset(ptts_text_t* t) { t->sp.reset(); }
B200_API int ptts_c_text_pop(ptts_text_t* t, char* buf, int buflen) {
    if (t->sp.sentences.empty()) return -1;
    const std::string s = t->sp.sentences.front(); t->sp.sentences.pop_front();
    const int m = std::min((int)s.size(), buflen - 1);
    memcpy(buf, s.data(), m); buf[m] = 0;
    return (int)s.size();
}
}
