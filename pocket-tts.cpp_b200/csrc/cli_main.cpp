// pocket-tts-b200 — command-line driver over the reference's pocket_tts API (SURVEY.md §8 row f4): the generation calls are the
// ones demos/pocket-tts.cpp makes (ptts_set_seed, ptts_init, ptts_get_sample_rate/frame_size, ptts_stream_from_safetensors,
// ptts_stream_send / flush / receive; reference demos/pocket-tts.cpp:201,233,368-371,456-520), linked against libptts_b200.so
// instead of the ggml build. `--bench` prints the reference's own result lines (seed / done generating / frame count / frame
// rate, :454,517-520) with the same defaults (bench sentence, seed 0, temperature 0, :229-236). Audio goes to a 16-bit PCM WAV
// file with -o (the reference encodes through FFmpeg or plays through SDL; neither belongs to the generation path).
#include "../../include/pocket_tts/pocket_tts.h"
#include "../../include/ptts_b200.h"

#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

namespace {

void usage(const char* prog) {
    fprintf(stderr,
            "usage: %s [options] \"text to speak\"\n"
            "  -m PATH,  --model PATH        model directory (tts_b6369a24.safetensors, tokenizer.model, embeddings/)\n"
            "  -v VOICE, --voice VOICE       voice name or path to a voice .safetensors (default cosette)\n"
            "  -o FILE,  --output FILE       write 24 kHz 16-bit mono WAV\n"
            "  -i FILE,  --input FILE        read the text from a file\n"
            "  -s N,     --seed N            RNG seed\n"
            "  -t T,     --temperature T     sampling temperature (default 0.7)\n"
            "            --lsd-decode-steps N  LSD decode steps of the flow head, 1..8 (default 1)\n"
            "            --noise-clamp A     truncate the sampling noise to [-A, A] (default 0 = off)\n"
            "            --eos-threshold T   end of speech when the EOS logit exceeds T (default -4)\n"
            "            --bench             fixed sentence, seed 0, temperature 0; prints frames/s like the reference\n",
            prog);
    exit(1);
}

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

void put_u32(std::vector<uint8_t>& b, uint32_t v) { for (int i = 0; i < 4; i++) b.push_back((uint8_t)(v >> (8 * i))); }
void put_u16(std::vector<uint8_t>& b, uint16_t v) { for (int i = 0; i < 2; i++) b.push_back((uint8_t)(v >> (8 * i))); }

bool write_wav(const std::string& path, const std::vector<float>& pcm, int sample_rate) {
    std::vector<uint8_t> b;
    const uint32_t data_bytes = (uint32_t)pcm.size() * 2;
    b.insert(b.end(), {'R', 'I', 'F', 'F'}); put_u32(b, 36 + data_bytes);
    b.insert(b.end(), {'W', 'A', 'V', 'E', 'f', 'm', 't', ' '}); put_u32(b, 16);
    put_u16(b, 1); put_u16(b, 1); put_u32(b, (uint32_t)sample_rate); put_u32(b, (uint32_t)sample_rate * 2); put_u16(b, 2); put_u16(b, 16);
    b.insert(b.end(), {'d', 'a', 't', 'a'}); put_u32(b, data_bytes);
    for (float v : pcm) {
        const float c = std::fmax(-1.0f, std::fmin(1.0f, v));
        put_u16(b, (uint16_t)(int16_t)std::lrintf(c * 32767.0f));
    }
    std::ofstream f(path, std::ios::binary);
    if (!f) return false;
    f.write((const char*)b.data(), (std::streamsize)b.size());
    return (bool)f;
}

}  // namespace

int main(int argc, char** argv) {
    std::string model_path = "kyutai/pocket-tts-without-voice-cloning/", voice = "cosette", output, input, text;
    bool bench = false, seed_set = false, temp_set = false, have_text = false;
    float temperature = 0.7f;
    b200_sampling sampling; b200_default_sampling(&sampling);
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto value = [&]() -> const char* { if (i + 1 >= argc) { fprintf(stderr, "error: \"%s\" requires value\n", argv[i]); exit(1); } return argv[++i]; };
        if (a == "-h" || a == "--help") usage(argv[0]);
        else if (a == "-m" || a == "--model") model_path = value();
        else if (a == "-v" || a == "--voice") voice = value();
        else if (a == "-o" || a == "--output") output = value();
        else if (a == "-i" || a == "--input") input = value();
        else if (a == "-s" || a == "--seed") { seed_set = true; ptts_set_seed((unsigned)std::stoi(value())); }
        else if (a == "-t" || a == "--temperature") { temp_set = true; temperature = (float)std::stod(value()); }
        else if (a == "--lsd-decode-steps") sampling.lsd_steps = std::stoi(value());
        else if (a == "--noise-clamp") sampling.noise_clamp = (float)std::stod(value());
        else if (a == "--eos-threshold") sampling.eos_threshold = (float)std::stod(value());
        else if (a == "--bench") bench = true;
        else if (!a.empty() && a[0] == '-') { fprintf(stderr, "error: unrecognized option \"%s\"\n", argv[i]); exit(1); }
        else if (!have_text) { text = a; have_text = true; }
        else { fprintf(stderr, "error: unexpected extra argument \"%s\"\n", argv[i]); exit(1); }
    }
    if (!input.empty()) {
        std::ifstream f(input);
        if (!f) { fprintf(stderr, "error: unable to read %s\n", input.c_str()); return 1; }
        std::stringstream ss; ss << f.rdbuf(); text = ss.str(); have_text = true;
    }
    if (bench) {
        if (!have_text) { text = "The quick brown fox jumped over the sleeping dog."; have_text = true; }
        if (!seed_set) ptts_set_seed(0);
        if (!temp_set) temperature = 0.f;
    }
    if (b200_sampling_check(&sampling) != B200_OK) {
        fprintf(stderr, "error: sampling controls out of range (--lsd-decode-steps 1..8, --noise-clamp >= 0, finite --eos-threshold)\n");
        return 1;
    }
    if (!have_text) usage(argv[0]);
    if (!model_path.empty() && model_path.back() != '/') model_path += '/';

    ptts_context_t* ctx = ptts_init(nullptr, nullptr, model_path.c_str());     // the engine is the backend: ggml pointers are ignored
    const int sample_rate = ptts_get_sample_rate(ctx), frame_size = ptts_get_frame_size(ctx);
    ptts_stream_t* stream = ptts_stream_from_safetensors(ctx, voice.c_str(), temperature);
    ptts_c_stream_set_sampling(stream, &sampling);

    printf("seed: %d\n", (int)ptts_get_seed());
    const double gen_start = now_ms();
    double lm_ms = 0.0;
    long lm_frames = 0;
    std::vector<float> frame((size_t)frame_size), pcm;
    const char* p = text.c_str();
    size_t left = text.size();
    bool active = true;
    while (active) {
        active = false;
        if (left) {                                            // 15 characters at a time, like the reference's streaming simulation
            const size_t n = left > 15 ? 15 : left;
            const std::string chunk(p, n);
            p += n; left -= n;
            const double t0 = now_ms();
            ptts_stream_send(stream, chunk.c_str());
            if (left == 0) ptts_stream_flush(stream);
            lm_ms += now_ms() - t0;
            active = true;
        }
        const double t0 = now_ms();
        if (ptts_stream_receive(stream, frame.data())) {
            lm_ms += now_ms() - t0;
            lm_frames++;
            if (!output.empty()) pcm.insert(pcm.end(), frame.begin(), frame.end());
            active = true;
        }
    }
    const double gen_end = now_ms();
    printf("done generating. %f\n", (gen_end - gen_start) / 1000.0);
    printf("frame count: %4d frames\n", (int)lm_frames);
    printf("frame rate:  %f frames/s\n", lm_frames * 1000.0 / (lm_ms > 0 ? lm_ms : 1e-9));
    if (!output.empty()) {
        if (!write_wav(output, pcm, sample_rate)) { fprintf(stderr, "error: unable to write %s\n", output.c_str()); return 1; }
        printf("wrote %s (%.2f s of audio)\n", output.c_str(), (double)pcm.size() / sample_rate);
    }
    return 0;
}
