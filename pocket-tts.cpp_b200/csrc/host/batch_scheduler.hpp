// Continuous batching over the engine's slots.
//
// The reference serves ONE stream and rolls to the next sentence inside ptts_stream_receive (src/pocket_tts.cpp:494-519): every
// sentence restarts from the voice-conditioned state and resets the Mimi decoder (_stream_sentence_init :416-444), so sentences are
// independent units of work even inside one utterance. This scheduler exploits that: sentences ("jobs") of many utterances are queued,
// longest first; every step covers the slot range in use; a slot whose sentence finished (EOS rule or cap, decided on the device) is
// refilled with the next queued sentence while the other slots keep generating. Nothing here synchronises the device except the
// collect of the oldest in-flight frame: sentence starts are enqueued between steps (b200_begin_sentences_ex is asynchronous).
//
// The loop is resumable (pump): utterances may be added, their audio handed out in order (pop) and cancelled between two calls, so
// one scheduler serves requests that arrive over time. run() is pump until idle.
//
// The engine is reached through a table of calls so that the scheduling logic can be driven by a mock engine in CPU tests.
#pragma once
#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdint>
#include <cstring>
#include <deque>
#include <string>
#include <vector>

namespace ptts_host {

struct BatchOps {
    void* user = nullptr;
    // per-sentence arrays of length n; tokens concatenated, tok_off[n+1]; returns 0 on success
    int (*begin)(void* user, int n, const int32_t* slots, const int32_t* voices, const int32_t* tokens, const int32_t* tok_off,
                 const int32_t* max_gen_len, const int32_t* frames_after_eos, const float* temp, const uint32_t* rng_stream) = nullptr;
    int (*submit)(void* user, int slot0, int n) = nullptr;                           // enqueue one step of slots [slot0, slot0 + n)
    int (*collect)(void* user, float* pcm, int32_t* produced) = nullptr;              // oldest in-flight step: [n][1920], [n]; returns n
    // optional: the sentences of these slots end before the next submitted step (slots freed by cancel and not refilled); null = such
    // slots keep generating on the engine, unattributed, until a sentence start reuses them
    int (*end)(void* user, int n, const int32_t* slots) = nullptr;
};

struct BatchStats {
    long long steps = 0;          // engine steps submitted
    long long frames = 0;         // audio frames produced (all utterances)
    long long slot_steps = 0;     // sum over steps of the stepped slot count (idle fraction = 1 - frames / slot_steps)
    long long sentences = 0;      // sentences completed
    long long refills = 0;        // sentence-start calls
    double wall_ms = 0.0;         // run() / pump() wall time
    double begin_ms = 0.0, submit_ms = 0.0, collect_ms = 0.0;   // host time inside the three engine calls (collect includes waiting for the GPU)
};

class BatchScheduler {
public:
    struct Job {
        int utt = 0, index = 0;              // utterance id, sentence index inside it
        int voice = 0; float temp = 0.7f;
        std::vector<int32_t> ids;            // SentencePiece ids
        int max_gen = 0, fae = 0;            // reference stop rule: cap int((words + 2) * 12.5), frames_after_eos (src/pocket_tts.cpp:429-430,504-506)
        uint32_t rng_stream = 0;
        std::vector<float> pcm; int frames = 0; bool done = false, started = false;
    };
    enum { kQueued = 0, kRunning = 1, kDone = 2, kCancelled = 3 };

    BatchScheduler(const BatchOps& ops, int n_slots, int frame = 1920) : ops_(ops), n_slots_(n_slots), frame_(frame), slots_(n_slots) {}

    // Tunables: refill as soon as `refill_min` slots are free or `refill_every` steps passed since the last sentence start (each
    // sentence start costs a prefill pass over the weights, so single-slot refills every step would not pay); range granularity.
    int refill_min = 8, refill_every = 8, range_quantum = 32, depth = 2;
    bool keep_pcm = true;

    int add_utterance() { utts_.emplace_back(); return (int)utts_.size() - 1; }
    int sentences(int utt) const { return (int)utts_[utt].jobs.size(); }
    // j.utt must come from add_utterance(); an utterance's audio is its jobs' frames in the order they were added
    int add_job(Job j) {
        j.rng_stream = j.rng_stream ? j.rng_stream : (uint32_t)jobs_.size() + 1;
        utts_[j.utt].jobs.push_back((int)jobs_.size());
        jobs_.push_back(std::move(j));
        return (int)jobs_.size() - 1;
    }
    const std::vector<Job>& jobs() const { return jobs_; }
    const BatchStats& stats() const { return stats_; }
    // effective cap of a job after the engine's KV-capacity clamp (host copy of the rule in b200_begin_sentences): set by the owner
    std::vector<int> room_of_voice;          // kv_capacity - voice_len[v]; empty = no clamp known
    int effective_cap(const Job& j) const {
        int cap = j.max_gen;
        if (j.voice >= 0 && j.voice < (int)room_of_voice.size()) cap = std::min(cap, room_of_voice[j.voice] - (int)j.ids.size());
        return std::max(cap, 0);
    }

    // Runs every queued job to completion. Returns the number of frames produced, or a negative engine error.
    long long run() { return pump(INT_MAX); }

    // Runs the refill -> submit -> collect loop until `max_steps` steps have been collected and at least one frame was produced, and
    // returns with `depth` steps in flight; once nothing is queued or running it drains the pipeline and returns. Jobs added since the last
    // call join the back of the queue, longest cap first. Returns the frames produced (0 = idle) or a negative engine error.
    long long pump(int max_steps) {
        using clk = std::chrono::steady_clock;
        admit();
        if (pending_.empty() && inflight_n_.empty() && busy_slots() == 0) return 0;
        const auto t0 = clk::now();
        if (pcm_.empty()) { pcm_.resize((size_t)n_slots_ * frame_); produced_.resize(n_slots_); }
        const long long frames0 = stats_.frames;
        long long collected = 0;
        for (;;) {
            if (!at_collect_) {
                int busy = 0, top = 0, n_free = 0;
                for (int s = 0; s < n_slots_; s++) { if (slots_[s].job >= 0) { busy++; top = s + 1; } else n_free++; }
                // ---- refill free slots ----
                if (!pending_.empty() && n_free > 0 && (busy == 0 || n_free >= std::min(refill_min, (int)pending_.size()) || since_refill_ >= refill_every)) {
                    std::vector<int32_t> sl, vo, toks, off{0}, mg, fae; std::vector<float> tp; std::vector<uint32_t> rs;
                    for (int s = 0; s < n_slots_ && !pending_.empty(); s++) {
                        if (slots_[s].job >= 0) continue;
                        const int j = pending_.front(); pending_.pop_front();
                        Job& J = jobs_[j];
                        if (effective_cap(J) <= 0) { J.done = true; stats_.sentences++; s--; continue; }   // no room (or empty cap): nothing to generate
                        slots_[s].job = j; slots_[s].live_from = submit_idx_; J.started = true;
                        // one allocation per sentence, sized by its cap (virtual memory only until frames arrive): growing the buffer frame by
                        // frame re-faulted every page several times and cost more host time per step than the GPU step itself
                        if (keep_pcm) J.pcm.reserve((size_t)effective_cap(J) * frame_);
                        sl.push_back(s); vo.push_back(J.voice); toks.insert(toks.end(), J.ids.begin(), J.ids.end()); off.push_back((int32_t)toks.size());
                        mg.push_back(J.max_gen); fae.push_back(J.fae); tp.push_back(J.temp); rs.push_back(J.rng_stream);
                    }
                    if (!sl.empty()) {
                        const auto tb = clk::now();
                        const int rc = ops_.begin(ops_.user, (int)sl.size(), sl.data(), vo.data(), toks.data(), off.data(), mg.data(), fae.data(), tp.data(), rs.data());
                        stats_.begin_ms += std::chrono::duration<double, std::milli>(clk::now() - tb).count();
                        if (rc != 0) return rc;
                        stats_.refills++; since_refill_ = 0;
                    }
                    busy = 0; top = 0;
                    for (int s = 0; s < n_slots_; s++) if (slots_[s].job >= 0) { busy++; top = s + 1; }
                }
                // ---- slots freed by cancel() that the refill did not reuse end on the engine before the next step ----
                if (!to_end_.empty()) {
                    std::vector<int32_t> ended;
                    for (int s : to_end_) if (slots_[s].job < 0) ended.push_back(s);
                    to_end_.clear();
                    if (!ended.empty() && ops_.end) {
                        const int rc = ops_.end(ops_.user, (int)ended.size(), ended.data());
                        if (rc != 0) return rc;
                    }
                }
                if (busy == 0 && pending_.empty() && inflight_n_.empty()) break;
                // ---- submit a step while work remains and the pipeline has room ----
                if (busy > 0 && (int)inflight_n_.size() < depth) {
                    int n = std::min(n_slots_, (top + range_quantum - 1) / range_quantum * range_quantum);
                    const auto ts = clk::now();
                    const int rc = ops_.submit(ops_.user, 0, n);
                    stats_.submit_ms += std::chrono::duration<double, std::milli>(clk::now() - ts).count();
                    if (rc != 0) return rc;
                    inflight_n_.push_back(n); submit_idx_++; since_refill_++;
                    stats_.steps++; stats_.slot_steps += n;
                    if ((int)inflight_n_.size() < depth) continue;     // fill the pipeline before the first collect
                }
                if (inflight_n_.empty()) continue;
                // enough for this call: stop in front of the collect with the pipeline full, the next call resumes right here
                if (busy > 0 && collected >= max_steps && stats_.frames > frames0) { at_collect_ = true; break; }
            }
            at_collect_ = false;
            // ---- collect the oldest step ----
            const int n = inflight_n_.front(); inflight_n_.pop_front();
            const auto tc0 = clk::now();
            const int rc = ops_.collect(ops_.user, pcm_.data(), produced_.data());
            stats_.collect_ms += std::chrono::duration<double, std::milli>(clk::now() - tc0).count();
            if (rc < 0) return rc;
            for (int s = 0; s < n; s++) {
                Slot& S = slots_[s];
                if (S.job < 0 || collect_idx_ < S.live_from) continue;          // frame of a previous (finished or cancelled) sentence in this slot
                Job& J = jobs_[S.job];
                bool finished = !produced_[s];
                if (produced_[s]) {
                    if (keep_pcm) J.pcm.insert(J.pcm.end(), pcm_.begin() + (size_t)s * frame_, pcm_.begin() + (size_t)(s + 1) * frame_);
                    J.frames++; stats_.frames++;
                    if (J.frames >= effective_cap(J)) finished = true;           // the device stops it at the cap as well: no need to wait for a 0 flag
                }
                if (finished) { J.done = true; stats_.sentences++; S.job = -1; }
            }
            collect_idx_++; collected++;
        }
        stats_.wall_ms += std::chrono::duration<double, std::milli>(clk::now() - t0).count();
        return stats_.frames - frames0;
    }

    // Collects the steps still in flight and drops their frames (the engine's submit ring is left empty).
    void drain() {
        if (pcm_.empty()) { pcm_.resize((size_t)n_slots_ * frame_); produced_.resize(n_slots_); }
        while (!inflight_n_.empty()) {
            inflight_n_.pop_front();
            if (ops_.collect(ops_.user, pcm_.data(), produced_.data()) < 0) break;
        }
        at_collect_ = false;
    }

    bool valid_utt(int utt) const { return utt >= 0 && utt < (int)utts_.size(); }
    int frames(int utt) const { int n = 0; for (int j : utts_[utt].jobs) n += jobs_[j].frames; return n; }

    // Frames pop() would hand out now: every frame of the sentences in order up to and including the first one still running.
    int ready(int utt) const {
        const Utt& U = utts_[utt];
        int n = 0;
        for (size_t k = U.next; k < U.jobs.size(); k++) {
            const Job& J = jobs_[U.jobs[k]];
            n += kept(J) - (k == U.next ? U.next_frame : 0);
            if (!J.done) break;
        }
        return n;
    }

    int pop(int utt, float* out, int max_frames) {
        Utt& U = utts_[utt];
        int n = 0;
        while (U.next < U.jobs.size()) {
            Job& J = jobs_[U.jobs[U.next]];
            const int m = std::min(kept(J) - U.next_frame, max_frames - n);
            if (m > 0) {
                memcpy(out + (size_t)n * frame_, J.pcm.data() + (size_t)U.next_frame * frame_, (size_t)m * frame_ * sizeof(float));
                n += m; U.next_frame += m;
            }
            if (!J.done || U.next_frame < kept(J)) break;
            std::vector<float>().swap(J.pcm);     // done and handed out: a streaming consumer holds only audio it has not received yet
            U.next++; U.next_frame = 0;
        }
        return n;
    }

    // The frames not popped yet, in order (all of them when pop() is not used).
    int read(int utt, float* out, int max_frames) const {
        const Utt& U = utts_[utt];
        int n = 0;
        for (size_t k = U.next; k < U.jobs.size() && n < max_frames; k++) {
            const Job& J = jobs_[U.jobs[k]];
            const int f0 = k == U.next ? U.next_frame : 0;
            const int m = std::min(kept(J) - f0, max_frames - n);
            if (m > 0) { memcpy(out + (size_t)n * frame_, J.pcm.data() + (size_t)f0 * frame_, (size_t)m * frame_ * sizeof(float)); n += m; }
        }
        return n;
    }

    // Queued sentences are dropped; running ones give up their slot at once: frames of steps already in flight for it are not attributed
    // (the slot's job is cleared, or the refill moves live_from past them) and the slot is ended on the engine before the next step unless a
    // refill reuses it. The utterance's audio not popped yet is freed.
    void cancel(int utt) {
        Utt& U = utts_[utt];
        if (U.cancelled || status(utt, nullptr) == kDone) return;
        U.cancelled = true;
        for (int j : U.jobs) {
            Job& J = jobs_[j];
            std::vector<float>().swap(J.pcm);
            if (J.done) continue;
            J.done = true;
            for (int s = 0; s < n_slots_; s++) if (slots_[s].job == j) { slots_[s].job = -1; to_end_.push_back(s); }
        }
        pending_.erase(std::remove_if(pending_.begin(), pending_.end(), [&](int j) { return jobs_[j].utt == utt; }), pending_.end());
    }

    int status(int utt, int* ready_frames) const {
        const Utt& U = utts_[utt];
        if (ready_frames) *ready_frames = U.cancelled ? 0 : ready(utt);
        if (U.cancelled) return kCancelled;
        bool all_done = true, any_started = false;
        for (int j : U.jobs) { all_done = all_done && jobs_[j].done; any_started = any_started || jobs_[j].started || jobs_[j].done; }
        return all_done ? kDone : any_started ? kRunning : kQueued;
    }

private:
    struct Slot { int job = -1; long long live_from = 0; };
    struct Utt { std::vector<int> jobs; size_t next = 0; int next_frame = 0; bool cancelled = false; };   // next / next_frame: pop cursor
    int kept(const Job& J) const { return (int)(J.pcm.size() / (size_t)frame_); }
    int busy_slots() const { int b = 0; for (const Slot& S : slots_) b += S.job >= 0; return b; }
    // jobs added since the last admission join the back of the queue, longest processing time (frame cap) first: within one admission the
    // long sentences start early and the tail is made of short ones; across admissions the queue is first come, first served
    void admit() {
        std::vector<int> order;
        for (size_t i = admitted_; i < jobs_.size(); i++) if (!jobs_[i].done) order.push_back((int)i);
        admitted_ = jobs_.size();
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return jobs_[a].max_gen > jobs_[b].max_gen; });
        pending_.insert(pending_.end(), order.begin(), order.end());
    }

    BatchOps ops_; int n_slots_, frame_;
    std::vector<Slot> slots_;
    std::vector<Job> jobs_;
    std::vector<Utt> utts_;
    BatchStats stats_;
    // loop state carried between pump() calls
    std::deque<int> pending_;                 // admitted jobs not started yet, in start order
    std::deque<int> inflight_n_;              // stepped slot count of each in-flight step, oldest first
    long long submit_idx_ = 0, collect_idx_ = 0;
    int since_refill_ = 1 << 30;
    bool at_collect_ = false;                 // the last pump stopped in front of a collect
    size_t admitted_ = 0;                     // jobs_[0, admitted_) have been admitted
    std::vector<int> to_end_;                 // slots freed by cancel() since the last iteration
    std::vector<float> pcm_; std::vector<int32_t> produced_;   // collect staging
};

}  // namespace ptts_host
