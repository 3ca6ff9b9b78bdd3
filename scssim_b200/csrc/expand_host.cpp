// Host expansion of packed FASTQ slabs (wire.h) into FASTQ text.
#include "expand_host.h"

#include <immintrin.h>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

#include "wire.h"

namespace scs {

namespace {

constexpr size_t kMaxText = 3 + 255 + 2 * 65535 + 4;   // largest text of one record (a verbatim record is smaller)

int64_t expand_scalar(const uint8_t* w, uint64_t n, char* out, int qchar0) {
    uint64_t i = 0; int64_t o = 0;
    while (i < n) {
        if (n - i < 3) return -1;
        const uint32_t hl = w[i], len = w[i + 1] | ((uint32_t)w[i + 2] << 8);
        i += 3;
        if (hl == (uint32_t)wire::kVerbatim) {
            if (n - i < len) return -1;
            memcpy(out + o, w + i, len); o += len; i += len;
            continue;
        }
        if (n - i < (uint64_t)hl + len) return -1;
        memcpy(out + o, w + i, hl); o += hl; i += hl;
        char* s = out + o; char* q = s + len + 3;
        for (uint32_t k = 0; k < len; k++) { s[k] = "ACGT"[w[i + k] & 3]; q[k] = (char)(qchar0 + (w[i + k] >> 2)); }
        s[len] = '\n'; s[len + 1] = '+'; s[len + 2] = '\n'; q[len] = '\n';
        o += 2 * (int64_t)len + 4; i += len;
    }
    return o;
}

#pragma GCC push_options
#pragma GCC target("avx2")
// AVX2: records are expanded with plain stores into a small per-thread buffer that is kept at the destination's 32-byte
// phase, and every full 32-byte line of it leaves with a streaming store, so the destination is never read for ownership.
// Only the first and last partial lines of a call are written with ordinary stores.
struct alignas(64) Bounce {
    static constexpr size_t kFlush = 16384;
    char buf[kFlush + kMaxText + 64];
};

void flush_lines(char*& dst, char* buf, size_t& n, size_t& skip) {
    const size_t lines = n / 32;
    size_t l = 0;
    if (skip && lines) { memcpy(dst + skip, buf + skip, 32 - skip); skip = 0; l = 1; }
    for (; l < lines; l++) _mm256_stream_si256(reinterpret_cast<__m256i*>(dst + 32 * l), _mm256_load_si256(reinterpret_cast<const __m256i*>(buf + 32 * l)));
    const size_t rest = n - 32 * lines;
    if (lines) { memcpy(buf, buf + 32 * lines, rest); dst += 32 * lines; n = rest; }
}

int64_t expand_avx2(const uint8_t* w, uint64_t n, char* out, int qchar0) {
    static thread_local Bounce* B = nullptr;
    if (!B) { B = static_cast<Bounce*>(aligned_alloc(64, sizeof(Bounce))); if (!B) return expand_scalar(w, n, out, qchar0); }
    char* const buf = B->buf;
    char* dst = reinterpret_cast<char*>(reinterpret_cast<uintptr_t>(out) & ~(uintptr_t)31);
    size_t skip = (size_t)(out - dst), fill = skip;   // buf[0, skip) stands for bytes before `out`: never written
    const __m256i lut = _mm256_setr_epi8('A', 'C', 'G', 'T', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 'A', 'C', 'G', 'T', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0);
    const __m256i m3 = _mm256_set1_epi8(3), m63 = _mm256_set1_epi8(63), qoff = _mm256_set1_epi8((char)qchar0);
    const uint8_t* const wend = w + n;
    uint64_t i = 0; int64_t total = 0;
    while (i < n) {
        if (n - i < 3) return -1;
        const uint32_t hl = w[i], len = w[i + 1] | ((uint32_t)w[i + 2] << 8);
        i += 3;
        char* o = buf + fill;
        if (hl == (uint32_t)wire::kVerbatim) {
            if (n - i < len) return -1;
            memcpy(o, w + i, len); i += len; fill += len; total += len;
        } else {
            if (n - i < (uint64_t)hl + len) return -1;
            const uint8_t* h = w + i;
            if (h + ((hl + 31) & ~31u) <= wend)
                for (uint32_t k = 0; k < hl; k += 32) _mm256_storeu_si256(reinterpret_cast<__m256i*>(o + k), _mm256_loadu_si256(reinterpret_cast<const __m256i*>(h + k)));
            else memcpy(o, h, hl);
            const uint8_t* c = h + hl; char* s = o + hl; char* q = s + len + 3;
            auto put = [&](uint32_t k) {
                const __m256i v = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(c + k));
                _mm256_storeu_si256(reinterpret_cast<__m256i*>(s + k), _mm256_shuffle_epi8(lut, _mm256_and_si256(v, m3)));
                _mm256_storeu_si256(reinterpret_cast<__m256i*>(q + k), _mm256_add_epi8(_mm256_and_si256(_mm256_srli_epi16(v, 2), m63), qoff));
            };
            uint32_t k = 0;
            for (; k + 32 <= len; k += 32) put(k);
            if (k < len) {
                if (len >= 32) put(len - 32);   // the last 32 positions again: no read past the record
                else for (; k < len; k++) { s[k] = "ACGT"[c[k] & 3]; q[k] = (char)(qchar0 + (c[k] >> 2)); }
            }
            s[len] = '\n'; s[len + 1] = '+'; s[len + 2] = '\n'; q[len] = '\n';
            const uint32_t t = hl + 2 * len + 4;
            i += hl + len; fill += t; total += t;
        }
        if (fill >= Bounce::kFlush) flush_lines(dst, buf, fill, skip);
    }
    flush_lines(dst, buf, fill, skip);
    if (fill > skip) memcpy(dst + skip, buf + skip, fill - skip);
    _mm_sfence();
    return total;
}
#pragma GCC pop_options

}  // namespace

bool expand_has_avx2() {
    static const bool yes = __builtin_cpu_supports("avx2");
    return yes;
}

int64_t expand_wire(const uint8_t* w, uint64_t n, char* out, int qchar0, bool simd) {
    return simd && expand_has_avx2() ? expand_avx2(w, n, out, qchar0) : expand_scalar(w, n, out, qchar0);
}

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

ExpandPool::ExpandPool(int device, int threads) : device_(device) {
    for (int t = 0; t < std::max(1, threads); t++) th_.emplace_back([this] { run(); });
}

ExpandPool::~ExpandPool() {
    { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
    cv_work_.notify_all();
    for (auto& t : th_) t.join();
}

void ExpandPool::submit(ExpandJob* j) {
    {
        std::lock_guard<std::mutex> lk(mu_);
        j->seq = ++seq_; j->done = false; j->failed = false; j->left = 0;
        active_jobs_++;
        q_.push_back({j, -1, 0});
    }
    queued_ += j->text_bytes[0] + j->text_bytes[1];
    cv_work_.notify_one();
}

bool ExpandPool::query(ExpandJob* j) { std::lock_guard<std::mutex> lk(mu_); return j->done; }

int ExpandPool::wait(ExpandJob* j) {
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] { return j->done; });
    return j->failed ? 1 : 0;
}

void ExpandPool::drain() {
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] { return active_jobs_ == 0; });
}

// called with mu_ held
void ExpandPool::finish_one(ExpandJob* j) {
    if (--j->left > 0) return;
    const double t = now_s(), dt = t - std::max(j->t_start, t_last_);
    const uint64_t text = j->text_bytes[0] + j->text_bytes[1];
    if (!j->failed && dt > 0 && text) {
        const double r = text / dt, old = rate_.load();
        rate_ = old > 0 ? 0.75 * old + 0.25 * r : r;
    }
    t_last_ = t;
    queued_ -= text;
    j->done = true; active_jobs_--;
    cv_done_.notify_all();
}

void ExpandPool::run() {
    if (device_ >= 0) cudaSetDevice(device_);
    for (;;) {
        Task t;
        {
            std::unique_lock<std::mutex> lk(mu_);
            cv_work_.wait(lk, [&] { return stop_ || !q_.empty(); });
            if (q_.empty()) return;
            t = q_.front(); q_.pop_front();
        }
        ExpandJob* j = t.j;
        if (t.f < 0) {   // the copy of the wire slab must land before any piece of it is read
            cudaError_t e = cudaSuccess;
            if (j->landed) while ((e = cudaEventQuery(j->landed)) == cudaErrorNotReady) std::this_thread::sleep_for(std::chrono::microseconds(20));
            std::lock_guard<std::mutex> lk(mu_);
            j->t_start = now_s();
            j->left = 1;   // released below, after every piece is queued
            if (e != cudaSuccess) j->failed = true;
            else {
                // pieces go to the front of the queue, in slab order, ahead of later jobs
                std::vector<Task> pieces;
                for (int f = 0; f < 2; f++) for (uint32_t k = 0; k < j->nsplit[f]; k++) pieces.push_back({j, f, (int)k});
                for (auto it = pieces.rbegin(); it != pieces.rend(); ++it) q_.push_front(*it);
                j->left += (int)pieces.size();
            }
            finish_one(j);
            cv_work_.notify_all();
            continue;
        }
        const wire::Split* sp = reinterpret_cast<const wire::Split*>(j->wire[t.f]);
        const uint8_t* rec = j->wire[t.f] + (size_t)j->nsplit[t.f] * sizeof(wire::Split);
        const wire::Split a = sp[t.k];
        const wire::Split b = (uint32_t)t.k + 1 < j->nsplit[t.f] ? sp[t.k + 1] : wire::Split{j->wire_bytes[t.f], j->text_bytes[t.f]};
        bool ok = a.wire <= b.wire && b.wire <= j->wire_bytes[t.f] && a.text <= b.text && b.text <= j->text_bytes[t.f];
        if (ok) ok = expand_wire(rec + a.wire, b.wire - a.wire, j->out[t.f] + a.text, j->qchar0, !j->scalar) == (int64_t)(b.text - a.text);
        std::lock_guard<std::mutex> lk(mu_);
        if (!ok) j->failed = true;
        finish_one(j);
    }
}

}  // namespace scs
