// Host side of the packed FASTQ slabs (wire.h): the expander that turns wire records back into FASTQ text.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

#include "wire.h"

namespace scs {

// Expand the wire records [w, w + n) into FASTQ text at `out`; qchar0 = '!' + qlo. Returns the text bytes written, or -1 when
// a record runs past n. simd = false forces the scalar path (the AVX2 path is taken only where the CPU has AVX2).
int64_t expand_wire(const uint8_t* w, uint64_t n, char* out, int qchar0, bool simd = true);
bool expand_has_avx2();

// One packed slab (both files) on its way from a pinned wire slot into the text slot that the consumer hands out.
struct ExpandJob {
    cudaEvent_t landed = nullptr;              // the wire slabs (and their split tables) sit in host memory once this fires (null: already there)
    const uint8_t* wire[2] = {nullptr, nullptr};   // per file: split table of nsplit entries, then the records
    uint32_t nsplit[2] = {0, 0};
    uint64_t wire_bytes[2] = {0, 0}, text_bytes[2] = {0, 0};   // records only
    char* out[2] = {nullptr, nullptr};
    int qchar0 = 33;
    bool scalar = false;                       // tests: the scalar expander
    // pool state
    uint64_t seq = 0; int left = 0; bool done = true, failed = false; double t_start = 0;
};

// Persistent host threads that expand packed slabs into FASTQ text. Jobs are taken in submission order; the first free thread
// waits for a job's copy to land, then every thread takes pieces of it (one split-table entry each).
class ExpandPool {
  public:
    ExpandPool(int device, int threads);   // device < 0: jobs carry no CUDA event
    ~ExpandPool();   // joins every thread; jobs still queued are finished first
    int threads() const { return (int)th_.size(); }
    void submit(ExpandJob* j);
    bool query(ExpandJob* j);
    int wait(ExpandJob* j);   // 0 when the job's text is complete, 1 when a slab was malformed or its copy failed
    void drain();             // every submitted job has finished
    double rate() const { return rate_.load(); }        // text bytes per second, moving average over finished jobs
    uint64_t queued_text() const { return queued_.load(); }

  private:
    struct Task { ExpandJob* j; int f, k; };   // f < 0: wait for the copy, then split the job into pieces
    void run();
    void finish_one(ExpandJob* j);
    int device_;
    std::mutex mu_; std::condition_variable cv_work_, cv_done_;
    std::deque<Task> q_; std::vector<std::thread> th_;
    bool stop_ = false; int active_jobs_ = 0; uint64_t seq_ = 0; double t_last_ = 0;
    std::atomic<double> rate_{0}; std::atomic<uint64_t> queued_{0};
};

}  // namespace scs
