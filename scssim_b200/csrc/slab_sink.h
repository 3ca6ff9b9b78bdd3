// Consumer side of the FASTQ slab pipeline (replaces the hand-off between Amplicon::yieldReads' per-thread buffers and
// SeqWriter::write, /root/reference/lib/amplicon/Amplicon.cpp:413-424,536-541, lib/seqwriter/SeqWriter.cpp:41-54).
//
// The read stage produces packed slabs on the device and copies each one into a slot of a ring of pinned host buffers.
// A consumer decides how many slots the ring has and when a slot may be overwritten:
//   * CallbackConsumer (scs_yield_reads_sink): 4 slots, the user's function is called on the launching thread, in file order;
//     it also takes slabs that host threads expand from packed records (host_expand), so emit (k), copy (k-1) and expansion
//     (k-2) overlap;
//   * AsyncFileConsumer (scs_yield_reads, file_sink.h): N slots drained by writer threads — the launching thread only
//     blocks when every slot is still waiting for the disk.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/scssim_b200.h"

namespace scs {

class ExpandPool; struct ExpandJob;

struct SlabConsumer {
    virtual ~SlabConsumer() {}
    // pinned ring slots per file (>= 2)
    virtual int ring_slots() const = 0;
    // Offset inside the pinned slot at which the next slab of `file` must start (< 4096). File sinks that write with O_DIRECT
    // ask for the slab to sit at its file offset modulo the block size, so memory and file alignment agree; 0 otherwise.
    virtual uint64_t phase(int file) const = 0;
    // Block until ring slot `slot` may be overwritten. Returns non-zero on a sink failure.
    virtual int acquire(int slot) = 0;
    // The copies of one slab into `slot` have been enqueued; `copied` fires when they have landed. p[f] points at the first byte
    // of file f's data (slot base + phase), bytes[f] may be 0.
    virtual int submit(int slot, cudaEvent_t copied, char* const p[2], const uint64_t bytes[2]) = 0;
    // Same for a slab whose text the expansion pool writes into `slot`: ready once pool->wait(job) returns. Only consumers
    // whose takes_expanded() is true receive such slabs.
    virtual bool takes_expanded() const { return false; }
    virtual int submit_expanded(int, ExpandPool*, ExpandJob*, char* const[2], const uint64_t[2]) { return 1; }
    // Give the consumer a chance to work on the launching thread (callback sinks call the user function here).
    virtual int service() = 0;
    // Everything submitted is consumed when this returns.
    virtual int finish() = 0;
};

// scs_sink_fn adapter: kSlots ring slots, the user's function runs on the launching thread in slab order (fn may be null: discard)
struct CallbackConsumer : SlabConsumer {
    static constexpr int kSlots = 4;
    CallbackConsumer(scs_sink_fn f, void* u);
    int ring_slots() const override { return kSlots; }
    uint64_t phase(int) const override { return 0; }
    int acquire(int slot) override;
    int submit(int slot, cudaEvent_t copied, char* const p[2], const uint64_t bytes[2]) override;
    bool takes_expanded() const override { return true; }
    int submit_expanded(int slot, ExpandPool* pool, ExpandJob* job, char* const p[2], const uint64_t bytes[2]) override;
    int service() override;
    int finish() override;

  private:
    int consume_front(bool wait);
    struct Pending {
        bool live = false; cudaEvent_t ev = nullptr; ExpandPool* pool = nullptr; ExpandJob* job = nullptr;
        char* p[2] = {nullptr, nullptr}; uint64_t n[2] = {0, 0};
    } pend[kSlots];
    scs_sink_fn fn; void* user; int head = 0, count = 0;
};

}  // namespace scs
