// Packed FASTQ slab ("wire" slab): what the read stage sends over the host link for a slab that host threads expand back into
// FASTQ text (expand_host.h). Shared by the device packer (reads.cu) and the host expander.
//
// A wire slab is a sequence of records, each one of
//   packed:   u8 hl (< kVerbatim), u16 np (little endian), hl bytes of header text ("@amp#frag/m\n"), then np code bytes
//             base | (q - qlo) << 2, base in ACGT = 0..3 and q the Phred index; it expands to
//             header, np bases, "\n+\n", np characters '!' + q, "\n"  (hl + 2 np + 4 bytes of text)
//   verbatim: u8 kVerbatim, u16 n, then n bytes of text unchanged (a record with an N base or a quality outside
//             [qlo, qlo + 63] — so any genome and any profile round-trips exactly)
// Next to the records, a split table gives one {wire offset, text offset} pair for every kSplitEvery-th record, so that host
// threads can expand independent pieces of one slab.
#pragma once
#include <stdint.h>

namespace scs {
namespace wire {

constexpr int kVerbatim = 0xFF;
constexpr int kQualSpan = 64;
constexpr int kSplitEvery = 2048;

struct Split { uint64_t wire, text; };

#ifdef __CUDACC__
__host__ __device__
#endif
inline uint32_t packed_bytes(uint32_t hl, uint32_t np) { return 3u + hl + np; }

}  // namespace wire
}  // namespace scs
