// DEFLATE (RFC 1951) on the device, one warp per gzip member: what lets block-gzip FASTQ (BGZF -- bgzip, bcl-convert) cross
// PCIe COMPRESSED and be inflated in HBM, straight into the text ring of the device-side FASTQ reader (ingest.cu).  The
// reference inflates with zlib on its one reader thread (byteme::GzipFileReader, inst/include/byteme/GzipFileReader.hpp:39-51).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

namespace scg {

// One member: a raw deflate stream and where its text goes.
struct InflateMember {
    uint32_t in_off;    // byte offset of the raw deflate stream in the compressed image
    uint32_t in_len;    // its length in bytes
    uint32_t out_off;   // byte offset of the member's text in the output
    uint32_t out_len;   // bytes of text (ISIZE of the gzip trailer)
    uint32_t crc;       // CRC-32 of the text (gzip trailer)
};

// Inflates members [0, n) of `comp` into `out`, then checks every member's CRC-32.  errors (device, one word, not reset here)
// is OR-ed with 1 when a stream is malformed or does not produce exactly out_len bytes, with 2 when a CRC does not match.  `comp`
// must be readable for 512 bytes beyond the last member (the readers fetch whole 128-byte lines ahead).  Returns the number of
// kernels launched.
int launch_inflate(const uint8_t* comp, const InflateMember* members, int n, uint8_t* out, uint32_t* errors, int sm_count, cudaStream_t stream);

} // namespace scg
