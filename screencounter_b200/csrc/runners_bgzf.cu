// Block gzip through the C ABI: the compressor that writes test and benchmark inputs (the counterpart of what bgzip /
// bcl-convert produce), and the device inflater on its own (what the device-side FASTQ reader runs per chunk, ingest.cu),
// for tests and measurements.
#include <algorithm>
#include <cstring>

#include "api_common.hpp"
#include "bgzf.hpp"
#include "inflate.cuh"

using namespace scg;

extern "C" {

int scg_bgzf_compress(const char* text, size_t size, int level, int block_text, int nthreads, void* out, size_t capacity, size_t* used) {
    try {
        if (!used) throw Error("scg_bgzf_compress: null output size");
        *used = bgzf_compress(text, size, level, block_text > 0 ? (size_t)block_text : 0xff00, std::max(1, nthreads),
                              static_cast<unsigned char*>(out), capacity);
        return 0;
    } catch (const std::exception& e) {
        creation_error() = e.what();
        return 1;
    }
}

int scg_bgzf_inflate(scg_ctx* ctx, const void* image, size_t size, char* text, size_t capacity, size_t* text_size, double* device_ms) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        BgzfIndex index;
        if (!bgzf_index(static_cast<const unsigned char*>(image), size, index)) throw Error("not a block-gzip image");
        if (text_size) *text_size = index.text_size();
        if (!text) return;
        if (capacity < index.text_size()) throw Error("scg_bgzf_inflate: output buffer too small");
        if (size >= (1ull << 32) || index.text_size() >= (1ull << 32)) throw Error("scg_bgzf_inflate: images of 4 GiB or more are inflated chunk by chunk by the reader");
        c.ensure_ready();
        const size_t n = index.blocks.size();
        std::vector<InflateMember> members(n);
        for (size_t b = 0; b < n; ++b) {
            const BgzfBlock& blk = index.blocks[b];
            members[b] = InflateMember{ (uint32_t)blk.data, blk.csize, (uint32_t)index.text_off[b], blk.isize, blk.crc };
        }
        DeviceBuffer d_comp, d_members, d_out, d_err;
        d_comp.alloc(size + 1024, false);
        d_members.upload(members.data(), n * sizeof(InflateMember), c.stream);
        d_out.alloc(index.text_size() + 256, false);
        d_err.alloc(16, true);
        SCG_CUDA_CHECK(cudaMemcpyAsync(d_comp.ptr, image, size, cudaMemcpyHostToDevice, c.stream));
        cudaEvent_t e0, e1;
        SCG_CUDA_CHECK(cudaEventCreate(&e0));
        SCG_CUDA_CHECK(cudaEventCreate(&e1));
        SCG_CUDA_CHECK(cudaEventRecord(e0, c.stream));
        c.launches += launch_inflate(d_comp.as<uint8_t>(), d_members.as<InflateMember>(), (int)n, d_out.as<uint8_t>(), d_err.as<uint32_t>(),
                                     c.sm_count, c.stream);
        SCG_CUDA_CHECK(cudaGetLastError());
        SCG_CUDA_CHECK(cudaEventRecord(e1, c.stream));
        uint32_t err = 0;
        SCG_CUDA_CHECK(cudaMemcpyAsync(&err, d_err.ptr, sizeof err, cudaMemcpyDeviceToHost, c.stream));
        if (index.text_size()) SCG_CUDA_CHECK(cudaMemcpyAsync(text, d_out.ptr, index.text_size(), cudaMemcpyDeviceToHost, c.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        if (device_ms) *device_ms = ms;
        if (err & 1u) throw Error("failed to inflate the block-gzip file (corrupt member)");
        if (err & 2u) throw Error("failed to inflate the block-gzip file (corrupt member: CRC mismatch)");
    });
}

} // extern "C"
