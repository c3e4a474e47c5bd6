// Run-time specialisation of the scan kernel: the template in use is compiled into the kernel with
// NVRTC (libnvrtc is opened with dlopen; nothing links against it), the cubin is loaded through the
// CUDA runtime's library API and cached for the life of the process.
#pragma once

#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "handlers_params.hpp"
#include "template_spec.hpp"

namespace scg {

struct SpecSingleConfig {
    std::string fbases, rbases;   // forward / reverse-complemented template, '-' for variable positions
    int T = 0, fwd = 0, rev = 0;
    int W = 0;                    // words per plane of the batch
    int nb = 1;                   // window blocks needed by the longest read of the batch
    int cb = 0, mm = 0, maxmm = 0, use_first = 1;
    int fstart = 0, rstart = 0, keylen = 0;
    std::vector<uint32_t> seed_masks;   // pigeonhole seeds of the libraries (empty = deferred reads take the generic search)
    int dup_first = 0;
    // > 0: every read of the batch has this length (or, with `ragged`, at most this length): the uniform-length kernel (filter + verify
    // scan, several tiles per bulk copy) is compiled instead of the general one
    int ulen = 0;
    int info = 1;                 // the per-read info word may be asked for
    int joint = 0;                // the joint exact table of both strands is there (keys of up to 31 bases)
    int has_index = 1;            // the per-read index is asked for
    int ibuckets = 0;             // seed buckets with the first candidate inline are there
    int ragged = 0;               // the batch carries per-read lengths (ulen is then the longest read)
    int hist = 0;                 // > 0: counters privatised in shared memory, this many (pool size rounded up), flushed at the end
    std::string key() const;
};

// One run-time compiled module: program text (a few #defines + an #include of an embedded header) and the kernels wanted
// from it.  Modules are cached per process (by device and text) and ON DISK (SCG_CACHE_DIR, else $XDG_CACHE_HOME or
// ~/.cache/screencounter_b200; SCG_NO_DISK_CACHE=1 turns it off), keyed by the program text, a hash of the embedded headers,
// the NVRTC version and the target, so that a fresh process pays a file read instead of a compilation.
struct JitProgram {
    std::string name;                  // file name shown in diagnostics
    std::string text;
    std::vector<std::string> kernels;  // extern "C" kernel names
};
struct JitModule {
    cudaLibrary_t library = nullptr;
    std::vector<cudaKernel_t> kernels; // in the order asked for
    std::string problem;
    bool from_disk = false;
    double build_s = 0;                // compile (or disk read) + load
};
// nullptr (reason in *why) when run-time compilation is unavailable, disabled (SCG_NO_SPECIALIZE=1) or fails.  Thread-safe.
const JitModule* jit_module(const JitProgram& prog, int device, std::string* why);
// seconds this process has spent building or loading modules so far (reported as part of setup_s)
double jit_seconds_total();
// integer tuning knob from the environment, clamped to [lo, hi]
int jit_env_int(const char* name, int fallback, int lo, int hi);

// Returns a launchable kernel for the configuration, or nullptr (with the reason in *why) when
// run-time compilation is unavailable or disabled (SCG_NO_SPECIALIZE=1); callers then use the
// generic kernel.  Thread-safe.
// With cfg.ulen > 0 the module also holds the follow-up kernel for the reads the uniform-length kernel lists as needing
// the full per-read search; *slow receives it.
cudaKernel_t specialised_single_kernel(const SpecSingleConfig& cfg, int device, std::string* why, cudaKernel_t* slow = nullptr);

// Blocks of 128 threads of a specialised kernel that fit on one SM (occupancy query, cached per kernel).
int specialised_blocks_per_sm(cudaKernel_t kernel);

// Human-readable status of the run-time compiler ("nvrtc 12.9 from <path>" or why it is missing).
std::string jit_status();

} // namespace scg
