#include "jit.hpp"

#include <dlfcn.h>
#include <sys/stat.h>
#include <sys/types.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cstdio>

#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <sstream>
#include <vector>

#include "common.hpp"
#include "layout.hpp"

namespace scg {

namespace {

struct EmbeddedSource {
    const char* name;
    const char* text;
};
#include "embedded_sources.inc"

// the handful of NVRTC entry points used, resolved at run time
typedef struct _nvrtcProgram* nvrtcProgram;
typedef int nvrtcResult;
struct Nvrtc {
    void* handle = nullptr;
    std::string where;
    nvrtcResult (*Version)(int*, int*) = nullptr;
    nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    nvrtcResult (*DestroyProgram)(nvrtcProgram*) = nullptr;
    nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
    nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
    nvrtcResult (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
    nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
    nvrtcResult (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
    const char* (*GetErrorString)(nvrtcResult) = nullptr;
    std::string problem;
};

Nvrtc& nvrtc() {
    static Nvrtc n;
    static std::once_flag once;
    std::call_once(once, [] {
        std::vector<std::string> candidates;
        if (const char* env = std::getenv("SCG_NVRTC_PATH")) candidates.push_back(env);
        for (const char* name : { "libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so",
                                  "libnvrtc.so.13", "libnvrtc.so" }) {
            candidates.push_back(name);
        }
        // An explicit path wins; otherwise the NEWEST of the candidates: a host process may already carry an older NVRTC
        // under the bare soname (PyTorch bundles one), and the kernels are written against the toolkit's PTX version.
        int best_version = -1;
        for (size_t k = 0; k < candidates.size(); ++k) {
            void* h = dlopen(candidates[k].c_str(), RTLD_NOW | RTLD_LOCAL);
            if (!h) continue;
            int major = 0, minor = 0;
            auto version = reinterpret_cast<nvrtcResult (*)(int*, int*)>(dlsym(h, "nvrtcVersion"));
            if (version) version(&major, &minor);
            const int v = (k == 0 && std::getenv("SCG_NVRTC_PATH")) ? (1 << 30) : major * 1000 + minor;
            if (v > best_version) {
                if (n.handle) dlclose(n.handle);
                n.handle = h;
                n.where = candidates[k];
                best_version = v;
            } else {
                dlclose(h);
            }
        }
        if (!n.handle) {
            n.problem = "libnvrtc not found (set SCG_NVRTC_PATH)";
            return;
        }
#define SCG_NVRTC_SYM(field, name)                                                       \
    n.field = reinterpret_cast<decltype(n.field)>(dlsym(n.handle, name));                \
    if (!n.field) {                                                                      \
        n.problem = std::string("libnvrtc lacks ") + name;                               \
        return;                                                                          \
    }
        SCG_NVRTC_SYM(Version, "nvrtcVersion")
        SCG_NVRTC_SYM(CreateProgram, "nvrtcCreateProgram")
        SCG_NVRTC_SYM(DestroyProgram, "nvrtcDestroyProgram")
        SCG_NVRTC_SYM(CompileProgram, "nvrtcCompileProgram")
        SCG_NVRTC_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
        SCG_NVRTC_SYM(GetProgramLog, "nvrtcGetProgramLog")
        SCG_NVRTC_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
        SCG_NVRTC_SYM(GetCUBIN, "nvrtcGetCUBIN")
        SCG_NVRTC_SYM(GetErrorString, "nvrtcGetErrorString")
#undef SCG_NVRTC_SYM
    });
    return n;
}

std::mutex g_mutex;
std::map<std::string, JitModule> g_cache;
double g_jit_seconds = 0;

// ---- on-disk cache of compiled modules ------------------------------------------------------------------------------
// A fresh process (every R session, every BiocParallel worker) would otherwise pay NVRTC for a kernel it compiled
// yesterday.  File = header (magic, key length, cubin length) + key text + cubin; the key holds the whole program text,
// a hash of the embedded headers, the NVRTC version and the target, and is compared in full on a hit.
std::string cache_dir() {
    if (const char* off = std::getenv("SCG_NO_DISK_CACHE")) {
        if (off[0] && off[0] != '0') return "";
    }
    std::string dir;
    if (const char* d = std::getenv("SCG_CACHE_DIR")) {
        dir = d;
    } else if (const char* x = std::getenv("XDG_CACHE_HOME")) {
        dir = std::string(x) + "/screencounter_b200";
    } else if (const char* h = std::getenv("HOME")) {
        dir = std::string(h) + "/.cache/screencounter_b200";
    } else {
        return "";
    }
    // mkdir -p, one level at a time
    for (size_t k = 1; k <= dir.size(); ++k) {
        if (k == dir.size() || dir[k] == '/') {
            const std::string part = dir.substr(0, k);
            if (::mkdir(part.c_str(), 0700) != 0 && errno != EEXIST) {
                struct stat sb;
                if (::stat(part.c_str(), &sb) != 0) return "";
            }
        }
    }
    return dir;
}

void hash_text(const std::string& text, unsigned long long& a, unsigned long long& b) {
    size_t i = 0;
    for (; i + 8 <= text.size(); i += 8) {
        unsigned long long w;
        std::memcpy(&w, text.data() + i, 8);
        a = mix64(a ^ w);
        b = (b ^ w) * 1099511628211ull + (b >> 29);
    }
    unsigned long long w = 0;
    if (i < text.size()) std::memcpy(&w, text.data() + i, text.size() - i);
    a = mix64(a ^ w ^ ((unsigned long long)text.size() << 40));
    b = (b ^ w) * 1099511628211ull + (b >> 29);
}

const std::string& embedded_fingerprint() {
    static const std::string fp = [] {
        unsigned long long a = 1469598103934665603ull, b = 0x9E3779B97F4A7C15ull;
        for (const auto& e : kEmbeddedSources) {
            hash_text(e.name, a, b);
            hash_text(e.text, a, b);
        }
        char buf[40];
        std::snprintf(buf, sizeof buf, "%016llx%016llx", a, b);
        return std::string(buf);
    }();
    return fp;
}

std::string disk_path(const std::string& dir, const std::string& disk_key) {
    unsigned long long a = 1469598103934665603ull, b = 0x9E3779B97F4A7C15ull;
    hash_text(disk_key, a, b);
    char buf[64];
    std::snprintf(buf, sizeof buf, "/%016llx%016llx.cubin", a, b);
    return dir + buf;
}

constexpr unsigned long long kDiskMagic = 0x3142554347435300ull;   // "\0SCGCUB1"

bool disk_load(const std::string& path, const std::string& disk_key, std::vector<char>& cubin) {
    FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) return false;
    unsigned long long head[3] = { 0, 0, 0 };
    bool ok = std::fread(head, sizeof head, 1, f) == 1 && head[0] == kDiskMagic && head[1] == disk_key.size() && head[2] > 0 &&
              head[2] < (1ull << 30);
    if (ok) {
        std::string key(head[1], '\0');
        ok = std::fread(&key[0], 1, key.size(), f) == key.size() && key == disk_key;
    }
    if (ok) {
        cubin.resize(head[2]);
        ok = std::fread(cubin.data(), 1, cubin.size(), f) == cubin.size();
    }
    std::fclose(f);
    return ok;
}

void disk_store(const std::string& path, const std::string& disk_key, const std::vector<char>& cubin) {
    const std::string tmp = path + ".tmp" + std::to_string((long long)::getpid());
    FILE* f = std::fopen(tmp.c_str(), "wb");
    if (!f) return;
    const unsigned long long head[3] = { kDiskMagic, disk_key.size(), cubin.size() };
    const bool ok = std::fwrite(head, sizeof head, 1, f) == 1 && std::fwrite(disk_key.data(), 1, disk_key.size(), f) == disk_key.size() &&
                    std::fwrite(cubin.data(), 1, cubin.size(), f) == cubin.size();
    if (std::fclose(f) == 0 && ok) {
        if (std::rename(tmp.c_str(), path.c_str()) != 0) std::remove(tmp.c_str());   // atomic: readers see a whole file or none
    } else {
        std::remove(tmp.c_str());
    }
}

double wall_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

} // namespace

std::string SpecSingleConfig::key() const {
    std::ostringstream o;
    o << fbases << '|' << rbases << '|' << T << '|' << fwd << rev << '|' << W << '|' << nb << '|' << cb << '|' << mm << '|' << maxmm << '|' << use_first << '|'
      << fstart << '|' << rstart << '|' << keylen << '|' << dup_first << '|' << ulen << '|' << info << '|' << joint << '|' << has_index << '|' << ibuckets << '|' << ragged
      << '|' << hist;
    for (uint32_t m : seed_masks) o << '|' << m;
    return o.str();
}

int specialised_blocks_per_sm(cudaKernel_t kernel) {
    static std::mutex m;
    static std::map<cudaKernel_t, int> cache;
    std::lock_guard<std::mutex> lock(m);
    auto it = cache.find(kernel);
    if (it != cache.end()) return it->second;
    int blocks = 0;
    // the tile rings live in (static) shared memory: ask for the largest carve-out so that registers, not the default
    // L1/shared split, decide how many blocks are resident
    if (const char* v = std::getenv("SCG_SPEC_CARVEOUT")) {
        cudaFuncSetAttribute(reinterpret_cast<const void*>(kernel), cudaFuncAttributePreferredSharedMemoryCarveout, std::atoi(v));
        cudaGetLastError();
    }
    cudaError_t st = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, reinterpret_cast<const void*>(kernel), 128, 0);
    if (st != cudaSuccess || blocks < 1) {
        cudaGetLastError();
        blocks = 4;
    }
    // SCG_SPEC_MAX_BLOCKS: fewer blocks than fit (every block's tile ring is shared memory taken from L1, which the scattered probes need)
    if (const char* v = std::getenv("SCG_SPEC_MAX_BLOCKS")) blocks = std::max(1, std::min(blocks, std::atoi(v)));
    cache[kernel] = blocks;
    return blocks;
}

std::string jit_status() {
    Nvrtc& n = nvrtc();
    if (!n.problem.empty()) return n.problem;
    int major = 0, minor = 0;
    n.Version(&major, &minor);
    return "nvrtc " + std::to_string(major) + "." + std::to_string(minor) + " from " + n.where;
}

const JitModule* jit_module(const JitProgram& prog, int device, std::string* why) {
    auto fail = [&](const std::string& msg) -> const JitModule* {
        if (why) *why = msg;
        return nullptr;
    };
    if (const char* env = std::getenv("SCG_NO_SPECIALIZE")) {
        if (env[0] && env[0] != '0') return fail("disabled by SCG_NO_SPECIALIZE");
    }
    Nvrtc& n = nvrtc();
    if (!n.problem.empty()) return fail(n.problem);
    const std::string key = std::to_string(device) + "#" + prog.text;
    std::lock_guard<std::mutex> lock(g_mutex);
    auto it = g_cache.find(key);
    if (it != g_cache.end()) {
        if (!it->second.problem.empty()) return fail(it->second.problem);
        return &it->second;
    }
    JitModule entry;
    auto remember = [&](const std::string& problem) -> const JitModule* {
        entry.problem = problem;
        g_cache[key] = entry;
        if (why) *why = problem;
        return nullptr;
    };
    const double t0 = wall_s();
    int major = 0, minor = 0;
    n.Version(&major, &minor);
    const std::string disk_key = "sm_100a|nvrtc " + std::to_string(major) + "." + std::to_string(minor) + "|" + embedded_fingerprint() + "|" + prog.text;
    const std::string dir = cache_dir();
    const std::string path = dir.empty() ? std::string() : disk_path(dir, disk_key);
    std::vector<char> cubin;
    if (!path.empty() && disk_load(path, disk_key, cubin)) {
        entry.from_disk = true;
    } else {
        std::vector<const char*> header_text, header_name;
        for (const auto& e : kEmbeddedSources) {
            header_text.push_back(e.text);
            header_name.push_back(e.name);
        }
        nvrtcProgram p = nullptr;
        nvrtcResult rc = n.CreateProgram(&p, prog.text.c_str(), prog.name.c_str(), (int)header_text.size(), header_text.data(), header_name.data());
        if (rc != 0) return remember(std::string("nvrtcCreateProgram: ") + n.GetErrorString(rc));
        const char* options[] = { "--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo" };
        rc = n.CompileProgram(p, (int)(sizeof(options) / sizeof(options[0])), options);
        if (rc != 0) {
            size_t log_size = 0;
            n.GetProgramLogSize(p, &log_size);
            std::string log(log_size, '\0');
            if (log_size) n.GetProgramLog(p, &log[0]);
            n.DestroyProgram(&p);
            return remember(std::string("nvrtcCompileProgram: ") + n.GetErrorString(rc) + "\n" + log);
        }
        size_t cubin_size = 0;
        n.GetCUBINSize(p, &cubin_size);
        cubin.resize(cubin_size);
        rc = n.GetCUBIN(p, cubin.data());
        n.DestroyProgram(&p);
        if (rc != 0 || cubin_size == 0) return remember("nvrtcGetCUBIN failed");
        if (!path.empty()) disk_store(path, disk_key, cubin);
    }
    if (const char* dump = std::getenv("SCG_DUMP_CUBIN")) {
        // profiling aid (tools/sass_hist.py): the module as loaded, one file per program name
        const std::string out = std::string(dump) + "/" + prog.name + ".cubin";
        if (FILE* f = std::fopen(out.c_str(), "wb")) {
            std::fwrite(cubin.data(), 1, cubin.size(), f);
            std::fclose(f);
        }
    }
    cudaError_t st = cudaLibraryLoadData(&entry.library, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (st != cudaSuccess) {
        cudaGetLastError();
        return remember(std::string("cudaLibraryLoadData: ") + cudaGetErrorString(st));
    }
    for (const std::string& name : prog.kernels) {
        cudaKernel_t k = nullptr;
        st = cudaLibraryGetKernel(&k, entry.library, name.c_str());
        if (st != cudaSuccess) {
            cudaGetLastError();
            return remember("cudaLibraryGetKernel(" + name + "): " + cudaGetErrorString(st));
        }
        entry.kernels.push_back(k);
    }
    entry.build_s = wall_s() - t0;
    g_jit_seconds += entry.build_s;
    auto& slot = g_cache[key];
    slot = entry;
    return &slot;
}

double jit_seconds_total() { return g_jit_seconds; }

int jit_env_int(const char* name, int fallback, int lo, int hi) {
    const char* v = std::getenv(name);
    if (!v || !*v) return fallback;
    int x = std::atoi(v);
    return x < lo ? lo : (x > hi ? hi : x);
}

cudaKernel_t specialised_single_kernel(const SpecSingleConfig& cfg, int device, std::string* why, cudaKernel_t* slow) {
    auto fail = [&](const std::string& msg) -> cudaKernel_t {
        if (why) *why = msg;
        return nullptr;
    };
    // register budget: 4 mismatch planes of W + 2 words must stay in registers (the uniform-length kernel, which does not keep
    // bit-sliced counters beside them, affords 10 words at 4 blocks/SM without spilling)
    if (cfg.W > (cfg.ulen > 0 ? 10 : 6)) {
        return fail(cfg.ulen > 0 ? "reads longer than 320 bases use the generic kernel" : "reads longer than 192 bases use the generic kernel");
    }
    if (cfg.T > 128) return fail("templates longer than 128 bases use the generic kernel");
    if (cfg.cb > 3) return fail("mismatch budgets above 7 use the generic kernel");
    if (cfg.keylen > 32) return fail("variable regions longer than 32 bases use the generic kernel");

    // tuning knobs (occupancy target and TMA ring depth) can be overridden for experiments
    // the uniform-length kernel keeps a read's words and mismatch planes in registers: 8 blocks of 128 threads fit up to
    // 96-base reads at 64 registers, longer reads trade occupancy for registers (the ALU pipe bounds those, and the sweeps in
    // profiles/r1_v10_long_reads_perf.txt are flat within 3 % between 4 and 8 blocks)
    const int min_blocks = jit_env_int("SCG_SPEC_MIN_BLOCKS", cfg.ulen > 0 ? (cfg.W <= 3 ? 8 : (cfg.W <= 6 ? 6 : 4)) : 4, 1, 16);
    const int stages = jit_env_int("SCG_SPEC_STAGES", 2, 1, 8);
    // tiles per bulk copy: two, or one where two would not fit the static shared memory (or would cost resident blocks: 192-base reads)
    const int group = jit_env_int("SCG_SPEC_GROUP", (cfg.ulen > 0 && cfg.W >= 6) ? 1 : 2, 1, 8);
    const int samples = jit_env_int("SCG_SPEC_SAMPLES", 8, 1, 32);

    std::string seed_list = "{ ";
    for (size_t k = 0; k < cfg.seed_masks.size(); ++k) seed_list += (k ? ", " : "") + std::to_string(cfg.seed_masks[k]) + "u";
    if (cfg.seed_masks.empty()) seed_list += "0u";
    seed_list += " }";
    std::ostringstream src;
    const int nb_max = (32 * cfg.W - cfg.T + 1 + 31) / 32;
    const int nb = std::max(1, std::min(cfg.nb, nb_max));
    src << "#define SPEC_CUSTOM 1\n"
        << "#define SPEC_T " << cfg.T << "\n"
        << "#define SPEC_FBASES \"" << cfg.fbases << "\"\n"
        << "#define SPEC_RBASES \"" << cfg.rbases << "\"\n"
        << "#define SPEC_FWD " << cfg.fwd << "\n"
        << "#define SPEC_REV " << cfg.rev << "\n"
        << "#define SPEC_W " << cfg.W << "\n"
        << "#define SPEC_NB " << nb << "\n"
        << "#define SPEC_CB " << cfg.cb << "\n"
        << "#define SPEC_MM " << cfg.mm << "\n"
        << "#define SPEC_MAXMM " << cfg.maxmm << "\n"
        << "#define SPEC_USE_FIRST " << cfg.use_first << "\n"
        << "#define SPEC_FSTART " << cfg.fstart << "\n"
        << "#define SPEC_RSTART " << cfg.rstart << "\n"
        << "#define SPEC_KEYLEN " << cfg.keylen << "\n"
        << "#define SPEC_NSEEDS " << cfg.seed_masks.size() << "\n"
        << "#define SPEC_SEEDMASKS " << seed_list << "\n"
        << "#define SPEC_DUP_FIRST " << cfg.dup_first << "\n"
        << "#define SPEC_NAME spec_single_kernel\n"
        << "#define SPEC_MIN_BLOCKS " << min_blocks << "\n"
        << "#define SPEC_STAGES " << stages << "\n"
        << "#define SPEC_ULEN " << cfg.ulen << "\n"
        << "#define SPEC_NAME_U spec_single_kernel_u\n"
        << "#define SPEC_NAME_SLOW spec_single_kernel_slow\n"
        << "#define SPEC_GROUP " << group << "\n"
        << "#define SPEC_SAMPLES " << samples << "\n"
        << "#define SPEC_INFO " << cfg.info << "\n"
        << "#define SPEC_JOINT " << cfg.joint << "\n"
        << "#define SPEC_HAS_INDEX " << cfg.has_index << "\n"
        << "#define SPEC_IBUCKETS " << cfg.ibuckets << "\n"
        << "#define SPEC_RAGGED " << cfg.ragged << "\n"
        << "#define SPEC_HIST " << cfg.hist << "\n"
        << "#define SPEC_UWARP " << jit_env_int("SCG_SPEC_UWARP", 0, 0, 1) << "\n"
        << "#define SPEC_SKIP_GENERAL " << (cfg.ulen > 0 ? 1 : 0) << "\n"
        << "#include \"spec_single.cuh\"\n";
    JitProgram prog;
    prog.name = "spec_single_jit.cu";
    prog.text = src.str();
    if (cfg.ulen > 0) {
        prog.kernels = { "spec_single_kernel_u", "spec_single_kernel_slow" };
    } else {
        prog.kernels = { "spec_single_kernel" };
    }
    const JitModule* mod = jit_module(prog, device, why);
    if (!mod) return nullptr;
    if (slow) *slow = cfg.ulen > 0 ? mod->kernels[1] : nullptr;
    return mod->kernels[0];
}

} // namespace scg
