// Run-time specialisation of the generic one-launch program: NVRTC compiles generic_program_jit.cuh with the
// registration (schema, systems, checksummed byte ranges) as compile-time constants, the cubin is loaded with
// cudaLibraryLoadData and launched like any other kernel of the engine.
//
// * libnvrtc is dlopen()ed on first use: the shared library has no link-time dependency on it, and an installation
//   without NVRTC simply keeps the interpreter kernel (generic_program.cuh) — still the GPU, never a CPU path.
// * the kernel sources are the .cuh files next to the shared library (<dir of libbevy_ggrs_b200.so>/csrc, or
//   $BGR_JIT_SRC_DIR); they are handed to NVRTC as in-memory headers, no include path, no host headers.
// * compiled programs are cached per process by their generated prelude: engines with the same registration share one.
// * for registrations of compiled-in systems every failure (no NVRTC, no sources, compile error) is reported once on
//   stderr when BGR_JIT_VERBOSE is set and otherwise silently falls back to the interpreter; results are identical either
//   way (tests run both).  A registration with user systems (user_system.cuh) has no interpreter: bgr_build fails with
//   the reason, and with NVRTC's log for a compile error.
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <map>
#include <mutex>
#include <sstream>
#include <string>
#include <vector>

namespace bgr {

struct JitKernel {
    const void* fn = nullptr;  // cudaKernel_t, usable wherever the runtime takes a kernel's `const void* func`
    int threads = 0;
    int item_rows = 0;         // rows per work item (set by the caller)
    int bps = 0;               // resident blocks per SM (occupancy query)
};

namespace jit_detail {

typedef struct _nvrtcProgram* nvrtcProgram;
struct NvrtcApi {
    void* h = nullptr;
    int (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
    int (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
    int (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
    int (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
    int (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
    int (*DestroyProgram)(nvrtcProgram*) = nullptr;
    bool ok = false;
};

inline NvrtcApi& nvrtc() {
    static NvrtcApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"};
        for (const char* n : names)
            if ((api.h = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
        if (!api.h) return;
        auto sym = [&](const char* s) { return dlsym(api.h, s); };
        api.CreateProgram = reinterpret_cast<decltype(api.CreateProgram)>(sym("nvrtcCreateProgram"));
        api.CompileProgram = reinterpret_cast<decltype(api.CompileProgram)>(sym("nvrtcCompileProgram"));
        api.GetCUBINSize = reinterpret_cast<decltype(api.GetCUBINSize)>(sym("nvrtcGetCUBINSize"));
        api.GetCUBIN = reinterpret_cast<decltype(api.GetCUBIN)>(sym("nvrtcGetCUBIN"));
        api.GetProgramLogSize = reinterpret_cast<decltype(api.GetProgramLogSize)>(sym("nvrtcGetProgramLogSize"));
        api.GetProgramLog = reinterpret_cast<decltype(api.GetProgramLog)>(sym("nvrtcGetProgramLog"));
        api.DestroyProgram = reinterpret_cast<decltype(api.DestroyProgram)>(sym("nvrtcDestroyProgram"));
        api.ok = api.CreateProgram && api.CompileProgram && api.GetCUBINSize && api.GetCUBIN && api.GetProgramLogSize &&
                 api.GetProgramLog && api.DestroyProgram;
    });
    return api;
}

inline bool read_file(const std::string& path, std::string* out) {
    std::ifstream f(path, std::ios::binary);
    if (!f) return false;
    std::ostringstream ss;
    ss << f.rdbuf();
    *out = ss.str();
    return true;
}

// directory of the kernel sources: next to this shared library
inline std::string source_dir(const void* any_symbol_of_this_library) {
    if (const char* d = std::getenv("BGR_JIT_SRC_DIR")) return d;
    Dl_info info;
    if (!dladdr(any_symbol_of_this_library, &info) || !info.dli_fname) return "";
    std::string p = info.dli_fname;
    const size_t slash = p.find_last_of('/');
    return (slash == std::string::npos ? std::string(".") : p.substr(0, slash)) + "/csrc";
}

struct Cached {
    JitKernel k;               // fn == nullptr: the compile failed
    std::string why;           // ... and why
    bool compile_error = false;  // NVRTC rejected the source (as opposed to: no NVRTC, no sources, load failure)
};
struct Cache {
    std::mutex mu;
    std::map<std::string, Cached> programs;  // by prelude
};
inline Cache& cache() { static Cache c; return c; }

}  // namespace jit_detail

// Compile (or fetch) the specialised kernel for `prelude` (the generated #defines and user sources).  Returns false and
// leaves the reason in *why (*compile_error: NVRTC rejected the source, *why holds its log) when it cannot be had.
inline bool jit_generic_program(const std::string& prelude, int threads, const void* any_symbol_of_this_library, JitKernel* out,
                                std::string* why, bool* compile_error) {
    using namespace jit_detail;
    Cache& c = cache();
    std::lock_guard<std::mutex> lock(c.mu);
    *compile_error = false;
    auto it = c.programs.find(prelude);
    if (it != c.programs.end()) {
        *out = it->second.k;
        *why = it->second.why;
        *compile_error = it->second.compile_error;
        return out->fn != nullptr;
    }
    JitKernel k;
    auto finish = [&](bool ok) {
        Cached& e = c.programs[prelude];
        e.k = ok ? k : JitKernel{};
        e.why = ok ? std::string() : *why;
        e.compile_error = *compile_error;
        if (ok) *out = k;
        return ok;
    };
    NvrtcApi& api = nvrtc();
    if (!api.ok) { *why = "libnvrtc not found"; return finish(false); }
    const std::string dir = source_dir(any_symbol_of_this_library);
    const char* files[] = {"generic_program_jit.cuh", "generic_program.cuh", "kernels.cuh", "seahash.cuh", "tma_copy.cuh", "rtc_prelude.cuh",
                           "user_system.cuh"};
    std::vector<std::string> contents(sizeof files / sizeof *files);
    for (size_t i = 0; i < contents.size(); ++i)
        if (!read_file(dir + "/" + files[i], &contents[i])) { *why = "kernel source not found: " + dir + "/" + files[i]; return finish(false); }
    std::vector<const char*> hdr, names;
    for (size_t i = 0; i < contents.size(); ++i) { hdr.push_back(contents[i].c_str()); names.push_back(files[i]); }
    const std::string src = prelude + "#include \"generic_program_jit.cuh\"\n";
    nvrtcProgram prog = nullptr;
    if (api.CreateProgram(&prog, src.c_str(), "bgr_generic_jit.cu", int(hdr.size()), hdr.data(), names.data()) != 0) {
        *why = "nvrtcCreateProgram failed";
        return finish(false);
    }
    int dev = 0, major = 0, minor = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    // sm_100a like the rest of the library on a B200; the device's own architecture elsewhere
    const std::string arch = "--gpu-architecture=sm_" + std::to_string(major * 10 + minor) + (major >= 9 ? "a" : "");
    // -fmad=false: every f32 mul / add individually rounded, like the library's own build (bit-exact with the CPU)
    const char* opts[] = {arch.c_str(), "-std=c++17", "-fmad=false", "-lineinfo"};
    const int rc = api.CompileProgram(prog, int(sizeof opts / sizeof *opts), opts);
    if (rc != 0) {
        size_t n = 0;
        api.GetProgramLogSize(prog, &n);
        std::string log(n, '\0');
        if (n) api.GetProgramLog(prog, &log[0]);
        api.DestroyProgram(&prog);
        *why = "NVRTC compile error:\n" + log;
        *compile_error = true;
        return finish(false);
    }
    size_t n = 0;
    api.GetCUBINSize(prog, &n);
    std::vector<char> cubin(n);
    api.GetCUBIN(prog, cubin.data());
    api.DestroyProgram(&prog);
    cudaLibrary_t lib = nullptr;
    cudaError_t e = cudaLibraryLoadData(&lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) { *why = std::string("cudaLibraryLoadData: ") + cudaGetErrorString(e); (void)cudaGetLastError(); return finish(false); }
    cudaKernel_t kern = nullptr;
    e = cudaLibraryGetKernel(&kern, lib, "k_generic_jit");
    if (e != cudaSuccess) { *why = std::string("cudaLibraryGetKernel: ") + cudaGetErrorString(e); (void)cudaGetLastError(); cudaLibraryUnload(lib); return finish(false); }
    k.fn = reinterpret_cast<const void*>(kern);
    k.threads = threads;
    int nb = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k.fn, threads, 0);
    if (e != cudaSuccess) { (void)cudaGetLastError(); nb = 2; }
    k.bps = nb > 0 ? nb : 1;
    return finish(true);  // the library stays loaded for the life of the process (shared by every engine with this registration)
}

}  // namespace bgr
