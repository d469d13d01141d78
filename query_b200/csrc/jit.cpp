// jit.cpp — see jit.hpp
#include "jit.hpp"

#include <atomic>

#include <cuda.h>
#include <dlfcn.h>
#include <unistd.h>
#include <limits.h>
#include <nvrtc.h>
#include <stdlib.h>

#include <map>
#include <mutex>

#ifndef N1_CUDA_LIB
#define N1_CUDA_LIB "/usr/local/cuda/lib64"
#endif

namespace n1 {

// n1ql_device.cuh and the n1ql_value.cuh it includes, embedded at build time (Makefile: device_src.inc, value_src.inc)
static const char* k_device_header =
#include "device_src.inc"
    ;
static const char* k_value_header =
#include "value_src.inc"
    ;

std::atomic<u64> g_launches{0};

namespace {
struct Driver {
    decltype(&cuModuleLoadData) ModuleLoadData = nullptr;
    decltype(&cuModuleUnload) ModuleUnload = nullptr;
    decltype(&cuModuleGetFunction) ModuleGetFunction = nullptr;
    decltype(&cuLaunchKernel) LaunchKernel = nullptr;
    decltype(&cuLaunchKernelEx) LaunchKernelEx = nullptr;
    decltype(&cuFuncGetAttribute) FuncGetAttribute = nullptr;
    decltype(&cuFuncSetAttribute) FuncSetAttribute = nullptr;
    decltype(&cuOccupancyMaxActiveBlocksPerMultiprocessor) Occupancy = nullptr;
    decltype(&cuGetErrorString) GetErrorString = nullptr;
    bool ready = false;
};
Driver g_drv;
std::mutex g_mu;
std::map<std::string, std::shared_ptr<JitKernel>> g_cache;
std::map<std::string, std::string> g_cubin_cache;

template <class F> void resolve(F& fn, const char* name) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    cudaError_t e = cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &qr);
    if (e != cudaSuccess || !p) N1_THROW(N1GPU_E_CUDA, "CUDA driver entry point %s unavailable: %s", name, cudaGetErrorString(e));
    fn = (F)p;
}

Driver& driver() {
    if (!g_drv.ready) {
        CK(cudaFree(0));  // make sure the primary context exists and is current
        resolve(g_drv.ModuleLoadData, "cuModuleLoadData");
        resolve(g_drv.ModuleUnload, "cuModuleUnload");
        resolve(g_drv.ModuleGetFunction, "cuModuleGetFunction");
        resolve(g_drv.LaunchKernel, "cuLaunchKernel");
        resolve(g_drv.LaunchKernelEx, "cuLaunchKernelEx");
        resolve(g_drv.FuncGetAttribute, "cuFuncGetAttribute");
        resolve(g_drv.FuncSetAttribute, "cuFuncSetAttribute");
        resolve(g_drv.Occupancy, "cuOccupancyMaxActiveBlocksPerMultiprocessor");
        resolve(g_drv.GetErrorString, "cuGetErrorString");
        g_drv.ready = true;
    }
    return g_drv;
}

// NVRTC is bound at run time from the CUDA toolkit this library was built against, by ABSOLUTE path and
// with RTLD_LOCAL | RTLD_DEEPBIND: a host process (e.g. one that imported torch) may already hold an older
// libnvrtc.so.12 under the same soname, and symbol interposition would silently hand us that compiler.
struct Nvrtc {
    decltype(&nvrtcCreateProgram) CreateProgram = nullptr;
    decltype(&nvrtcCompileProgram) CompileProgram = nullptr;
    decltype(&nvrtcGetProgramLogSize) GetProgramLogSize = nullptr;
    decltype(&nvrtcGetProgramLog) GetProgramLog = nullptr;
    decltype(&nvrtcGetCUBINSize) GetCUBINSize = nullptr;
    decltype(&nvrtcGetCUBIN) GetCUBIN = nullptr;
    decltype(&nvrtcDestroyProgram) DestroyProgram = nullptr;
    decltype(&nvrtcVersion) Version = nullptr;
    int major = 0, minor = 0;
    bool ready = false;
};
Nvrtc g_nvrtc;

Nvrtc& nvrtc() {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_nvrtc.ready) return g_nvrtc;
    std::vector<std::string> tried;
    void* h = nullptr;
    const char* env = getenv("N1GPU_NVRTC");
    std::vector<std::string> cands;
    if (env && *env) cands.push_back(env);
    cands.push_back(std::string(N1_CUDA_LIB) + "/libnvrtc.so");
    cands.push_back("/usr/local/cuda/lib64/libnvrtc.so");
    cands.push_back("libnvrtc.so.12");
    for (auto& c : cands) {
        std::string path = c;
        char real[PATH_MAX];
        if (c.find('/') != std::string::npos && realpath(c.c_str(), real)) path = real;
        // its builtins library is looked up by soname from inside NVRTC: load it first from the same directory
        size_t slash = path.rfind('/');
        if (slash != std::string::npos) {
            std::string b = path.substr(0, slash) + "/libnvrtc-builtins.so";
            char rb[PATH_MAX];
            if (realpath(b.c_str(), rb)) dlopen(rb, RTLD_NOW | RTLD_GLOBAL);
        }
        h = dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL | RTLD_DEEPBIND);
        if (h) break;
        tried.push_back(path + ": " + (dlerror() ? dlerror() : "?"));
    }
    if (!h) {
        std::string all;
        for (auto& t : tried) all += t + "; ";
        N1_THROW(N1GPU_E_CUDA, "cannot load NVRTC (%s)", all.c_str());
    }
    auto sym = [&](const char* n) { void* p = dlsym(h, n); if (!p) N1_THROW(N1GPU_E_CUDA, "NVRTC lacks %s", n); return p; };
    g_nvrtc.CreateProgram = (decltype(g_nvrtc.CreateProgram))sym("nvrtcCreateProgram");
    g_nvrtc.CompileProgram = (decltype(g_nvrtc.CompileProgram))sym("nvrtcCompileProgram");
    g_nvrtc.GetProgramLogSize = (decltype(g_nvrtc.GetProgramLogSize))sym("nvrtcGetProgramLogSize");
    g_nvrtc.GetProgramLog = (decltype(g_nvrtc.GetProgramLog))sym("nvrtcGetProgramLog");
    g_nvrtc.GetCUBINSize = (decltype(g_nvrtc.GetCUBINSize))sym("nvrtcGetCUBINSize");
    g_nvrtc.GetCUBIN = (decltype(g_nvrtc.GetCUBIN))sym("nvrtcGetCUBIN");
    g_nvrtc.DestroyProgram = (decltype(g_nvrtc.DestroyProgram))sym("nvrtcDestroyProgram");
    g_nvrtc.Version = (decltype(g_nvrtc.Version))sym("nvrtcVersion");
    g_nvrtc.Version(&g_nvrtc.major, &g_nvrtc.minor);
    g_nvrtc.ready = true;
    return g_nvrtc;
}

void cu_check(CUresult r, const char* what) {
    if (r == CUDA_SUCCESS) return;
    const char* msg = "?";
    if (g_drv.GetErrorString) g_drv.GetErrorString(r, &msg);
    N1_THROW(N1GPU_E_CUDA, "%s failed: %s", what, msg);
}
}  // namespace

JitKernel::~JitKernel() {
    if (module && g_drv.ModuleUnload) g_drv.ModuleUnload((CUmodule)module);
}

std::atomic<unsigned long long> g_jit_compiled{0}, g_jit_reused{0};
void jit_stats(unsigned long long* compiled, unsigned long long* reused) { *compiled = g_jit_compiled.load(); *reused = g_jit_reused.load(); }

static u64 fnv1a(const char* p, size_t n) {
    u64 h = 1469598103934665603ULL;
    for (size_t i = 0; i < n; ++i) { h ^= (unsigned char)p[i]; h *= 1099511628211ULL; }
    return h;
}

std::string jit_compile_cubin(const std::string& source, std::string* log) {
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_cubin_cache.find(source);
        if (it != g_cubin_cache.end()) { g_jit_reused.fetch_add(1); return it->second; }
    }
    g_jit_compiled.fetch_add(1);
    Nvrtc& rt = nvrtc();
    // Optional on-disk kernel cache (N1GPU_KERNEL_CACHE_DIR): NVRTC + ptxas cost 0.25-0.45 s per new query shape, which a
    // restarted server would otherwise pay again for every prepared statement.  The key covers everything the cubin
    // depends on: generated source, device library and value model, NVRTC version, target.
    std::string cache_file;
    if (const char* dir = getenv("N1GPU_KERNEL_CACHE_DIR")) {
        if (*dir) {
            u64 h = 1469598103934665603ULL;
            auto mix = [&](const char* p, size_t n) { for (size_t i = 0; i < n; ++i) { h ^= (unsigned char)p[i]; h *= 1099511628211ULL; } };
            mix(source.data(), source.size());
            mix(k_device_header, strlen(k_device_header));
            mix(k_value_header, strlen(k_value_header));
            const std::string ver = strf("nvrtc %d.%d sm_100a fmad=false v1", rt.major, rt.minor);
            mix(ver.data(), ver.size());
            cache_file = std::string(dir) + strf("/nq_%016llx_%zu.cubin", (unsigned long long)h, source.size());
            FILE* f = fopen(cache_file.c_str(), "rb");
            if (f) {
                std::string cubin;
                char buf[1 << 16];
                for (size_t n; (n = fread(buf, 1, sizeof buf, f)) > 0;) cubin.append(buf, n);
                fclose(f);
                // an entry = the ELF cubin + 16 trailing bytes ("N1CUBIN1" + FNV-1a of the cubin): a truncated or damaged file
                // (or any other ELF that happens to sit under this name) is ignored and replaced by a fresh compile
                bool good = cubin.size() > 64 + 16 && memcmp(cubin.data(), "\x7f" "ELF", 4) == 0 &&
                            memcmp(cubin.data() + cubin.size() - 16, "N1CUBIN1", 8) == 0;
                if (good) {
                    u64 want;
                    memcpy(&want, cubin.data() + cubin.size() - 8, 8);
                    cubin.resize(cubin.size() - 16);
                    good = want == fnv1a(cubin.data(), cubin.size());
                }
                if (good) {
                    if (log) log->clear();
                    std::lock_guard<std::mutex> lk(g_mu);
                    g_cubin_cache[source] = cubin;
                    return cubin;
                }
            }
        }
    }
    nvrtcProgram prog;
    const char* hdr_names[] = {"n1ql_device.cuh", "n1ql_value.cuh"};
    const char* hdr_srcs[] = {k_device_header, k_value_header};
    if (rt.CreateProgram(&prog, source.c_str(), "nq_scan.cu", 2, hdr_srcs, hdr_names) != NVRTC_SUCCESS)
        N1_THROW(N1GPU_E_CUDA, "nvrtcCreateProgram failed");
    // -fmad=false: float64 arithmetic must round like the reference's separate Go operations.
    // 256-bit global loads need the PTX ISA 8.8 assembler of CUDA >= 12.9; older NVRTC gets 2 x 128-bit.
    bool ld256 = rt.major > 12 || (rt.major == 12 && rt.minor >= 9);
    std::vector<const char*> opts = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo", "--fmad=false", "-default-device", "--device-int128"};
    if (!ld256) opts.push_back("-DNQ_NO_LD256=1");
    nvrtcResult r = rt.CompileProgram(prog, (int)opts.size(), opts.data());
    size_t ls = 0;
    rt.GetProgramLogSize(prog, &ls);
    std::string lg(ls, '\0');
    if (ls) rt.GetProgramLog(prog, &lg[0]);
    if (log) *log = lg;
    if (r != NVRTC_SUCCESS) {
        rt.DestroyProgram(&prog);
        N1_THROW(N1GPU_E_CUDA, "NVRTC %d.%d compilation failed: %s\n--- source ---\n%s", rt.major, rt.minor, lg.c_str(), source.c_str());
    }
    size_t cs = 0;
    rt.GetCUBINSize(prog, &cs);
    std::string cubin(cs, '\0');
    rt.GetCUBIN(prog, &cubin[0]);
    rt.DestroyProgram(&prog);
    if (!cache_file.empty()) {  // best effort: a cache that cannot be written only costs the next compile
        const std::string tmp = cache_file + strf(".%d.tmp", (int)getpid());
        FILE* f = fopen(tmp.c_str(), "wb");
        if (f) {
            char trailer[16];
            memcpy(trailer, "N1CUBIN1", 8);
            const u64 sum = fnv1a(cubin.data(), cubin.size());
            memcpy(trailer + 8, &sum, 8);
            const bool ok = fwrite(cubin.data(), 1, cubin.size(), f) == cubin.size() && fwrite(trailer, 1, 16, f) == 16;
            if (fclose(f) != 0 || !ok || rename(tmp.c_str(), cache_file.c_str()) != 0) remove(tmp.c_str());
        }
    }
    std::lock_guard<std::mutex> lk(g_mu);
    g_cubin_cache[source] = cubin;
    return cubin;
}

std::shared_ptr<JitKernel> jit_load(const std::string& source, int dyn_smem, int block) {
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_cache.find(source);
        if (it != g_cache.end()) { g_jit_reused.fetch_add(1); return it->second; }
    }
    std::string cubin = jit_compile_cubin(source, nullptr);
    Driver& d = driver();
    auto k = std::make_shared<JitKernel>();
    k->cubin = cubin;
    CUmodule mod;
    cu_check(d.ModuleLoadData(&mod, k->cubin.data()), "cuModuleLoadData");
    k->module = mod;
    CUfunction fn;
    cu_check(d.ModuleGetFunction(&fn, mod, "nq_scan"), "cuModuleGetFunction(nq_scan)");
    k->function = fn;
    cu_check(d.FuncGetAttribute(&k->regs, CU_FUNC_ATTRIBUTE_NUM_REGS, fn), "cuFuncGetAttribute");
    cu_check(d.FuncGetAttribute(&k->static_smem, CU_FUNC_ATTRIBUTE_SHARED_SIZE_BYTES, fn), "cuFuncGetAttribute");
    k->dyn_smem = dyn_smem;
    k->block = block;
    if (dyn_smem > 0)  // static + dynamic may cross the 48 KiB default even when the dynamic part alone does not
        cu_check(d.FuncSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, dyn_smem), "cuFuncSetAttribute(max dynamic shared memory)");
    cu_check(d.Occupancy(&k->max_blocks_per_sm, fn, block, (size_t)dyn_smem), "cuOccupancyMaxActiveBlocksPerMultiprocessor");
    if (k->max_blocks_per_sm < 1) k->max_blocks_per_sm = 1;
    std::lock_guard<std::mutex> lk(g_mu);
    g_cache[source] = k;
    return k;
}

void jit_launch(const JitKernel& k, int grid, cudaStream_t stream, void* params, size_t, bool pdl) {
    void* args[] = {params};
    if (pdl && driver().LaunchKernelEx) {
        // Programmatic dependent launch: this grid may start while the previous kernel of the stream drains (that
        // kernel executed griddepcontrol.launch_dependents), so the launch ramp and the tail of back-to-back scans
        // overlap; the scan itself ends with griddepcontrol.wait, which keeps completion in stream order.
        CUlaunchConfig cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDimX = (unsigned)grid; cfg.gridDimY = 1; cfg.gridDimZ = 1;
        cfg.blockDimX = (unsigned)k.block; cfg.blockDimY = 1; cfg.blockDimZ = 1;
        cfg.sharedMemBytes = (unsigned)k.dyn_smem;
        cfg.hStream = (CUstream)stream;
        CUlaunchAttribute attr;
        memset(&attr, 0, sizeof attr);
        attr.id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
        attr.value.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = &attr;
        cfg.numAttrs = 1;
        cu_check(driver().LaunchKernelEx(&cfg, (CUfunction)k.function, args, nullptr), "cuLaunchKernelEx(nq_scan)");
    } else {
        cu_check(driver().LaunchKernel((CUfunction)k.function, (unsigned)grid, 1, 1, (unsigned)k.block, 1, 1, (unsigned)k.dyn_smem, (CUstream)stream, args, nullptr), "cuLaunchKernel(nq_scan)");
    }
    g_launches.fetch_add(1);
}

int device_sm_count() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        CK(cudaGetDevice(&dev));
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    }
    return sms;
}

}  // namespace n1
