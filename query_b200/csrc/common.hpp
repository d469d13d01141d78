// common.hpp — shared host-side definitions for libn1gpu.so
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <exception>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/n1gpu.h"
#include "final_group.hpp"

namespace n1 {

inline u32 bit(int c) { return 1u << c; }
const u32 M_NUM = (1u << C_INT) | (1u << C_FLOAT);
const u32 M_BOOL = (1u << C_FALSE) | (1u << C_TRUE);
const u32 M_ALL_SCALAR = 0x7f;

// An error carrying one of the N1GPU_E_* codes; the ABI layer turns it into a status + message.
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

inline std::string strf(const char* fmt, ...) {
    char buf[2048];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    return buf;
}

#define N1_THROW(code, ...) throw ::n1::Error((code), ::n1::strf(__VA_ARGS__))
#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            N1_THROW(N1GPU_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

extern std::atomic<u64> g_launches;  // every kernel launch made by this library

// A host value (result side): class + payload; strings own their bytes.
struct HValue {
    u8 cls = C_MISSING;
    i64 bits = 0;
    std::string s;
    HValue() = default;
    HValue(Val v) : cls((u8)v.c), bits(v.b) {}  // a value of n1ql_value.cuh (no string bytes)
    static HValue missing() { return HValue(); }
    static HValue null() { HValue v; v.cls = C_NULL; return v; }
    static HValue boolean(bool b) { HValue v; v.cls = b ? C_TRUE : C_FALSE; return v; }
    static HValue integer(i64 x) { HValue v; v.cls = C_INT; v.bits = x; return v; }
    static HValue flt(double d) { HValue v; v.cls = C_FLOAT; memcpy(&v.bits, &d, 8); return v; }
    static HValue str(const std::string& s) { HValue v; v.cls = C_STRING; v.s = s; return v; }
    double f() const { double d; memcpy(&d, &bits, 8); return d; }
    double num() const { return cls == C_INT ? (double)bits : f(); }
};

// caching allocators (mem.cpp)
void* dev_alloc(size_t n, size_t* actual);
void dev_free(void* p, size_t n);
void dev_pool_trim();
void* pin_alloc(size_t n, size_t* actual);
void pin_free(void* p, size_t n);

// Device buffer (pooled cudaMalloc) with RAII.
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf() {}
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { release(); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; return *this; }
    ~DevBuf() { release(); }
    void alloc(size_t n) {
        release();
        p = dev_alloc(n, &bytes);  // bytes = the (rounded-up) size actually held
    }
    void ensure(size_t n) { if (n > bytes) alloc(n); }
    void release() { if (p) dev_free(p, bytes); p = nullptr; bytes = 0; }
    template <class T> T* as() const { return (T*)p; }
};

struct PinnedBuf {
    void* p = nullptr;
    size_t bytes = 0;
    PinnedBuf() {}
    PinnedBuf(const PinnedBuf&) = delete;
    PinnedBuf& operator=(const PinnedBuf&) = delete;
    ~PinnedBuf() { if (p) pin_free(p, bytes); }
    void ensure(size_t n) {
        if (n <= bytes) return;
        if (p) pin_free(p, bytes);
        p = nullptr;
        p = pin_alloc(n, &bytes);
    }
    template <class T> T* as() const { return (T*)p; }
};

inline int bits_for(u64 n_values) {  // bits to represent values 0..n_values-1
    int b = 0;
    while (b < 64 && ((u64)1 << b) < n_values) ++b;
    return b;
}

// fn(0) .. fn(n - 1), each on its own thread (fn(0) on the caller's); returns when all have, rethrowing the first
// exception one of them threw
template <class F> void parallel_for(int n, F&& fn) {
    std::vector<std::exception_ptr> errs((size_t)(n > 0 ? n : 0));
    auto run = [&](int t) { try { fn(t); } catch (...) { errs[(size_t)t] = std::current_exception(); } };
    std::vector<std::thread> pool;
    try { for (int t = 1; t < n; ++t) pool.emplace_back(run, t); } catch (...) { for (auto& th : pool) th.join(); throw; }
    if (n > 0) run(0);
    for (auto& th : pool) th.join();
    for (auto& e : errs) if (e) std::rethrow_exception(e);
}

double now_sec();
bool have_device();  // a CUDA device is visible to this process

}  // namespace n1
