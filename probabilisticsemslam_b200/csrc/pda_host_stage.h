// pda_host_stage.h -- helpers for the *_host entry points: per-device staging state behind a per-device lock
// (DeviceScope), and checked async copies.
#ifndef PDA_HOST_STAGE_H
#define PDA_HOST_STAGE_H

#include "pda_internal.h"

#include <algorithm>
#include <atomic>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace pda {

// Per-device state of the *_host entry points: a grow-only device arena (a batch-of-one shim call does not pay
// cudaMalloc/cudaFree every time), three non-blocking streams (copy in / run / copy out), one pinned bounce buffer, and
// the mutex that serialises the *_host calls of ONE device.  Calls that name different devices run concurrently --
// that is what the multi-device entry points (pda_*_host_multi) do, one host thread per device.
constexpr int PDA_MAX_DEVICES = 64;
struct DeviceCtx {
    std::mutex mu;
    unsigned char* arena = nullptr; size_t arenaCap = 0;
    bool haveStreams = false; cudaStream_t in = nullptr, run = nullptr, out = nullptr;
    unsigned char* pinned = nullptr; size_t pinnedCap = 0;
};
extern DeviceCtx g_dev[PDA_MAX_DEVICES];

// Validates the device, takes its lock and makes it current; the destructor drains the device's streams if the call is
// leaving with work still queued (an error return), restores the caller's current device and releases the lock.
class DeviceScope {
public:
    DeviceScope() : dev_(-1), prev_(-1), fails_(0) {}
    int enter(int device) {
        static std::atomic<int> known(0);  // the device count does not change while the process lives
        int n = known.load(std::memory_order_relaxed);
        if (n == 0) {
            cudaError_t e = cudaGetDeviceCount(&n);
            if (e != cudaSuccess || n == 0) {
                (void)cudaGetLastError();
                return fail(PDA_ERR_CUDA, "no CUDA device available (libpda_b200 has no CPU fallback)");
            }
            known.store(n, std::memory_order_relaxed);
        }
        if (device < 0 || device >= n || device >= PDA_MAX_DEVICES) return fail(PDA_ERR_INVALID, "device %d out of range (have %d)", device, n);
        if (cudaGetDevice(&prev_) != cudaSuccess) { (void)cudaGetLastError(); prev_ = -1; }
        g_dev[device].mu.lock();
        dev_ = device;
        fails_ = failure_count();
        PDA_CUDA_TRY(cudaSetDevice(device));
        return PDA_OK;
    }
    ~DeviceScope() {
        if (dev_ < 0) return;
        if (failure_count() != fails_) {  // leaving on an error: nothing may still be running against the arena or the caller's buffers
            DeviceCtx& c = g_dev[dev_];
            if (c.haveStreams) { cudaStreamSynchronize(c.in); cudaStreamSynchronize(c.run); cudaStreamSynchronize(c.out); }
            cudaStreamSynchronize(0);
            (void)cudaGetLastError();
        }
        if (prev_ >= 0 && prev_ != dev_) cudaSetDevice(prev_);
        g_dev[dev_].mu.unlock();
    }
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
private:
    int dev_, prev_;
    unsigned long long fails_;
};

class Stage {
public:
    explicit Stage(int device) : device_(device), used_(0), base_(nullptr) {}
    // first pass: reserve() everything; then commit(); then at<T>(offset)
    size_t reserve(size_t bytes) { size_t o = used_; used_ += (bytes + 255) / 256 * 256; return o; }
    int commit() {
        DeviceCtx& a = g_dev[device_];
        if (a.arenaCap < used_) {
            if (a.arena) { cudaDeviceSynchronize(); cudaFree(a.arena); }
            a.arena = nullptr; a.arenaCap = 0;
            size_t want = used_ + used_ / 4;
            cudaError_t e = cudaMalloc(&a.arena, want);
            if (e != cudaSuccess) { (void)cudaGetLastError(); want = used_; e = cudaMalloc(&a.arena, want); }
            if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(host staging arena)");
            a.arenaCap = want;
        }
        base_ = a.arena;
        return PDA_OK;
    }
    template <class T> T* at(size_t off) const { return reinterpret_cast<T*>(base_ + off); }
    size_t used() const { return used_; }
    int device() const { return device_; }
private:
    int device_; size_t used_; unsigned char* base_;
};

struct HostStreams { cudaStream_t in, run, out; };
inline int host_streams(int device, HostStreams** out) {
    static thread_local HostStreams hs;
    DeviceCtx& c = g_dev[device];
    if (!c.haveStreams) {
        PDA_CUDA_TRY(cudaStreamCreateWithFlags(&c.in, cudaStreamNonBlocking));
        PDA_CUDA_TRY(cudaStreamCreateWithFlags(&c.run, cudaStreamNonBlocking));
        PDA_CUDA_TRY(cudaStreamCreateWithFlags(&c.out, cudaStreamNonBlocking));
        c.haveStreams = true;
    }
    hs.in = c.in; hs.run = c.run; hs.out = c.out;
    *out = &hs;
    return PDA_OK;
}

template <class T> inline int h2d(T* dst, const T* src, size_t n, cudaStream_t s) {
    if (n == 0) return PDA_OK;
    PDA_CUDA_TRY(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyHostToDevice, s));
    return PDA_OK;
}
template <class T> inline int d2h(T* dst, const T* src, size_t n, cudaStream_t s) {
    if (n == 0 || dst == nullptr) return PDA_OK;
    PDA_CUDA_TRY(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, s));
    return PDA_OK;
}
#define PDA_TRY(expr) do { int _rc = (expr); if (_rc != PDA_OK) return _rc; } while (0)

// Multi-device form of a *_host call over independent units: cuts [0, n) into one contiguous slice per device and runs
// f(first, last, device) for each slice on its own host thread (each thread takes that device's lock, arena and
// streams).  The first failure is reported with the device it happened on.
template <class F>
inline int run_sharded(int64_t n, const int32_t* devices, int32_t nDevices, F&& f) {
    const int shards = (int)std::min<int64_t>(nDevices, n);
    if (shards <= 1) return f((int64_t)0, n, (int)devices[0]);
    std::vector<int> rc((size_t)shards, PDA_OK);
    std::vector<std::string> msg((size_t)shards);
    std::vector<std::thread> th;
    th.reserve((size_t)shards);
    for (int s = 0; s < shards; ++s) {
        const int64_t p0 = n * s / shards, p1 = n * (s + 1) / shards;
        th.emplace_back([&, s, p0, p1]() {
            rc[(size_t)s] = f(p0, p1, (int)devices[s]);
            if (rc[(size_t)s] != PDA_OK) msg[(size_t)s] = pda_last_error();
        });
    }
    for (std::thread& t : th) t.join();
    for (int s = 0; s < shards; ++s)
        if (rc[(size_t)s] != PDA_OK) return fail(rc[(size_t)s], "device %d: %s", (int)devices[s], msg[(size_t)s].c_str());
    return PDA_OK;
}

// The host <-> device copies of a single-device *_host call, all on the device's `run` stream.  The call declares its
// arrays once -- in()s, then inout()s, then out()s, each returning its offset in the arena (a NULL pointer or 0 bytes
// reserves without copying) -- then reserves its scratch on the Stage and runs commit() -> upload() -> launches on
// stream() -> download(), which synchronises.
// Calls of at most PDA_PACKED_LIMIT bytes of declared arrays (a batch of one from the C++ shims, a handful of window
// frames) would be dominated by the fixed cost of each cudaMemcpy from pageable memory (~10 us apiece, a dozen per
// call): their arrays lie contiguously in the arena (in | inout | out), mirrored in ONE pinned host buffer, and each
// direction is a single copy.  Larger calls copy each array straight from and to the caller's memory, so the pinned
// buffer never grows beyond the limit's size.
constexpr size_t PDA_PACKED_LIMIT = 8u << 20;

class HostIO {
public:
    explicit HostIO(Stage& st) : st_(st), begin_(st.used()), inEnd_(begin_), ioEnd_(begin_), end_(begin_) {}
    size_t in(const void* src, size_t bytes) { const size_t o = add(const_cast<void*>(src), bytes, IN); inEnd_ = ioEnd_ = end_; return o; }
    size_t inout(void* p, size_t bytes) { const size_t o = add(p, bytes, INOUT); ioEnd_ = end_; return o; }
    size_t out(void* dst, size_t bytes) { return add(dst, bytes, OUT); }
    bool packed() const { return end_ - begin_ <= PDA_PACKED_LIMIT; }
    int commit() {
        PDA_TRY(st_.commit());
        HostStreams* hs = nullptr;
        PDA_TRY(host_streams(st_.device(), &hs));
        s_ = hs->run;
        return PDA_OK;
    }
    cudaStream_t stream() const { return s_; }
    int upload() {
        if (!packed()) {
            for (const Item& it : items_)
                if (it.dir != OUT)
                    PDA_CUDA_TRY(cudaMemcpyAsync(st_.at<unsigned char>(it.off), it.host, it.bytes, cudaMemcpyHostToDevice, s_));
            return PDA_OK;
        }
        const size_t need = end_ - begin_;
        DeviceCtx& c = g_dev[st_.device()];
        if (c.pinnedCap < need) {
            if (c.pinned) { cudaDeviceSynchronize(); cudaFreeHost(c.pinned); }  // an earlier transfer may still be reading it
            c.pinned = nullptr; c.pinnedCap = 0;
            const size_t want = need + need / 2 + 4096;
            PDA_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&c.pinned), want, cudaHostAllocDefault));
            c.pinnedCap = want;
        }
        pin_ = c.pinned;
        for (const Item& it : items_)
            if (it.dir != OUT) memcpy(pin_ + (it.off - begin_), it.host, it.bytes);
        if (ioEnd_ > begin_)
            PDA_CUDA_TRY(cudaMemcpyAsync(st_.at<unsigned char>(begin_), pin_, ioEnd_ - begin_, cudaMemcpyHostToDevice, s_));
        return PDA_OK;
    }
    int download() {
        if (!packed()) {
            for (const Item& it : items_)
                if (it.dir != IN)
                    PDA_CUDA_TRY(cudaMemcpyAsync(it.host, st_.at<unsigned char>(it.off), it.bytes, cudaMemcpyDeviceToHost, s_));
            PDA_CUDA_TRY(cudaStreamSynchronize(s_));
            return PDA_OK;
        }
        if (end_ > inEnd_)
            PDA_CUDA_TRY(cudaMemcpyAsync(pin_ + (inEnd_ - begin_), st_.at<unsigned char>(inEnd_), end_ - inEnd_,
                                         cudaMemcpyDeviceToHost, s_));
        PDA_CUDA_TRY(cudaStreamSynchronize(s_));
        for (const Item& it : items_)
            if (it.dir != IN) memcpy(it.host, pin_ + (it.off - begin_), it.bytes);
        return PDA_OK;
    }
private:
    enum Dir { IN, INOUT, OUT };
    struct Item { size_t off; void* host; size_t bytes; Dir dir; };
    size_t add(void* host, size_t bytes, Dir dir) {
        const size_t o = st_.reserve(bytes);
        if (host && bytes) items_.push_back({o, host, bytes, dir});
        end_ = st_.used();
        return o;
    }
    Stage& st_;
    cudaStream_t s_ = nullptr;
    unsigned char* pin_ = nullptr;
    size_t begin_, inEnd_, ioEnd_, end_;
    std::vector<Item> items_;
};

}  // namespace pda
#endif
