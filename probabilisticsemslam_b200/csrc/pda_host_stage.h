// pda_host_stage.h -- the staging of the *_host entry points: per-device state behind a per-device lock (DeviceScope),
// and HostIO, which lays out a call's arrays in the device arena and moves them between the caller's memory and the
// device on the device's one stream.
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
// cudaMalloc/cudaFree every time), one pinned bounce buffer, the non-blocking stream every copy and launch of a *_host
// call goes to (created on first use), and the mutex that serialises the *_host calls of ONE device.  Calls that name
// different devices run concurrently -- that is what the multi-device entry points (pda_*_host_multi) do, one host
// thread per device.
constexpr int PDA_MAX_DEVICES = 64;
struct DeviceCtx {
    std::mutex mu;
    unsigned char* arena = nullptr; size_t arenaCap = 0;
    unsigned char* pinned = nullptr; size_t pinnedCap = 0;
    cudaStream_t run = nullptr;
};
extern DeviceCtx g_dev[PDA_MAX_DEVICES];

// Whether `p` lies in a buffer from pda_host_alloc (page-locked, portable and mapped: every device may use it in place).
bool in_portable_range(const void* p);

// If `p` is page-locked host memory that `device` can address (cudaHostAlloc / cudaHostRegister under unified
// addressing), returns the device-side alias, else NULL.
inline void* mapped_alias(const void* p, int device) {
    if (!p) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    // page-locked by a context of THIS device, or handed out by pda_host_alloc (portable).  Memory pinned for another
    // device's context by somebody else is only guaranteed to be addressable there: copy it instead.
    if (at.type != cudaMemoryTypeHost) return nullptr;
    return (at.device == device || in_portable_range(p)) ? at.devicePointer : nullptr;
}

// Validates the device, takes its lock and makes it current; the destructor drains the device's stream if the call is
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
            if (g_dev[dev_].run) cudaStreamSynchronize(g_dev[dev_].run);
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

#define PDA_TRY(expr) do { int _rc = (expr); if (_rc != PDA_OK) return _rc; } while (0)

// Multi-device form of a *_host call over independent units: cuts [0, n) into one contiguous slice per device and runs
// f(first, last, device) for each slice on its own host thread (each thread takes that device's lock, arena and
// stream).  The first failure is reported with the device it happened on.
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

// The arena layout and the host <-> device copies of a single-device *_host call, all on the device's `run` stream.
// The call declares its arrays -- in(), inout(), out(), each returning a handle (a NULL pointer or 0 bytes reserves
// room without copying) -- and its device-only scratch(), then runs commit() -> upload() -> launches on stream() that
// read device pointers through at<T>(handle) -> download(), which synchronises.
// Calls of at most PDA_PACKED_LIMIT bytes of declared arrays (a batch of one from the C++ shims, a handful of window
// frames) would be dominated by the fixed cost of each cudaMemcpy from pageable memory (~10 us apiece, a dozen per
// call): their arrays lie contiguously in the arena (in | inout | out), mirrored in ONE pinned host buffer, and each
// direction is a single copy.  Larger calls copy each array straight from and to the caller's memory, so the pinned
// buffer never grows beyond the limit's size.  In such a call an array declared IN_PLACE -- one the kernel touches
// once, such as a matrix a warp reads when it takes the problem or a table it writes when it is done -- that lies in
// page-locked memory this device can address (mapped_alias) is not staged at all: the kernel reads or writes the
// caller's memory, and the transfer hides under the computing instead of standing in front of or behind it.  Whether a
// call is packed counts IN_PLACE arrays too, and a packed call never uses caller memory in place: a kernel that reads
// such an array more than once would do that over PCIe.
constexpr size_t PDA_PACKED_LIMIT = 8u << 20;

class HostIO {
public:
    enum Use { COPY, IN_PLACE };
    explicit HostIO(int device) : device_(device) {}
    size_t in(const void* src, size_t bytes, Use use = COPY) { return add(const_cast<void*>(src), bytes, IN, use); }
    size_t inout(void* p, size_t bytes) { return add(p, bytes, INOUT, COPY); }
    size_t out(void* dst, size_t bytes, Use use = COPY) { return add(dst, bytes, OUT, use); }
    size_t scratch(size_t bytes) { return add(nullptr, bytes, SCRATCH, COPY); }
    int commit() {
        size_t declared = 0;
        for (const Item& it : items_)
            if (it.dir != SCRATCH) declared += WorkspaceLayout::round(it.bytes);
        packed_ = declared <= PDA_PACKED_LIMIT;
        // in | inout | out | scratch, each in declaration order; an array used in place takes no room
        size_t used = 0;
        size_t* const ends[] = {&inEnd_, &ioEnd_, &end_, &used};
        for (int d = IN; d <= SCRATCH; ++d) {
            for (Item& it : items_) {
                if (it.dir != d) continue;
                void* const alias = !packed_ && it.use == IN_PLACE ? mapped_alias(it.host, device_) : nullptr;
                if (alias) { it.dev = static_cast<unsigned char*>(alias); it.host = nullptr; continue; }  // nothing to copy
                it.off = used;
                used += WorkspaceLayout::round(it.bytes);
            }
            *ends[d] = used;
        }
        DeviceCtx& c = g_dev[device_];
        if (c.arenaCap < used) {
            if (c.arena) { cudaDeviceSynchronize(); cudaFree(c.arena); }
            c.arena = nullptr; c.arenaCap = 0;
            size_t want = used + used / 4;
            cudaError_t e = cudaMalloc(&c.arena, want);
            if (e != cudaSuccess) { (void)cudaGetLastError(); want = used; e = cudaMalloc(&c.arena, want); }
            if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(host staging arena)");
            c.arenaCap = want;
        }
        for (Item& it : items_)
            if (!it.dev) it.dev = c.arena + it.off;
        if (!c.run) PDA_CUDA_TRY(cudaStreamCreateWithFlags(&c.run, cudaStreamNonBlocking));
        s_ = c.run;
        return PDA_OK;
    }
    template <class T> T* at(size_t h) const { return reinterpret_cast<T*>(items_[h].dev); }
    cudaStream_t stream() const { return s_; }
    int upload() {
        if (!packed_) {
            for (const Item& it : items_)
                if (it.copied() && it.dir != OUT) PDA_CUDA_TRY(cudaMemcpyAsync(it.dev, it.host, it.bytes, cudaMemcpyHostToDevice, s_));
            return PDA_OK;
        }
        DeviceCtx& c = g_dev[device_];
        if (c.pinnedCap < end_) {
            if (c.pinned) { cudaDeviceSynchronize(); cudaFreeHost(c.pinned); }  // an earlier transfer may still be reading it
            c.pinned = nullptr; c.pinnedCap = 0;
            const size_t want = end_ + end_ / 2 + 4096;
            PDA_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&c.pinned), want, cudaHostAllocDefault));
            c.pinnedCap = want;
        }
        pin_ = c.pinned;
        for (const Item& it : items_)
            if (it.copied() && it.dir != OUT) memcpy(pin_ + it.off, it.host, it.bytes);
        if (ioEnd_ > 0) PDA_CUDA_TRY(cudaMemcpyAsync(c.arena, pin_, ioEnd_, cudaMemcpyHostToDevice, s_));
        return PDA_OK;
    }
    int download() {
        if (!packed_) {
            for (const Item& it : items_)
                if (it.copied() && it.dir != IN) PDA_CUDA_TRY(cudaMemcpyAsync(it.host, it.dev, it.bytes, cudaMemcpyDeviceToHost, s_));
            PDA_CUDA_TRY(cudaStreamSynchronize(s_));
            return PDA_OK;
        }
        if (end_ > inEnd_)
            PDA_CUDA_TRY(cudaMemcpyAsync(pin_ + inEnd_, g_dev[device_].arena + inEnd_, end_ - inEnd_, cudaMemcpyDeviceToHost, s_));
        PDA_CUDA_TRY(cudaStreamSynchronize(s_));
        for (const Item& it : items_)
            if (it.copied() && it.dir != IN) memcpy(it.host, pin_ + it.off, it.bytes);
        return PDA_OK;
    }
private:
    enum Dir { IN, INOUT, OUT, SCRATCH };
    struct Item {
        void* host; size_t bytes; Dir dir; Use use;
        size_t off; unsigned char* dev;
        bool copied() const { return host && bytes; }
    };
    size_t add(void* host, size_t bytes, Dir dir, Use use) {
        items_.push_back({host, bytes, dir, use, 0, nullptr});
        return items_.size() - 1;
    }
    int device_;
    bool packed_ = false;
    cudaStream_t s_ = nullptr;
    unsigned char* pin_ = nullptr;
    size_t inEnd_ = 0, ioEnd_ = 0, end_ = 0;
    std::vector<Item> items_;
};

}  // namespace pda
#endif
