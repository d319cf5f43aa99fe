// hostcopy.cuh -- staged host<->device copies for the single-frame calls of the C ABI (host code, api.cu; pipeline.cu
// includes it through api.cuh only for API_BEGIN's per-call reset of the stager).
//
// The reference-facing calls take ordinary (pageable) numpy arrays.  cudaMemcpyAsync on pageable memory goes through the
// driver's own staging buffers on ONE host thread and blocks the caller; at config 3 a frame moves 5.5 MB up and up to
// 8.3 MB down, and those copies were about half of compute_depth's 2.9 ms.  Here large copies go through a page-locked
// arena owned by the context: a few worker threads copy user memory <-> arena in parallel, the DMA engine moves arena <->
// HBM asynchronously (chunk by chunk on the way up, so the DMA of chunk i runs under the memcpy of chunk i+1), and results
// are copied out to the caller's arrays as their DMA events complete while the GPU is still working on the rest of the call.
// L3D_COPY_THREADS=n: threads per large copy (default 2: measured 3.01 -> 2.74 ms for compute_depth at config 3, 4 threads 2.82, 8 threads 3.02; 1 = staged but single-threaded; 0 = the driver's pageable path).
#pragma once
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include <unistd.h>

#include <cuda_runtime.h>

namespace l3d {

class CopyPool {
  public:
    explicit CopyPool(int nthreads) : workers_(nthreads > 1 ? nthreads - 1 : 0), pid_(getpid()), sync_(new Sync) {}
    ~CopyPool() {
        if (getpid() != pid_) {
            // a fork()ed child: the worker threads do not exist here.  Nothing to join, and the mutex / condition variable
            // must not be destroyed either (their copied state still counts the parent's waiters: pthread_cond_destroy
            // would wait for them forever) -- both are left behind.
            new std::vector<std::thread>(std::move(th_));
            return;
        }
        if (!th_.empty()) {
            { std::lock_guard<std::mutex> g(sync_->m); stop_ = true; gen_.fetch_add(1, std::memory_order_release); }
            sync_->cv.notify_all();
            for (auto& t : th_) t.join();
        }
        delete sync_;
    }
    CopyPool(const CopyPool&) = delete;
    CopyPool& operator=(const CopyPool&) = delete;
    // memcpy split over the calling thread and the workers; returns when every part is done
    void copy(void* dst, const void* src, size_t bytes) {
        if (workers_ == 0 || bytes < kParallelMin || getpid() != pid_) { memcpy(dst, src, bytes); return; }
        if (th_.empty()) for (int i = 0; i < workers_; i++) th_.emplace_back(&CopyPool::run, this, i + 1);
        const size_t parts = (size_t)workers_ + 1;
        part_ = ((bytes + parts - 1) / parts + 4095) & ~(size_t)4095;
        dst_ = (char*)dst; src_ = (const char*)src; bytes_ = bytes;
        remaining_.store(workers_, std::memory_order_relaxed);
        gen_.fetch_add(1, std::memory_order_release);
        { std::lock_guard<std::mutex> g(sync_->m); }  // a worker between its predicate check and its wait sees the new gen
        sync_->cv.notify_all();
        do_part(0);
        while (remaining_.load(std::memory_order_acquire) > 0) std::this_thread::yield();
    }

  private:
    static constexpr size_t kParallelMin = 512 << 10;
    void do_part(int i) {
        const size_t a = (size_t)i * part_;
        if (a >= bytes_) return;
        const size_t n = bytes_ - a < part_ ? bytes_ - a : part_;
        memcpy(dst_ + a, src_ + a, n);
    }
    void run(int idx) {
        unsigned long long seen = 0;
        for (;;) {
            // copies come in bursts (two views up, three images down): poll briefly before sleeping
            for (int spin = 0; spin < 300 && gen_.load(std::memory_order_acquire) == seen; spin++) std::this_thread::yield();
            if (gen_.load(std::memory_order_acquire) == seen) {
                std::unique_lock<std::mutex> lk(sync_->m);
                sync_->cv.wait(lk, [&] { return gen_.load(std::memory_order_acquire) != seen; });
            }
            seen = gen_.load(std::memory_order_acquire);
            if (stop_) return;
            do_part(idx);
            remaining_.fetch_sub(1, std::memory_order_release);
        }
    }
    const int workers_;
    const pid_t pid_;   // the process that owns the worker threads (they do not survive a fork)
    struct Sync { std::mutex m; std::condition_variable cv; };
    Sync* const sync_;   // on the heap: a forked child leaves it alone (see the destructor)
    std::vector<std::thread> th_;
    std::atomic<unsigned long long> gen_{0};
    std::atomic<int> remaining_{0};
    bool stop_ = false;
    char* dst_ = nullptr;
    const char* src_ = nullptr;
    size_t bytes_ = 0, part_ = 0;
};

class HostStager {
  public:
    HostStager() : threads_(env_threads()), pool_(threads_) {}
    ~HostStager() {
        for (auto& b : blocks_) cudaFreeHost(b.p);
        for (auto e : events_) cudaEventDestroy(e);
    }
    bool enabled() const { return threads_ > 0; }
    bool wants(size_t bytes) const { return threads_ > 0 && bytes >= kStageMin && bytes <= kStageMax; }

    // new API call: whatever an earlier (failed) call left behind is dropped
    void begin() { pending_.clear(); ev_used_ = 0; reset_arena(); }

    cudaError_t h2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
        char* p = alloc(bytes);
        if (!p) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s);
        for (size_t off = 0; off < bytes; off += kChunk) {
            const size_t n = bytes - off < kChunk ? bytes - off : kChunk;
            pool_.copy(p + off, (const char*)src + off, n);
            cudaError_t e = cudaMemcpyAsync((char*)dst + off, p + off, n, cudaMemcpyHostToDevice, s);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    }
    // the DMA into the arena is enqueued now; the copy into the caller's memory happens in finish()
    cudaError_t d2h(void* dst, const void* src, size_t bytes, cudaStream_t s) {
        char* p = alloc(bytes);
        if (!p) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s);
        cudaError_t e = cudaMemcpyAsync(p, src, bytes, cudaMemcpyDeviceToHost, s);
        if (e != cudaSuccess) return e;
        if (ev_used_ == events_.size()) {
            cudaEvent_t ev;
            e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
            if (e != cudaSuccess) return e;
            events_.push_back(ev);
        }
        cudaEvent_t ev = events_[ev_used_++];
        e = cudaEventRecord(ev, s);
        if (e != cudaSuccess) return e;
        pending_.push_back({dst, p, bytes, ev});
        return cudaSuccess;
    }
    // copies every staged result out as its DMA completes, then waits for the stream
    cudaError_t finish(cudaStream_t s) {
        cudaError_t first = cudaSuccess;
        for (auto& q : pending_) {
            cudaError_t e = cudaEventSynchronize(q.ev);
            if (e != cudaSuccess) { first = e; break; }
            pool_.copy(q.dst, q.pinned, q.bytes);
        }
        pending_.clear();
        ev_used_ = 0;
        cudaError_t e = cudaStreamSynchronize(s);
        reset_arena();
        return first != cudaSuccess ? first : e;
    }

  private:
    static constexpr size_t kStageMin = 256 << 10;   // below: the driver's path is as fast
    static constexpr size_t kStageMax = 64 << 20;    // above (debug volumes): not worth pinning host memory for
    static constexpr size_t kArenaMax = 256 << 20;
    static constexpr size_t kChunk = 1 << 20;
    struct Block { char* p; size_t cap, used; };
    struct Pending { void* dst; const char* pinned; size_t bytes; cudaEvent_t ev; };

    static int env_threads() {
        const char* e = getenv("L3D_COPY_THREADS");
        int n = e ? atoi(e) : 2;
        const int hw = (int)std::thread::hardware_concurrency();
        if (hw > 0 && n > hw) n = hw;
        return n < 0 ? 0 : (n > 16 ? 16 : n);
    }
    char* alloc(size_t bytes) {
        const size_t need = (bytes + 4095) & ~(size_t)4095;
        for (auto& b : blocks_)
            if (b.cap - b.used >= need) { char* p = b.p + b.used; b.used += need; return p; }
        size_t total = 0;
        for (auto& b : blocks_) total += b.cap;
        const size_t cap = need > ((size_t)8 << 20) ? need : ((size_t)8 << 20);
        if (total + cap > kArenaMax) return nullptr;
        void* p = nullptr;
        if (cudaHostAlloc(&p, cap, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        blocks_.push_back({(char*)p, cap, need});
        return (char*)p;
    }
    // nothing is in flight here.  Several blocks = the arena grew during the call: one block of the total size next time
    void reset_arena() {
        if (blocks_.size() > 1) {
            size_t total = 0;
            for (auto& b : blocks_) { total += b.cap; cudaFreeHost(b.p); }
            blocks_.clear();
            void* p = nullptr;
            if (cudaHostAlloc(&p, total, cudaHostAllocDefault) == cudaSuccess) blocks_.push_back({(char*)p, total, 0});
            else cudaGetLastError();
        }
        for (auto& b : blocks_) b.used = 0;
    }
    const int threads_;
    CopyPool pool_;
    std::vector<Block> blocks_;
    std::vector<Pending> pending_;
    std::vector<cudaEvent_t> events_;
    size_t ev_used_ = 0;
};

}  // namespace l3d
