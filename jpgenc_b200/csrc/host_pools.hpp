// Host-side worker threads of the C-ABI layer: HostPool (parallel_for shared by the pipeline lanes of a batched call) and
// TablePool (the four Huffman tables of one image side by side).
#pragma once

#include <atomic>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace jpgenc {

// The four Huffman tables of an image are independent and the build is sequential host work (tens of microseconds
// for a dozen symbols, half a millisecond for a full AC alphabet) during which the GPU has nothing to do.  A worker
// thread (up to three) and the calling thread build them side by side.  Waking a sleeping thread costs about as much as a
// small table, so the workers are ARMED (woken, then spinning) when the statistics kernel is launched and find the
// histogram as soon as it arrives; they go back to sleep after every image.
// parallel_for over n jobs on persistent host threads (the 4 * F table builds of a batch of F frames).  One pool serves
// all pipeline lanes of a context: several parallel_for calls may be in flight at once, every idle worker helps whichever
// call still has jobs to hand out, and the caller works on its own call too -- a lane whose tables are due gets all the
// cores that the other lanes are not using right now.
class HostPool {
public:
    explicit HostPool(unsigned workers) {
        for (unsigned i = 0; i < workers; ++i) threads_.emplace_back([this] { run(); });
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            quit_ = true;
        }
        cv_.notify_all();
        for (std::thread& t : threads_) t.join();
    }
    template <class F>
    void parallel_for(uint32_t n, F&& fn) {
        if (n == 0) return;
        auto call = std::make_shared<Call>();
        call->fn = fn;
        call->n = n;
        {
            std::lock_guard<std::mutex> lk(m_);
            calls_.push_back(call);
        }
        cv_.notify_all();
        drain(*call);
        if (call->done.load(std::memory_order_acquire) < n) {   // the last few jobs are still running on other threads
            std::unique_lock<std::mutex> lk(m_);
            done_cv_.wait(lk, [&] { return call->done.load(std::memory_order_acquire) >= n; });
        }
    }

private:
    struct Call {
        std::function<void(uint32_t)> fn;
        uint32_t n = 0;
        std::atomic<uint32_t> next{0}, done{0};
    };
    void drain(Call& c) {
        for (;;) {
            const uint32_t i = c.next.fetch_add(1, std::memory_order_relaxed);
            if (i >= c.n) return;
            c.fn(i);
            if (c.done.fetch_add(1, std::memory_order_acq_rel) + 1 == c.n) {     // the call is complete: wake its owner
                std::lock_guard<std::mutex> lk(m_);
                done_cv_.notify_all();
            }
        }
    }
    void run() {
        for (;;) {
            std::shared_ptr<Call> call;
            {
                std::unique_lock<std::mutex> lk(m_);
                for (;;) {
                    while (!calls_.empty() && calls_.front()->next.load(std::memory_order_relaxed) >= calls_.front()->n) calls_.pop_front();
                    if (quit_ || !calls_.empty()) break;
                    cv_.wait(lk);
                }
                if (quit_) return;
                call = calls_.front();
            }
            drain(*call);
        }
    }
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cv_, done_cv_;
    bool quit_ = false;
    std::deque<std::shared_ptr<Call>> calls_;
};

class TablePool {
public:
    // `workers` 1..3 threads beside the caller.  The caller always builds the luma AC table (normally the largest alphabet:
    // 10 us against 3 us for each of the others on a photograph); with three workers each of the other tables has a thread
    // of its own, with one worker that thread builds all three one after the other -- about as long as the luma AC table
    // takes, with one spinning thread instead of three (what capi.cu uses: kTableWorkers).
    explicit TablePool(int workers = 1) : nworkers_(workers < 1 ? 1 : workers > 3 ? 3 : workers) {
        for (int i = 0; i < nworkers_; ++i) workers_[i] = std::thread([this, i] { run(i); });
    }
    ~TablePool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            quit_ = true;
        }
        cv_.notify_all();
        for (int i = 0; i < nworkers_; ++i) workers_[i].join();
    }
    void arm() {
        {
            std::lock_guard<std::mutex> lk(m_);
            ++armed_;
        }
        cv_.notify_all();
    }
    // after arm(): builds tables[t] from count[t] / first[t] for t = 0..3 (with null pointers: just releases the workers)
    int build(const uint32_t (*count)[256], const uint64_t (*first)[256], jpgenc_huff_table* tables) {
        count_ = count; first_ = first; tables_ = tables;
        for (int& r : rc_) r = JPGENC_OK;
        done_.store(0, std::memory_order_relaxed);
        published_.store(armed_, std::memory_order_release);
        static const int kMine = 1;                                   // Y_AC: normally the largest alphabet
        if (count) rc_[kMine] = jpgenc_build_huffman(count[kMine], first[kMine], &tables[kMine]);
        while (done_.load(std::memory_order_acquire) != nworkers_) cpu_relax();
        for (int r : rc_) if (r) return r;
        return JPGENC_OK;
    }

private:
    static void cpu_relax() {
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    void run(int idx) {
        static const int kTable[3] = {0, 2, 3};                       // Y_DC, C_DC, C_AC
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return quit_ || armed_ != seen; });
                if (quit_) return;
                seen = armed_;
            }
            while (published_.load(std::memory_order_acquire) != seen) cpu_relax();
            if (count_)
                for (int k = idx; k < 3; k += nworkers_) {            // worker idx of n takes tables idx, idx + n, ...
                    const int t = kTable[k];
                    rc_[t] = jpgenc_build_huffman(count_[t], first_[t], &tables_[t]);
                }
            done_.fetch_add(1, std::memory_order_release);
        }
    }
    const int nworkers_;
    std::thread workers_[3];
    std::mutex m_;
    std::condition_variable cv_;
    bool quit_ = false;
    uint64_t armed_ = 0;
    std::atomic<uint64_t> published_{0};
    std::atomic<int> done_{0};
    const uint32_t (*count_)[256] = nullptr;
    const uint64_t (*first_)[256] = nullptr;
    jpgenc_huff_table* tables_ = nullptr;
    int rc_[4] = {0, 0, 0, 0};
};
}
