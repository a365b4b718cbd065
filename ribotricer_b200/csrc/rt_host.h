// rt_host.h -- the host-side mechanisms the native commands share: uninitialised column storage, thread counts and
// fork-join loops, the parallel whole-file read, line-aligned chunking, integer formatting and the write-behind writer.
// Internal to the library: not installed, and everything here has internal linkage, so nothing of it is exported.
#pragma once

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "ribotricer_b200.h"

void rt_io_set_error(const std::string& msg);   // rt_host_io.cpp: the slot rt_io_last_error reads

// The buffer behind an rt_text handle: malloc storage of n bytes and a NUL at p[n] (rt_text_alloc, rt_bgzf_inflate).
struct rt_text {
    char* p = nullptr;
    size_t n = 0;
};

namespace {

// Plain uninitialised malloc storage: the threads that fill a large array are the first to touch its pages (a
// std::vector would have one thread zero-fill it).
template <class T>
struct HostArr {
    T* p = nullptr;
    size_t n = 0;
    HostArr() = default;
    HostArr(const HostArr&) = delete;
    HostArr& operator=(const HostArr&) = delete;
    ~HostArr() { free(p); }
    bool alloc(size_t m) {
        free(p);
        p = static_cast<T*>(malloc(std::max<size_t>(m, 1) * sizeof(T)));
        n = p ? m : 0;
        return p != nullptr;
    }
    T& operator[](size_t i) { return p[i]; }
    const T& operator[](size_t i) const { return p[i]; }
    T* data() const { return p; }
    size_t size() const { return n; }
    T* begin() const { return p; }
    T* end() const { return p + n; }
};

// Text under construction: a growable char buffer written through a raw pointer (no per-character capacity checks).
struct TextBuf {
    char* base = nullptr;
    size_t len = 0, cap = 0;
    TextBuf() = default;
    TextBuf(TextBuf&& o) noexcept : base(o.base), len(o.len), cap(o.cap) { o.base = nullptr; o.len = o.cap = 0; }
    TextBuf& operator=(TextBuf&& o) noexcept {
        if (this != &o) { free(base); base = o.base; len = o.len; cap = o.cap; o.base = nullptr; o.len = o.cap = 0; }
        return *this;
    }
    TextBuf(const TextBuf&) = delete;
    TextBuf& operator=(const TextBuf&) = delete;
    ~TextBuf() { free(base); }
    // room for n more bytes; returns where to write them (nullptr: out of memory)
    char* need(size_t n) {
        if (cap - len < n) {
            const size_t want = std::max(len + n, cap + cap / 2 + (1u << 16));
            char* q = static_cast<char*>(realloc(base, want));
            if (!q) return nullptr;
            base = q;
            cap = want;
        }
        return base + len;
    }
    void advance_to(char* p) { len = (size_t)(p - base); }
    void append(const char* d, size_t n) {
        if (char* p = need(n)) { memcpy(p, d, n); len += n; }
    }
};

// Threads for `units` pieces of work: max(1, min(hardware threads, cap, units)).  When `env` names a set variable, its
// value (clamped to 1..64) is used instead.
inline int host_threads(size_t units, size_t cap, const char* env = nullptr) {
    if (env)
        if (const char* e = getenv(env)) return std::max(1, std::min(64, atoi(e)));
    return (int)std::max<size_t>(1, std::min<size_t>({(size_t)std::thread::hardware_concurrency(), cap, units}));
}

// f(k) for k in [0, n), each on a thread of its own; part 0 runs on the calling thread.  Returns once all are joined.
template <class F>
void run_parallel(int n, F&& f) {
    std::vector<std::thread> pool;
    for (int k = 1; k < n; ++k) pool.emplace_back([&f, k] { f(k); });
    if (n > 0) f(0);
    for (auto& th : pool) th.join();
}

// f(i) for every i in [0, n_items): `n_threads` workers take the items from a shared counter.
template <class F>
void claim_parallel(int n_threads, size_t n_items, F&& f) {
    std::atomic<size_t> next{0};
    run_parallel(std::max(1, n_threads), [&](int) {
        for (size_t i; (i = next.fetch_add(1)) < n_items;) f(i);
    });
}

// The whole file in `buf`, read in slices by min(cores, 16, size / 4 MiB) threads; buf[buf.size()] is a NUL.  The
// pages are first touched by the threads that fill them.  Returns RT_OK, or an error code with the error set.
inline int read_file(const char* path, HostArr<char>& buf) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { rt_io_set_error(std::string("cannot open ") + path); return RT_EINVAL; }
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); rt_io_set_error(std::string("cannot stat ") + path); return RT_EINVAL; }
    const size_t size = (size_t)st.st_size;
    if (!buf.alloc(size + 1)) { close(fd); rt_io_set_error("out of memory"); return RT_ENOMEM; }
    const int n_thr = host_threads(size >> 22, 16);
    std::atomic<bool> ok{true};
    run_parallel(n_thr, [&](int k) {
        size_t at = size * (size_t)k / n_thr;
        const size_t hi = size * (size_t)(k + 1) / n_thr;
        while (at < hi) {
            const ssize_t got = pread(fd, buf.p + at, hi - at, (off_t)at);
            if (got <= 0) { ok = false; return; }
            at += (size_t)got;
        }
    });
    close(fd);
    buf.p[size] = '\0';
    buf.n = size;
    if (!ok) { rt_io_set_error(std::string("short read of ") + path); return RT_EINVAL; }
    return RT_OK;
}

// The text of `t` moved into `buf` without a copy; `t` itself is freed.  The *_text loaders take their input so.
inline void adopt_text(rt_text* t, HostArr<char>& buf) {
    free(buf.p);
    buf.p = t->p;
    buf.n = t->n;
    delete t;
}

// Boundaries of n chunks of [lo, hi): n + 1 pointers; every chunk but the last ends after a '\n'.
inline std::vector<const char*> cut_lines(const char* lo, const char* hi, int n) {
    std::vector<const char*> cut{lo};
    for (int k = 1; k < n; ++k) {
        const char* guess = std::max(cut.back(), lo + (size_t)(hi - lo) * (size_t)k / n);
        const char* nl = guess < hi ? (const char*)memchr(guess, '\n', (size_t)(hi - guess)) : nullptr;
        cut.push_back(nl ? nl + 1 : hi);
    }
    cut.push_back(hi);
    return cut;
}

// Decimal digits of v at p; returns the end.  Coverage profiles are mostly one-digit numbers.
inline char* put_int(char* p, long long v) {
    static const char pairs[] =
        "00010203040506070809101112131415161718192021222324252627282930313233343536373839404142434445464748495051525354555657585960616263"
        "646566676869707172737475767778798081828384858687888990919293949596979899";
    unsigned long long u = (unsigned long long)v;
    if (v < 0) { *p++ = '-'; u = 0ull - u; }
    if (u < 10) { *p++ = (char)('0' + u); return p; }
    if (u < 100) { memcpy(p, pairs + 2 * u, 2); return p + 2; }
    char tmp[24];
    int k = 24;
    while (u >= 100) {
        const unsigned r = (unsigned)(u % 100);
        u /= 100;
        k -= 2;
        memcpy(tmp + k, pairs + 2 * r, 2);
    }
    if (u >= 10) { k -= 2; memcpy(tmp + k, pairs + 2 * u, 2); }
    else tmp[--k] = (char)('0' + u);
    memcpy(p, tmp + k, (size_t)(24 - k));
    return p + (24 - k);
}

// An output file with a write-behind thread: pieces of text are queued and written in order while the caller formats
// the next piece (or waits for the GPU).  At most kPendingMax bytes wait in the queue.  The first failed write is
// sticky: every later put and finish() report it, and nothing more is written.
class WriteBehind {
public:
    explicit WriteBehind(FILE* fh) : fh_(fh) {}
    WriteBehind(const WriteBehind&) = delete;
    WriteBehind& operator=(const WriteBehind&) = delete;
    ~WriteBehind() { finish(); }

    // text the writer owns from now on; false once a write has failed
    bool put(TextBuf&& b) {
        const size_t n = b.len;
        const char* p = b.base;
        return enqueue(Piece{std::move(b), p, n});
    }
    // [p, p + n) stays the caller's: it must stay valid and unchanged until wait_written() says it has been written
    bool put_view(const char* p, size_t n) { return enqueue(Piece{TextBuf(), p, n}); }
    // returns once the first k pieces are written; false once a write has failed
    bool wait_written(int64_t k) {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return written_ >= k || failed_; });
        return !failed_;
    }
    // drains the queue and joins the thread; false when any write failed
    bool finish() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            closing_ = true;
        }
        cv_.notify_all();
        if (th_.joinable()) th_.join();
        return !failed_;
    }

private:
    static constexpr size_t kPendingMax = 1ull << 30;
    struct Piece {
        TextBuf own;          // empty for a view
        const char* p;
        size_t n;
    };

    bool enqueue(Piece&& pc) {
        std::unique_lock<std::mutex> lk(mu_);
        if (failed_) return false;
        if (!th_.joinable()) th_ = std::thread([this] { run(); });
        cv_.wait(lk, [&] { return pending_ < kPendingMax || failed_; });
        pending_ += pc.n;
        queue_.push_back(std::move(pc));
        cv_.notify_all();
        return !failed_;
    }
    void run() {
        std::unique_lock<std::mutex> lk(mu_);
        for (;;) {
            cv_.wait(lk, [&] { return closing_ || !queue_.empty(); });
            if (queue_.empty()) return;
            Piece pc = std::move(queue_.front());
            queue_.pop_front();
            const bool skip = failed_;
            lk.unlock();
            const bool ok = skip || pc.n == 0 || fwrite(pc.p, 1, pc.n, fh_) == pc.n;
            lk.lock();
            pending_ -= pc.n;
            ++written_;
            if (!ok) failed_ = true;
            cv_.notify_all();
        }
    }

    FILE* fh_;
    std::thread th_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<Piece> queue_;
    size_t pending_ = 0;
    int64_t written_ = 0;
    bool closing_ = false, failed_ = false;
};

}  // namespace
