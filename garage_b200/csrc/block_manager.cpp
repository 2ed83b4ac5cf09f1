// block_manager.cpp -- C++ host-side mirror of garage_block::manager::BlockManager for the
// erasure-coded block path (see include/garage_block_manager.h for the mirrored surface and
// the reference file:line of every method).  Host code only: it reaches the GPU exclusively
// through the C ABI in include/garage_ec.h, exactly like the Rust shim of INTEGRATION.md would.
//
// Row f1 (batching front-end): rpc_put_block / reconstructing GETs / resync workers are called
// from many threads (reference: <= 3 blocks in flight per PUT, src/api/s3/put.rs:42; 8 resync
// workers, src/block/resync.rs:43).  One block per GPU call cannot amortise launch + PCIe
// latency, so calls are queued and dispatcher threads hand the GPU whole batches.  Data movement
// on the host is done by the CALLING threads, in parallel: a PUT lands its block in a pinned slot
// and later stores its shards straight out of the dispatcher's pinned parity buffer; a degraded
// GET / a resync worker reads the surviving shards from the node stores straight into its own
// pinned stripe slot, and the batch handed to the GPU is a list of slot pointers
// (garage_ec_reconstruct_stripes).  The dispatchers only issue the batch call.
#include "../../include/garage_block_manager.h"
#include "../../include/garage_ec.h"
#include "../../include/garage_placement.h"

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <deque>
#include <filesystem>
#include <functional>
#include <future>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

namespace {

using Hash = std::array<uint8_t, 32>;
using Clock = std::chrono::steady_clock;
struct HashHasher {
    size_t operator()(const Hash &h) const
    {
        size_t v;
        memcpy(&v, h.data() + 8, sizeof(v));  // content hashes are uniform already
        return v;
    }
};

Hash to_hash(const uint8_t *p)
{
    Hash h;
    memcpy(h.data(), p, 32);
    return h;
}

// copy into a pinned buffer the GPU reads next (landing copy of a PUT, survivors of a degraded GET)
inline void copy_for_dma(uint8_t *dst, const uint8_t *src, size_t n) { garage_ec_copy_for_dma(dst, src, n); }

uint32_t adler32_small(const uint8_t *p, size_t n)
{
    uint32_t a = 1, b = 0;
    for (size_t i = 0; i < n; i++) {
        a = (a + p[i]) % 65521;
        b = (b + a) % 65521;
    }
    return (b << 16) | a;
}

// ---------------------------------------------------------------- one node's local store
// mirrors BlockManagerLocked::write_block_inner / find_block / read_block_from /
// move_block_to_corrupted (src/block/manager.rs:720-819) with a map instead of a directory tree
struct ShardMeta {
    int index = -1;          // which of the k+m shards
    uint32_t block_len = 0;  // unpadded length of the whole block
    uint32_t shard_len = 0;
    uint8_t sum_kind = 0;    // GARAGE_EC_SUM_* of `sum`
    Hash sum{};              // integrity tag of the shard bytes (row f2)
};
// Memory of the in-memory node stores.  A 1 MiB PUT stores k+m = 14 buffers of ~100 KB: through malloc that is
// 1.4 MiB of fresh pages per block (~360 page faults, plus the allocator's own heap growth), all against one
// address space -- at 12 000 blocks/s the process spends its time in the kernel's fault path, not copying.  The arena
// carves cells out of large anonymous regions, hands freed cells back out (LIFO per size class), and can be
// filled ahead of time (reserve), the way the page cache of a disk-backed node is not charged to a PUT either.
class ShardArena {
public:
    static ShardArena &instance()
    {
        static ShardArena *a = new ShardArena();  // never destroyed: shards may outlive any one manager
        return *a;
    }
    static size_t cell_size(size_t n) { return n <= 4096 ? (n + 63) / 64 * 64 : (n + 4095) / 4096 * 4096; }
    uint8_t *alloc(size_t n, size_t *cap)
    {
        const size_t c = cell_size(n);
        *cap = c;
        if (c > kRegion / 4) return static_cast<uint8_t *>(malloc(c));
        std::lock_guard<std::mutex> lk(mu_);
        auto it = free_.find(c);
        if (it != free_.end() && !it->second.empty()) {
            uint8_t *p = it->second.back();
            it->second.pop_back();
            return p;
        }
        return carve(c);
    }
    void free(uint8_t *p, size_t cap)
    {
        if (!p) return;
        if (cap > kRegion / 4) return ::free(p);
        std::lock_guard<std::mutex> lk(mu_);
        free_[cap].push_back(p);
    }
    // make `count` cells for buffers of `n` bytes available with their pages already present
    void reserve(size_t n, size_t count)
    {
        const size_t c = cell_size(n);
        if (c > kRegion / 4 || count == 0) return;
        std::vector<uint8_t *> cells;
        {
            std::lock_guard<std::mutex> lk(mu_);
            auto &fl = free_[c];
            if (fl.size() >= count) return;  // recycled cells have been written before
            count -= fl.size();
            cells.reserve(count);
            for (size_t i = 0; i < count; i++) {
                uint8_t *p = carve(c);
                if (!p) break;
                cells.push_back(p);
            }
        }
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const size_t nt = std::min<size_t>(std::min(hw, 32u), cells.size() / 64 + 1);
        std::vector<std::thread> th;
        for (size_t t = 0; t < nt; t++)
            th.emplace_back([&, t] {
                for (size_t i = t; i < cells.size(); i += nt)
                    for (size_t o = 0; o < c; o += 4096) reinterpret_cast<volatile uint8_t *>(cells[i])[o] = 0;
            });
        for (auto &x : th) x.join();
        std::lock_guard<std::mutex> lk(mu_);
        auto &fl = free_[c];
        fl.insert(fl.end(), cells.begin(), cells.end());
    }

private:
    static constexpr size_t kRegion = (size_t)256 << 20;
    std::mutex mu_;
    uint8_t *cur_ = nullptr, *end_ = nullptr;
    std::unordered_map<size_t, std::vector<uint8_t *>> free_;
    uint8_t *carve(size_t c)  // mu_ held
    {
        if (cur_ == nullptr || (size_t)(end_ - cur_) < c) {
            void *m = mmap(nullptr, kRegion, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
            if (m == MAP_FAILED) return nullptr;
            cur_ = static_cast<uint8_t *>(m);  // the tail of the previous region is abandoned (< one cell)
            end_ = cur_ + kRegion;
        }
        uint8_t *p = cur_;
        cur_ += c;
        return p;
    }
};

// owning byte buffer in arena memory, with the slice of std::vector's interface the store uses
class ShardBytes {
public:
    ShardBytes() = default;
    ShardBytes(const ShardBytes &o) { assign(o.p_, o.p_ + o.n_); }
    ShardBytes(ShardBytes &&o) noexcept : p_(o.p_), n_(o.n_), cap_(o.cap_) { o.p_ = nullptr, o.n_ = o.cap_ = 0; }
    ShardBytes &operator=(const ShardBytes &o)
    {
        if (this != &o) assign(o.p_, o.p_ + o.n_);
        return *this;
    }
    ShardBytes &operator=(ShardBytes &&o) noexcept
    {
        if (this != &o) {
            ShardArena::instance().free(p_, cap_);
            p_ = o.p_, n_ = o.n_, cap_ = o.cap_;
            o.p_ = nullptr, o.n_ = o.cap_ = 0;
        }
        return *this;
    }
    ~ShardBytes() { ShardArena::instance().free(p_, cap_); }
    void resize(size_t n)  // contents are not preserved across a growth (no caller needs that)
    {
        if (n > cap_) {
            ShardArena::instance().free(p_, cap_);
            p_ = nullptr, cap_ = 0;
            p_ = ShardArena::instance().alloc(n, &cap_);
            if (!p_) {
                n_ = cap_ = 0;
                throw std::bad_alloc();
            }
        }
        n_ = n;
    }
    void assign(const uint8_t *b, const uint8_t *e)
    {
        const size_t n = (size_t)(e - b);
        if (p_ && b >= p_ && b < p_ + cap_) {  // source inside this buffer
            memmove(p_, b, n);
            n_ = n;
            return;
        }
        resize(n);
        if (n) memcpy(p_, b, n);
    }
    uint8_t *data() { return p_; }
    const uint8_t *data() const { return p_; }
    size_t size() const { return n_; }
    bool empty() const { return n_ == 0; }
    uint8_t &operator[](size_t i) { return p_[i]; }

private:
    uint8_t *p_ = nullptr;
    size_t n_ = 0, cap_ = 0;
};

struct StoredShard : ShardMeta {
    ShardBytes bytes;
};

// On-disk shard file (row f3; mirrors the tmp-file -> rename -> .corrupted life cycle of
// BlockManagerLocked::write_block_inner / move_block_to_corrupted, src/block/manager.rs:720-819,
// and the directory scheme data_dir/<h[0]>/<h[1]>/<hex(h)> of src/block/layout.rs:286-291):
//   <data_dir>/node<N>/<hh>/<hh>/<64 hex>.shard        64-byte header + shard bytes
// hdr_check covers the first 48 bytes (every field a reader acts on), so a flipped index /
// block_len / sum kind is caught like a flipped data byte.
struct ShardFileHeader {
    char magic[4];  // "GEC1"
    uint8_t k, m, index, sum_kind;
    uint32_t block_len;
    uint32_t shard_len;
    uint8_t sum[32];
    uint32_t hdr_check;  // Adler-32 of bytes [0, 48)
    uint8_t pad[12];
};
static_assert(sizeof(ShardFileHeader) == 64, "shard file header is 64 bytes");

std::string hex_of(const uint8_t *p, size_t n)
{
    static const char *d = "0123456789abcdef";
    std::string o;
    for (size_t i = 0; i < n; i++) {
        o.push_back(d[p[i] >> 4]);
        o.push_back(d[p[i] & 15]);
    }
    return o;
}

enum ReadResult { kReadOk = 0, kReadMissing = 1, kReadInvalid = 2 };

struct Node {
    std::mutex mu;  // stands in for the 256 hash-sharded mutexes (manager.rs:114,679-689)
    bool up = true;
    bool fsync_data = false;  // data_fsync (util/config.rs), manager.rs:775-789
    std::string dir;          // empty: in-memory store
    int k = 0, m = 0;
    // in-memory mode: immutable shards behind shared pointers, so the node lock only covers the map operation -- the
    // 100 KB copies happen outside it (the reference shards its lock 256 ways per node, manager.rs:114,679-689; with
    // one lock per node and the copies inside it, 128 clients serialised on 14 mutexes at ~12 GiB/s)
    using ShardPtr = std::shared_ptr<const StoredShard>;
    std::unordered_map<Hash, ShardPtr, HashHasher> shards;
    std::unordered_map<Hash, ShardPtr, HashHasher> corrupted;  // the ".corrupted" quarantine
    std::deque<Hash> resync_queue;                                // block_local_resync_queue (resync.rs:90)
    std::unordered_set<Hash, HashHasher> queued;

    std::string path_of(const Hash &h, const char *ext) const
    {
        return dir + "/" + hex_of(h.data(), 1) + "/" + hex_of(h.data() + 1, 1) + "/" + hex_of(h.data(), 32) + ext;
    }
    void store_put_ptr(const Hash &h, ShardPtr sp) { shards[h] = std::move(sp); }  // in-memory: the copy was made by the caller
    ShardPtr store_find(const Hash &h) const
    {
        auto it = shards.find(h);
        return it == shards.end() ? ShardPtr() : it->second;
    }
    bool meta_valid(const ShardMeta &mt) const
    {
        if (mt.index < 0 || mt.index >= k + m) return false;
        return mt.shard_len == (uint32_t)(((uint64_t)mt.block_len + (unsigned)k - 1) / (unsigned)k);
    }
    // all store_* are called with `mu` held
    bool store_put(const Hash &h, const ShardMeta &mt, const uint8_t *bytes, size_t n)
    {
        if (dir.empty()) {
            auto sp = std::make_shared<StoredShard>();
            static_cast<ShardMeta &>(*sp) = mt;
            sp->bytes.assign(bytes, bytes + n);
            shards[h] = std::move(sp);
            return true;
        }
        std::error_code ec;
        const std::string sub = dir + "/" + hex_of(h.data(), 1) + "/" + hex_of(h.data() + 1, 1);
        std::filesystem::create_directories(sub, ec);
        const std::string fin = path_of(h, ".shard"), tmp = fin + ".tmp" + std::to_string((unsigned long)::getpid());
        ShardFileHeader hd;
        memset(&hd, 0, sizeof(hd));
        memcpy(hd.magic, "GEC1", 4);
        hd.k = (uint8_t)k;
        hd.m = (uint8_t)m;
        hd.index = (uint8_t)mt.index;
        hd.sum_kind = mt.sum_kind;
        hd.block_len = mt.block_len;
        hd.shard_len = (uint32_t)n;
        memcpy(hd.sum, mt.sum.data(), 32);
        hd.hdr_check = adler32_small(reinterpret_cast<const uint8_t *>(&hd), 48);
        FILE *f = fopen(tmp.c_str(), "wb");
        if (!f) return false;
        bool ok = fwrite(&hd, sizeof(hd), 1, f) == 1 && (n == 0 || fwrite(bytes, n, 1, f) == 1);
        if (ok) ok = fflush(f) == 0;
        if (ok && fsync_data) ok = ::fsync(fileno(f)) == 0;  // manager.rs:775-777
        ok = (fclose(f) == 0) && ok;
        if (ok) ok = ::rename(tmp.c_str(), fin.c_str()) == 0;  // atomic publish (manager.rs:790-795)
        if (ok && fsync_data) {                                 // and the directory entry (manager.rs:797-803)
            const int dfd = ::open(sub.c_str(), O_RDONLY | O_DIRECTORY);
            if (dfd >= 0) {
                ok = ::fsync(dfd) == 0;
                ::close(dfd);
            }
        }
        if (!ok) ::remove(tmp.c_str());
        return ok;
    }
    // shard bytes straight into `dst` (cap bytes available), metadata into `mt`
    ReadResult store_read_into(const Hash &h, uint8_t *dst, size_t cap, ShardMeta &mt) const
    {
        if (dir.empty()) {
            auto it = shards.find(h);
            if (it == shards.end()) return kReadMissing;
            return copy_out(*it->second, dst, cap, mt);
        }
        FILE *f = fopen(path_of(h, ".shard").c_str(), "rb");  // find_block (manager.rs:627-662)
        if (!f) return kReadMissing;
        ShardFileHeader hd;
        ReadResult r = kReadInvalid;
        struct stat sb;
        // a header that fails any of these is a corrupt shard, never a reason to allocate or read
        // what it claims (a flipped shard_len must not become a 4 GiB resize)
        if (fread(&hd, sizeof(hd), 1, f) == 1 && memcmp(hd.magic, "GEC1", 4) == 0 &&
            hd.hdr_check == adler32_small(reinterpret_cast<const uint8_t *>(&hd), 48) && hd.k == k && hd.m == m &&
            fstat(fileno(f), &sb) == 0 && (uint64_t)sb.st_size == (uint64_t)hd.shard_len + sizeof(hd)) {
            mt.index = hd.index;
            mt.block_len = hd.block_len;
            mt.shard_len = hd.shard_len;
            mt.sum_kind = hd.sum_kind;
            memcpy(mt.sum.data(), hd.sum, 32);
            if (meta_valid(mt) && mt.shard_len <= cap && (mt.shard_len == 0 || fread(dst, mt.shard_len, 1, f) == 1))
                r = kReadOk;
        }
        fclose(f);
        return r;
    }
    ReadResult copy_out(const StoredShard &sh, uint8_t *dst, size_t cap, ShardMeta &mt, bool for_dma = false) const
    {
        mt = sh;
        if (!meta_valid(mt) || sh.bytes.size() != mt.shard_len || mt.shard_len > cap) return kReadInvalid;
        if (for_dma) copy_for_dma(dst, sh.bytes.data(), mt.shard_len);
        else if (mt.shard_len) memcpy(dst, sh.bytes.data(), mt.shard_len);
        return kReadOk;
    }
    bool store_get(const Hash &h, StoredShard &out) const  // a copy (scrub snapshots, inspection)
    {
        if (dir.empty()) {
            auto it = shards.find(h);
            if (it == shards.end()) return false;
            out = *it->second;
            return true;
        }
        std::error_code ec;
        const auto sz = std::filesystem::file_size(path_of(h, ".shard"), ec);
        if (ec || sz < sizeof(ShardFileHeader) || sz > (1ull << 31)) return false;
        out.bytes.resize((size_t)sz - sizeof(ShardFileHeader));
        ShardMeta mt;
        if (store_read_into(h, out.bytes.data(), out.bytes.size(), mt) != kReadOk) return false;
        static_cast<ShardMeta &>(out) = mt;
        return true;
    }
    bool store_has(const Hash &h) const
    {
        if (dir.empty()) return shards.count(h) != 0;
        std::error_code ec;
        return std::filesystem::exists(path_of(h, ".shard"), ec);
    }
    bool store_erase(const Hash &h)
    {
        if (dir.empty()) return shards.erase(h) != 0;
        return ::remove(path_of(h, ".shard").c_str()) == 0;
    }
    void store_quarantine(const Hash &h)  // move_block_to_corrupted (manager.rs:807-819)
    {
        if (dir.empty()) {
            auto it = shards.find(h);
            if (it != shards.end()) {
                corrupted[h] = std::move(it->second);
                shards.erase(it);
            }
            return;
        }
        ::rename(path_of(h, ".shard").c_str(), path_of(h, ".corrupted").c_str());
    }
    void store_list(std::vector<Hash> &out) const  // BlockStoreIterator (repair.rs:634-764)
    {
        if (dir.empty()) {
            for (auto &kv : shards) out.push_back(kv.first);
            return;
        }
        std::error_code ec;
        for (auto it = std::filesystem::recursive_directory_iterator(dir, ec);
             !ec && it != std::filesystem::recursive_directory_iterator(); it.increment(ec)) {
            const std::string name = it->path().filename().string();
            if (name.size() != 64 + 6 || name.compare(64, 6, ".shard") != 0) continue;
            Hash h;
            bool ok = true;
            for (int i = 0; i < 32 && ok; i++) {
                auto v = [&](char c) { return c >= '0' && c <= '9' ? c - '0' : (c >= 'a' && c <= 'f' ? c - 'a' + 10 : -1); };
                const int hi = v(name[2 * i]), lo = v(name[2 * i + 1]);
                ok = hi >= 0 && lo >= 0;
                h[i] = (uint8_t)((hi << 4) | lo);
            }
            if (ok) out.push_back(h);
        }
    }
};

// ---------------------------------------------------------------- counting semaphore (bytes)
// mirrors buffer_kb_semaphore (manager.rs:156, 380-385)
class ByteSemaphore {
public:
    explicit ByteSemaphore(uint64_t cap) : cap_(cap), avail_(cap) {}
    void acquire(uint64_t n)
    {
        if (n > cap_) n = cap_;
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return avail_ >= n; });
        avail_ -= n;
    }
    void release(uint64_t n)
    {
        if (n > cap_) n = cap_;
        {
            std::lock_guard<std::mutex> lk(mu_);
            avail_ += n;
        }
        cv_.notify_all();
    }

private:
    uint64_t cap_, avail_;
    std::mutex mu_;
    std::condition_variable cv_;
};

// ---------------------------------------------------------------- generic batcher (row f1)
template <class Item>
class Batcher {
public:
    using Run = std::function<void(int /*worker*/, std::vector<Item *> &)>;
    // `workers` dispatcher threads pull batches from one queue: while one batch is on the GPU the
    // next one is being collected (each worker owns a garage_ec context and buffers)
    Batcher(size_t max_items, unsigned linger_us, int workers, Run run, std::function<void()> on_thread_start)
        : max_(std::max<size_t>(1, max_items)), linger_(linger_us), run_(std::move(run))
    {
        for (int w = 0; w < std::max(1, workers); w++)
            th_.emplace_back([this, w, on_thread_start] {
                if (on_thread_start) on_thread_start();
                loop(w);
            });
    }
    ~Batcher()
    {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }
    // blocks the calling thread until its item has been processed in some batch
    int submit(Item &it)
    {
        std::future<int> f = it.done.get_future();
        {
            std::lock_guard<std::mutex> lk(mu_);
            q_.push_back(&it);
        }
        cv_.notify_all();
        return f.get();
    }
    uint64_t batches() const { return batches_.load(); }
    uint64_t items() const { return items_.load(); }

private:
    void loop(int w)
    {
        std::vector<Item *> batch;
        for (;;) {
            batch.clear();
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
                if (stop_ && q_.empty()) return;
                // linger: give concurrent callers a moment to join the batch
                const auto deadline = Clock::now() + std::chrono::microseconds(linger_);
                while (q_.size() < max_ && !stop_) {
                    if (cv_.wait_until(lk, deadline) == std::cv_status::timeout) break;
                }
                while (!q_.empty() && batch.size() < max_) {
                    batch.push_back(q_.front());
                    q_.pop_front();
                }
            }
            if (batch.empty()) continue;  // another worker took them
            batches_++;
            items_ += batch.size();
            // nothing may escape a dispatcher thread: an exception (bad_alloc in a staging vector)
            // fails the items of this batch instead of terminating the process
            try {
                run_(w, batch);  // sets every item's promise
            } catch (...) {
                for (Item *it : batch)
                    if (!it->fulfilled) {
                        it->fulfilled = true;
                        it->done.set_value(GARAGE_EC_E_NOMEM);
                    }
            }
        }
    }
    const size_t max_;
    const unsigned linger_;
    Run run_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<Item *> q_;
    bool stop_ = false;
    std::atomic<uint64_t> batches_{0}, items_{0};
    std::vector<std::thread> th_;
};

// pool of pinned slots: the calling thread fills its slot (in parallel with every other caller)
// so the dispatcher's DMA runs at PCIe speed from pinned, NUMA-local memory -- in Garage proper
// the body copy of BytesBuf::take_exact (src/net/bytes_buf.rs:66-117) would land here directly
class SlotPool {
public:
    bool init(garage_ec_ctx *ctx, size_t slots, size_t slot_bytes)
    {
        ctx_ = ctx;
        slot_bytes_ = (slot_bytes + 4095) / 4096 * 4096;
        if (garage_ec_host_alloc(ctx, &base_, slots * slot_bytes_) != GARAGE_EC_OK) return false;
        for (size_t i = 0; i < slots; i++) free_.push_back(static_cast<uint8_t *>(base_) + i * slot_bytes_);
        return true;
    }
    uint8_t *acquire()
    {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return !free_.empty(); });
        uint8_t *p = free_.back();
        free_.pop_back();
        return p;
    }
    void release(uint8_t *p)
    {
        {
            std::lock_guard<std::mutex> lk(mu_);
            free_.push_back(p);
        }
        cv_.notify_one();
    }
    size_t slot_bytes() const { return slot_bytes_; }
    void destroy()
    {
        if (base_) garage_ec_host_free(ctx_, base_);
        base_ = nullptr;
    }

private:
    garage_ec_ctx *ctx_ = nullptr;
    void *base_ = nullptr;
    size_t slot_bytes_ = 0;
    std::mutex mu_;
    std::condition_variable cv_;
    std::vector<uint8_t *> free_;
};
struct SlotLease {  // RAII: a slot goes back to its pool on every path
    SlotPool &pool;
    uint8_t *p;
    explicit SlotLease(SlotPool &pl) : pool(pl), p(pl.acquire()) {}
    ~SlotLease() { pool.release(p); }
    SlotLease(const SlotLease &) = delete;
    SlotLease &operator=(const SlotLease &) = delete;
};

// pinned output buffer of one encode batch (parity rows + shard tags).  The callers of the batch
// store their shards straight out of it; the dispatcher reuses it only when they are all done.
struct EncBatchBuf {
    garage_ec_ctx *ctx = nullptr;
    void *p = nullptr;
    size_t cap = 0;
    std::mutex mu;
    std::condition_variable cv;
    int pending = 0;
    uint8_t *get(size_t n)
    {
        if (n > cap) {
            if (p) garage_ec_host_free(ctx, p);
            p = nullptr;
            cap = 0;
            const size_t want = std::max(n, (size_t)1 << 20);
            if (garage_ec_host_alloc(ctx, &p, want) != GARAGE_EC_OK) return nullptr;
            cap = want;
        }
        return static_cast<uint8_t *>(p);
    }
    void wait_idle()
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return pending == 0; });
    }
    void set_pending(int n)
    {
        std::lock_guard<std::mutex> lk(mu);
        pending = n;
    }
    void done_one()
    {
        bool zero;
        {
            std::lock_guard<std::mutex> lk(mu);
            zero = --pending == 0;
        }
        if (zero) cv.notify_all();
    }
    void release()
    {
        if (p) garage_ec_host_free(ctx, p);
        p = nullptr;
        cap = 0;
    }
};

struct EncodeItem {
    const uint8_t *data = nullptr;  // the block (pinned slot, or the caller's buffer for oversize blocks)
    uint32_t len = 0;
    // filled by the dispatcher: parity row i at parity + i * pstride, tags of the k+m shards
    const uint8_t *parity = nullptr;
    size_t pstride = 0;
    const uint8_t *sums = nullptr;
    EncBatchBuf *buf = nullptr;  // to be released (done_one) once the shards are stored
    bool fulfilled = false;
    std::promise<int> done;
};

struct ReconItem {
    uint8_t *stripe = nullptr;  // pinned slot: k+m shards, `stride` apart, survivors filled in by the caller
    size_t stride = 0;
    uint32_t block_len = 0;
    uint8_t present[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M] = {0};
    uint8_t want[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M] = {0};
    bool fulfilled = false;
    std::promise<int> done;
};

// pinned scratch that grows on demand (owned by one thread at a time)
struct PinnedBuf {
    garage_ec_ctx *ctx = nullptr;
    void *p = nullptr;
    size_t cap = 0;
    uint8_t *get(size_t n)
    {
        if (n > cap) {
            if (p) garage_ec_host_free(ctx, p);
            p = nullptr;
            cap = 0;
            if (garage_ec_host_alloc(ctx, &p, n) != GARAGE_EC_OK) return nullptr;
            cap = n;
        }
        return static_cast<uint8_t *>(p);
    }
    void release()
    {
        if (p) garage_ec_host_free(ctx, p);
        p = nullptr;
        cap = 0;
    }
    ~PinnedBuf() { release(); }
};

struct RcEntry {
    int64_t count = 0;
    Clock::time_point zero_since{};  // when the count last dropped to 0 (BLOCK_GC_DELAY, manager.rs:49-52)
};

}  // namespace

// ================================================================= the manager
struct garage_bm {
    garage_bm_config cfg{};
    int k = 0, m = 0, tot = 0;
    int sum_kind = GARAGE_EC_SUM_ADLER8;
    size_t slot_stride = 0;  // stride of the largest block's shards: geometry of every stripe slot
    static constexpr int kWorkers = 3;  // dispatcher threads per batcher (overlap PCIe / GPU / collection)
    garage_ec_ctx *ec = nullptr;                   // scrub + geometry helpers
    garage_ec_ctx *enc_ctx[kWorkers] = {nullptr};  // one context (= its own staging lanes) per worker
    garage_ec_ctx *rec_ctx[kWorkers] = {nullptr};
    SlotPool put_slots;     // one block each
    SlotPool stripe_slots;  // (k+m) x slot_stride each: degraded GETs, resync workers
    std::vector<std::unique_ptr<Node>> nodes;
    // stands in for the block_ref / rc tables (src/model/s3/block_ref_table.rs, src/block/rc.rs):
    // which blocks exist and how long they are.  Lock order: refs_mu before any Node::mu.
    std::mutex refs_mu;
    std::unordered_map<Hash, uint32_t, HashHasher> refs;
    // block reference counts (src/block/rc.rs): only blocks that went through block_incref /
    // block_decref have an entry; a block without entry is treated as needed (rc > 0)
    std::unordered_map<Hash, RcEntry, HashHasher> rc;
    std::unique_ptr<ByteSemaphore> ram;
    std::unique_ptr<Batcher<EncodeItem>> enc_batcher;
    std::unique_ptr<Batcher<ReconItem>> rec_batcher;
    static constexpr int kEncBufs = 4;  // pinned output buffers per dispatcher: a batch's callers store their shards
                                        // out of one while the dispatcher fills the next ones
    EncBatchBuf enc_out[kWorkers][kEncBufs];
    int enc_next[kWorkers] = {0};
    PinnedBuf scrub_buf;
    std::mutex scrub_mu;
    std::atomic<bool> warmed{false};
    // metrics (src/block/metrics.rs)
    std::atomic<uint64_t> bytes_written{0}, bytes_read{0}, corruption_counter{0}, resync_counter{0},
        resync_error_counter{0}, resync_recv_counter{0}, delete_counter{0}, put_calls{0}, reconstruct_calls{0},
        scrub_checked{0}, scrub_corrupt{0}, enc_gpu_us{0}, rec_gpu_us{0}, corrupt_data_errors{0}, write_errors{0};
    std::atomic<uint64_t> put_ns_slot{0}, put_ns_land{0}, put_ns_wait{0}, put_ns_store{0};

    size_t shard_len_of(uint32_t block_len) const { return garage_ec_shard_len(block_len, k); }

    // rpc/layout/version.rs:117-137: top 8 bits of the hash -> partition -> k+m distinct nodes, shard i on the
    // i-th of them.  The ring is a garage_layout (row f4, include/garage_placement.h) filled at create with
    // partition p -> nodes (p mod n) + i; any other ring (zones, capacities: garage_layout_compute) plugs in here.
    garage_layout *layout = nullptr;
    ~garage_bm() { garage_layout_free(layout); }
    void storage_nodes_of(const Hash &h, int *out) const
    {
        static_assert(sizeof(int) == sizeof(int32_t), "node ids are 32-bit");
        if (layout && garage_layout_nodes_of(layout, h.data(), reinterpret_cast<int32_t *>(out)) == GARAGE_LAYOUT_OK) return;
        const int n = (int)nodes.size();  // more nodes than a ring row can name: the same rule, computed
        const int p = h[0] % n;
        for (int i = 0; i < tot; i++) out[i] = (p + i) % n;
    }

    void put_to_resync(int node, const Hash &h)  // manager.rs:592-605 / resync.rs:put_to_resync
    {
        Node &nd = *nodes[node];
        std::lock_guard<std::mutex> lk(nd.mu);
        if (nd.queued.insert(h).second) nd.resync_queue.push_back(h);
    }

    void shard_tag(const uint8_t *bytes, size_t n, Hash &out) const
    {
        garage_ec_shard_sum_host(sum_kind, bytes, n, out.data());
    }

    // manager.rs:517-530 write_block: false if the node is down or the store failed (ENOSPC, EACCES ...)
    bool write_shard(int node, const Hash &h, int index, uint32_t block_len, const uint8_t *bytes, size_t n,
                     const uint8_t *sum32)
    {
        ShardMeta mt;
        mt.index = index;
        mt.block_len = block_len;
        mt.shard_len = (uint32_t)n;
        mt.sum_kind = (uint8_t)sum_kind;
        memcpy(mt.sum.data(), sum32, 32);
        Node &nd = *nodes[node];
        bool ok;
        if (nd.dir.empty()) {
            auto sp = std::make_shared<StoredShard>();  // the copy happens before the node lock is taken
            static_cast<ShardMeta &>(*sp) = mt;
            sp->bytes.assign(bytes, bytes + n);
            Node::ShardPtr old;
            {
                std::lock_guard<std::mutex> lk(nd.mu);
                if (!nd.up) return false;
                auto &slot_ref = nd.shards[h];
                old.swap(slot_ref);
                slot_ref = std::move(sp);
            }
            ok = true;  // `old` (a replaced shard) is freed here, outside the lock
        } else {
            std::lock_guard<std::mutex> lk(nd.mu);
            if (!nd.up) return false;
            ok = nd.store_put(h, mt, bytes, n);
        }
        if (ok) bytes_written += n;
        else write_errors++;
        return ok;
    }

    void quarantine(int node, const Hash &h)
    {
        corruption_counter++;
        {
            Node &nd = *nodes[node];
            std::lock_guard<std::mutex> lk(nd.mu);
            nd.store_quarantine(h);
        }
        put_to_resync(node, h);
    }

    // manager.rs:554-609 read_block + read_block_from: the verified shard bytes land in `dst`.
    // A bad header or a tag mismatch quarantines the shard and queues a resync, like the reference.
    // `for_dma`: the GPU reads `dst` next (degraded GET, resync): see copy_for_dma
    bool read_shard_into(int node, const Hash &h, uint8_t *dst, size_t cap, ShardMeta &mt, bool for_dma = false)
    {
        Node &nd = *nodes[node];
        ReadResult r;
        const uint8_t *check = dst;
        Node::ShardPtr sp;
        if (nd.dir.empty()) {
            {
                std::lock_guard<std::mutex> lk(nd.mu);
                if (!nd.up) return false;
                sp = nd.store_find(h);
            }
            r = sp ? nd.copy_out(*sp, dst, cap, mt, for_dma) : kReadMissing;  // the copy happens outside the node lock
            if (sp && for_dma) check = sp->bytes.data();  // same bytes, and these are still in the cache
        } else {
            std::lock_guard<std::mutex> lk(nd.mu);
            if (!nd.up) return false;
            r = nd.store_read_into(h, dst, cap, mt);
        }
        if (r == kReadMissing) return false;
        if (r == kReadOk) {
            bytes_read += mt.shard_len;
            Hash got;
            if (garage_ec_shard_sum_host(mt.sum_kind, check, mt.shard_len, got.data()) == GARAGE_EC_OK && got == mt.sum)
                return true;
        }
        quarantine(node, h);
        return false;
    }

    // ---- batch runners (dispatcher threads) -------------------------------------------------
    void run_encode(int w, std::vector<EncodeItem *> &b)
    {
        const size_t n = b.size();
        uint32_t max_len = 0;
        std::vector<const uint8_t *> ptrs(n);
        std::vector<uint32_t> lens(n);
        for (size_t i = 0; i < n; i++) {
            ptrs[i] = b[i]->data;
            lens[i] = b[i]->len;
            max_len = std::max(max_len, b[i]->len);
        }
        const size_t stride = garage_ec_stride_for(garage_ec_shard_len(max_len, k));
        EncBatchBuf &bb = enc_out[w][enc_next[w] = (enc_next[w] + 1) % kEncBufs];
        bb.wait_idle();  // the callers of the batch that last used this buffer have stored their shards
        uint8_t *par = bb.get(n * m * stride + n * tot * 32);
        int rc = par ? GARAGE_EC_OK : GARAGE_EC_E_NOMEM;
        uint8_t *sums = par ? par + n * m * stride : nullptr;
        const auto t0 = Clock::now();
        if (rc == GARAGE_EC_OK)
            rc = garage_ec_encode_blocks_with_sums(enc_ctx[w], ptrs.data(), lens.data(), n, par, sums, stride);
        enc_gpu_us += (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(Clock::now() - t0).count();
        if (rc == GARAGE_EC_OK) bb.set_pending((int)n);
        for (size_t i = 0; i < n; i++) {
            if (rc == GARAGE_EC_OK) {
                b[i]->parity = par + i * m * stride;
                b[i]->pstride = stride;
                b[i]->sums = sums + i * tot * 32;
                b[i]->buf = &bb;
            }
            b[i]->fulfilled = true;
            b[i]->done.set_value(rc);
        }
    }

    void run_reconstruct(int w, std::vector<ReconItem *> &b)
    {
        const size_t n = b.size();
        std::vector<uint8_t *> stripes(n);
        std::vector<uint8_t> present(n * tot), want(n * tot);
        std::vector<uint32_t> lens(n);
        std::vector<int32_t> status(n, 0);
        for (size_t i = 0; i < n; i++) {
            stripes[i] = b[i]->stripe;
            lens[i] = (uint32_t)shard_len_of(b[i]->block_len);
            memcpy(present.data() + i * tot, b[i]->present, tot);
            memcpy(want.data() + i * tot, b[i]->want, tot);
        }
        const auto t0 = Clock::now();
        int rc = garage_ec_reconstruct_stripes(rec_ctx[w], stripes.data(), present.data(), want.data(), status.data(),
                                               lens.data(), slot_stride, n);
        rec_gpu_us += (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(Clock::now() - t0).count();
        for (size_t i = 0; i < n; i++) {
            int r = rc;
            if (rc == GARAGE_EC_OK || rc == GARAGE_EC_E_UNRECOVERABLE) r = status[i] ? GARAGE_BM_E_MISSING_BLOCK : GARAGE_BM_OK;
            b[i]->fulfilled = true;
            b[i]->done.set_value(r);
        }
    }

    // Read the valid shards of `h` from every up node except `skip_node` into the stripe slot
    // (shard i at slot + i*slot_stride).  Data shards first (a complete set needs no GPU), then only
    // as many parity shards as it takes to reach k -- the reference likewise stops at the first good
    // copy (manager.rs:292-334); RpcHelper::try_call_many with quorum k is the real-cluster form.
    // A shard whose header disagrees with the others on the block length, or that sits under the
    // wrong index, is treated like a corrupt one.  `all`: do not stop at k (corruption hunting).
    int gather_into(const Hash &h, int skip_node, uint8_t *slot, uint8_t *have, uint32_t &block_len, bool all = false,
                    bool for_gpu = false)
    {
        int who[64];
        storage_nodes_of(h, who);
        memset(have, 0, tot);
        uint32_t expect = 0;
        bool have_expect = false;
        {
            std::lock_guard<std::mutex> lk(refs_mu);
            auto it = refs.find(h);
            if (it != refs.end()) {
                expect = it->second;
                have_expect = true;
            }
        }
        int count = 0;
        auto try_shard = [&](int i) {
            if (who[i] == skip_node || have[i]) return;
            ShardMeta mt;
            if (!read_shard_into(who[i], h, slot + (size_t)i * slot_stride, slot_stride, mt, for_gpu)) return;
            if (mt.index != i || (have_expect && mt.block_len != expect)) {
                quarantine(who[i], h);  // a stale or misplaced shard with a self-consistent tag
                return;
            }
            if (!have_expect) {
                expect = mt.block_len;
                have_expect = true;
            }
            have[i] = 1;
            count++;
        };
        for (int i = 0; i < k; i++) {
            try_shard(i);
            for_gpu |= !have[i];  // a data shard is missing: this stripe goes through the GPU
        }
        for (int i = k; i < tot && (all || count < k); i++) try_shard(i);
        block_len = expect;
        return count;
    }

    int reconstruct_in_slot(uint8_t *slot, uint32_t block_len, const uint8_t *have, const uint8_t *want)
    {
        reconstruct_calls++;
        ReconItem it;
        it.stripe = slot;
        it.stride = slot_stride;
        it.block_len = block_len;
        memcpy(it.present, have, tot);
        memcpy(it.want, want, tot);
        return rec_batcher->submit(it);
    }

    void assemble(const uint8_t *slot, uint32_t block_len, uint8_t *out) const
    {
        const size_t L = shard_len_of(block_len);
        for (int j = 0; j < k; j++) {
            const size_t off = (size_t)j * L;
            if (off >= block_len) break;
            memcpy(out + off, slot + (size_t)j * slot_stride, std::min(L, (size_t)block_len - off));
        }
    }

    bool content_ok(const Hash &h, const uint8_t *data, size_t len) const
    {
        if (!cfg.verify_content_hash) return true;
        Hash got;
        garage_ec_blake2sum(data, len, got.data());  // DataBlock::verify, src/block/block.rs:69-83
        return got == h;
    }

    int rpc_put_block(const Hash &h, const uint8_t *data, size_t len)
    {
        if (len == 0 || len > cfg.block_size) return GARAGE_BM_E_MESSAGE;  // blocks are at most block_size (put.rs:583-617)
        int who[64];
        storage_nodes_of(h, who);  // manager.rs:373
        // DataBlock::from_buffer (manager.rs:376): compression is 'none' in this mirror
        const uint64_t permits = (uint64_t)len * tot / k;  // manager.rs:380-385, x (k+m)/k for the parity
        ram->acquire(permits);
        struct Permit {
            ByteSemaphore &s;
            uint64_t n;
            ~Permit() { s.release(n); }
        } permit{*ram, permits};
        put_calls++;
        // land the block in pinned memory (caller's thread, so copies of concurrent PUTs overlap)
        const auto t_in = Clock::now();
        SlotLease slot(put_slots);
        const auto t_slot = Clock::now();
        copy_for_dma(slot.p, data, len);  // landing copy: the GPU reads the slot next
        EncodeItem it;
        it.data = slot.p;
        it.len = (uint32_t)len;
        const auto t_sub = Clock::now();
        int rc = enc_batcher->submit(it);
        if (rc != GARAGE_EC_OK) return rc;
        const auto t_enc = Clock::now();
        struct PhaseNote {  // where a PUT's wall time goes (GARAGE_BM_TRACE prints the sums after a bench run)
            garage_bm &bm;
            Clock::time_point a, b, c, d;
            ~PhaseNote()
            {
                auto us = [](Clock::time_point x, Clock::time_point y) {
                    return (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(y - x).count();
                };
                bm.put_ns_slot += us(a, b);
                bm.put_ns_land += us(b, c);
                bm.put_ns_wait += us(c, d);
                bm.put_ns_store += us(d, Clock::now());
            }
        } note{*this, t_in, t_slot, t_sub, t_enc};
        struct BufRelease {
            EncBatchBuf *b;
            ~BufRelease() { b->done_one(); }
        } rel{it.buf};
        const size_t L = shard_len_of((uint32_t)len);
        std::vector<uint8_t> pad;
        int stored = 0;
        for (int i = 0; i < tot; i++) {  // try_write_many_sets (manager.rs:395-405): all at once
            const uint8_t *src;
            if (i < k) {
                const size_t off = (size_t)i * L;
                const size_t have = off < len ? std::min(L, len - off) : 0;
                if (have == L) {
                    src = slot.p + off;
                } else {  // zero padded tail shard (put.rs:611-615 short last block)
                    pad.assign(L, 0);
                    if (have) memcpy(pad.data(), slot.p + off, have);
                    src = pad.data();
                }
            } else {
                src = it.parity + (size_t)(i - k) * it.pstride;
            }
            // only a shard that is durably stored counts towards the quorum
            if (write_shard(who[i], h, i, (uint32_t)len, src, L, it.sums + (size_t)i * 32)) stored++;
        }
        {
            std::lock_guard<std::mutex> lk(refs_mu);
            refs[h] = (uint32_t)len;
        }
        const int quorum = garage_ec_write_quorum(k, m, GARAGE_CONSISTENT);  // k+1 capped at k+m (row f4, garage_placement.h)
        return stored >= quorum ? GARAGE_BM_OK : GARAGE_BM_E_QUORUM;
    }

    // manager.rs:344-363 + 276-339.  `out` must hold block_size bytes; *out_len = the block's length.
    int rpc_get_block(const Hash &h, uint8_t *out, size_t cap, size_t *out_len)
    {
        SlotLease slot(stripe_slots);
        uint8_t have[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M], want[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M] = {0};
        uint32_t block_len = 0;
        const int count = gather_into(h, -1, slot.p, have, block_len);
        if (count < k) return GARAGE_BM_E_MISSING_BLOCK;  // manager.rs:336-338
        *out_len = block_len;
        if (block_len > cap) return GARAGE_EC_E_INVALID;
        bool all_data = true;
        for (int j = 0; j < k; j++) {
            all_data &= have[j] != 0;
            want[j] = !have[j];
        }
        if (!all_data) {
            int rc = reconstruct_in_slot(slot.p, block_len, have, want);
            if (rc != GARAGE_BM_OK) return rc;
        }
        assemble(slot.p, block_len, out);
        if (content_ok(h, out, block_len)) return GARAGE_BM_OK;
        // Every shard passed its own tag, yet the block is not the one `h` names: some shard is
        // stale or was rebuilt wrongly.  Find it: gather everything, drop one shard at a time,
        // rebuild, re-check (manager.rs read path: CorruptData -> quarantine + resync).
        corrupt_data_errors++;
        const int avail = gather_into(h, -1, slot.p, have, block_len, /*all=*/true, /*for_gpu=*/true);
        if (avail > k && block_len <= cap) {
            int who[64];
            storage_nodes_of(h, who);
            SlotLease trial(stripe_slots);
            // First let the parity locate the wrong shards (up to floor((m - absent) / 2) of them, where the
            // search below finds one); a miscorrection cannot slip through, the content hash decides.
            {
                memcpy(trial.p, slot.p, (size_t)tot * slot_stride);
                int32_t st = 0;
                uint8_t fixed[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M] = {0};
                const uint32_t L = (uint32_t)shard_len_of(block_len);
                if (garage_ec_correct(ec, trial.p, have, &st, fixed, &L, slot_stride, 1, GARAGE_EC_MEM_HOST, nullptr) ==
                        GARAGE_EC_OK) {
                    assemble(trial.p, block_len, out);
                    if (content_ok(h, out, block_len)) {
                        for (int i = 0; i < tot; i++)
                            if (fixed[i]) quarantine(who[i], h);
                        *out_len = block_len;
                        return GARAGE_BM_OK;
                    }
                }
            }
            for (int x = 0; x < tot; x++) {
                if (!have[x]) continue;
                uint8_t h2[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M], w2[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M] = {0};
                memcpy(h2, have, tot);
                h2[x] = 0;
                bool need = false;
                for (int j = 0; j < k; j++) {
                    w2[j] = !h2[j];
                    need |= w2[j] != 0;
                }
                memcpy(trial.p, slot.p, (size_t)tot * slot_stride);
                if (need && reconstruct_in_slot(trial.p, block_len, h2, w2) != GARAGE_BM_OK) continue;
                assemble(trial.p, block_len, out);
                if (content_ok(h, out, block_len)) {
                    quarantine(who[x], h);  // the culprit
                    *out_len = block_len;
                    return GARAGE_BM_OK;
                }
            }
        }
        return GARAGE_BM_E_CORRUPT_DATA;
    }

    bool deletable_now(const Hash &h)  // refs_mu held.  rc.is_deletable() + BLOCK_GC_DELAY (rc.rs, manager.rs:49-52)
    {
        auto it = rc.find(h);
        if (it == rc.end() || it->second.count > 0) return false;
        return Clock::now() - it->second.zero_since >= std::chrono::milliseconds(cfg.block_gc_delay_ms);
    }

    int resync_block(int node, const Hash &h)
    {
        int who[64];
        storage_nodes_of(h, who);
        int idx = -1;
        for (int i = 0; i < tot; i++)
            if (who[i] == node) idx = i;
        if (idx < 0) return GARAGE_BM_OK;  // not a storage node for it any more (resync.rs:466-477)
        bool known, unneeded;
        {
            // the deletion decision and the deletion itself happen under BOTH locks (refs_mu, then the
            // node's): an incref / re-PUT cannot slip in between the check and the erase
            std::lock_guard<std::mutex> rl(refs_mu);
            known = refs.count(h) != 0;
            auto it = rc.find(h);
            unneeded = it != rc.end() && it->second.count <= 0;
            Node &nd = *nodes[node];
            std::lock_guard<std::mutex> lk(nd.mu);
            if (!nd.up) return GARAGE_BM_E_MESSAGE;
            const bool exists = nd.store_has(h);
            if (exists && unneeded) {  // offload branch, resync.rs:369-458: nobody needs it -> delete_if_unneeded
                if (!deletable_now(h)) {  // still inside the GC delay: look again later
                    if (nd.queued.insert(h).second) nd.resync_queue.push_back(h);
                    return GARAGE_BM_OK;
                }
                if (nd.store_erase(h)) delete_counter++;
                return GARAGE_BM_OK;
            }
            if (exists) return GARAGE_BM_OK;
        }
        if (!known || unneeded) return GARAGE_BM_OK;  // rc == 0: nothing to fetch
        SlotLease slot(stripe_slots);
        uint8_t have[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M], want[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M] = {0};
        uint32_t block_len = 0;
        const int count = gather_into(h, node, slot.p, have, block_len, false, /*for_gpu=*/true);
        if (count < k) {
            resync_error_counter++;
            return GARAGE_BM_E_MISSING_BLOCK;  // resync.rs:488-494
        }
        want[idx] = 1;
        int rc2 = reconstruct_in_slot(slot.p, block_len, have, want);
        if (rc2 != GARAGE_BM_OK) {
            resync_error_counter++;
            return rc2;
        }
        resync_recv_counter++;
        const size_t L = shard_len_of(block_len);
        const uint8_t *bytes = slot.p + (size_t)idx * slot_stride;
        Hash sum;
        shard_tag(bytes, L, sum);
        if (!write_shard(node, h, idx, block_len, bytes, L, sum.data())) {  // resync.rs:499
            resync_error_counter++;
            return GARAGE_BM_E_MESSAGE;  // Error::Io: stays queued, the caller backs off (resync.rs:300-315)
        }
        resync_counter++;
        return GARAGE_BM_OK;
    }

    // BlockManager::block_incref / block_decref (manager.rs:452-500), driven in Garage by
    // BlockRefTable::updated (src/model/s3/block_ref_table.rs:69-85): a 0 -> 1 transition queues a
    // resync on every storage node of the block (safety check that the shard really arrives), a
    // drop to 0 queues one too (so that the shard gets deleted once BLOCK_GC_DELAY has passed).
    void block_incref(const Hash &h)
    {
        bool first;
        {
            std::lock_guard<std::mutex> lk(refs_mu);
            RcEntry &c = rc[h];
            first = c.count <= 0;
            c.count = first ? 1 : c.count + 1;
        }
        if (first) queue_on_storage_nodes(h);
    }
    void block_decref(const Hash &h)
    {
        bool zero = false;
        {
            std::lock_guard<std::mutex> lk(refs_mu);
            auto it = rc.find(h);
            if (it == rc.end()) it = rc.emplace(h, RcEntry{1, {}}).first;  // an un-counted block counts as referenced once
            if (it->second.count > 0 && --it->second.count == 0) {
                it->second.zero_since = Clock::now();
                zero = true;
                refs.erase(h);
            }
        }
        if (zero) queue_on_storage_nodes(h);
    }
    void queue_on_storage_nodes(const Hash &h)
    {
        int who[64];
        storage_nodes_of(h, who);
        for (int i = 0; i < tot; i++) put_to_resync(who[i], h);
    }
    int64_t get_block_rc(const Hash &h)
    {
        std::lock_guard<std::mutex> lk(refs_mu);
        auto it = rc.find(h);
        return it == rc.end() ? -1 : it->second.count;
    }

    int resync_all(int node, int workers, uint64_t *resynced)
    {
        Node &nd = *nodes[node];
        std::vector<Hash> todo;
        {
            std::lock_guard<std::mutex> lk(nd.mu);
            todo.assign(nd.resync_queue.begin(), nd.resync_queue.end());
            nd.resync_queue.clear();
            nd.queued.clear();
        }
        std::atomic<size_t> next{0};
        std::atomic<uint64_t> ok{0};
        std::mutex failed_mu;
        std::vector<Hash> failed;
        workers = std::max(1, std::min(workers, 64));
        std::vector<std::thread> th;
        for (int w = 0; w < workers; w++)
            th.emplace_back([&] {
                garage_ec_bind_thread(ec);
                for (;;) {
                    const size_t i = next++;
                    if (i >= todo.size()) return;
                    int r;
                    try {
                        r = resync_block(node, todo[i]);
                    } catch (...) {
                        r = GARAGE_EC_E_NOMEM;
                    }
                    if (r == GARAGE_BM_OK) {
                        ok++;
                    } else {
                        std::lock_guard<std::mutex> lk(failed_mu);
                        failed.push_back(todo[i]);
                    }
                }
            });
        for (auto &t : th) t.join();
        for (const Hash &h : failed) put_to_resync(node, h);  // stays queued (backoff is the caller's)
        if (resynced) *resynced = ok.load();
        return (int)failed.size();
    }

    int repair_enqueue_missing(int node, uint64_t *enq)
    {
        std::vector<Hash> all;
        {
            std::lock_guard<std::mutex> lk(refs_mu);
            for (auto &kv : refs) all.push_back(kv.first);
        }
        uint64_t c = 0;
        for (const Hash &h : all) {
            int who[64];
            storage_nodes_of(h, who);
            bool mine = false;
            for (int i = 0; i < tot; i++) mine |= who[i] == node;
            if (!mine) continue;
            bool has;
            {
                std::lock_guard<std::mutex> lk(nodes[node]->mu);
                has = nodes[node]->store_has(h);
            }
            if (!has) {
                put_to_resync(node, h);
                c++;
            }
        }
        if (enq) *enq = c;
        return GARAGE_BM_OK;
    }

    // ScrubWorker sweep of one node (repair.rs:438-490) with the GPU computing the shard tags
    // `cursor`/`max_shards`: the scrub iterator checkpoint of the reference (ScrubWorker persists
    // its BlockStoreIterator position every 60 s, repair.rs:186-193,460-464, so a sweep survives a
    // restart): shards are visited in hash order, starting after *cursor (NULL = from the start),
    // at most max_shards of them (0 = all); *cursor_out receives the last hash visited and
    // *finished whether the end of the store was reached.
    int scrub(int node, uint64_t *checked, uint64_t *corrupt, const Hash *cursor = nullptr, size_t max_shards = 0,
              Hash *cursor_out = nullptr, int *finished = nullptr)
    {
        std::lock_guard<std::mutex> sl(scrub_mu);
        Node &nd = *nodes[node];
        std::vector<Hash> hashes;
        {
            std::lock_guard<std::mutex> lk(nd.mu);
            if (!nd.up) return GARAGE_BM_E_MESSAGE;
            nd.store_list(hashes);
        }
        std::sort(hashes.begin(), hashes.end());
        if (cursor) hashes.erase(hashes.begin(), std::upper_bound(hashes.begin(), hashes.end(), *cursor));
        bool done = true;
        if (max_shards && hashes.size() > max_shards) {
            hashes.resize(max_shards);
            done = false;
        }
        if (finished) *finished = done ? 1 : 0;
        if (cursor_out) {
            if (!hashes.empty()) *cursor_out = hashes.back();
            else if (cursor) *cursor_out = *cursor;
            else cursor_out->fill(0);
        }
        uint64_t nchecked = 0, nbad = 0;
        const size_t chunk = std::max<size_t>(1, (size_t)cfg.batch_max_blocks * tot);
        const size_t stride = slot_stride;
        for (size_t c0 = 0; c0 < hashes.size(); c0 += chunk) {
            const size_t n = std::min(chunk, hashes.size() - c0);
            uint8_t *buf = scrub_buf.get(n * stride + n * 32 + n + n * 4);
            if (!buf) return GARAGE_EC_E_NOMEM;
            uint8_t *expect = buf + n * stride, *bad = expect + n * 32;
            std::vector<uint32_t> lens(n, 0);
            std::vector<uint8_t> state(n, 0);  // 0 gone, 1 to be checked on the GPU, 2 corrupt already, 3 checked on the CPU
            {
                std::lock_guard<std::mutex> lk(nd.mu);
                for (size_t i = 0; i < n; i++) {
                    ShardMeta mt;
                    memset(expect + i * 32, 0, 32);
                    const ReadResult r = nd.store_read_into(hashes[c0 + i], buf + i * stride, stride, mt);
                    if (r == kReadMissing) continue;
                    if (r == kReadInvalid) {
                        state[i] = 2;
                        continue;
                    }
                    lens[i] = mt.shard_len;
                    bytes_read += mt.shard_len;
                    if (mt.sum_kind == sum_kind) {
                        memcpy(expect + i * 32, mt.sum.data(), 32);
                        state[i] = 1;
                    } else {  // written under another tag kind: check it on the CPU
                        Hash got;
                        garage_ec_shard_sum_host(mt.sum_kind, buf + i * stride, mt.shard_len, got.data());
                        state[i] = got == mt.sum ? 3 : 2;
                        lens[i] = 0;
                    }
                }
            }
            int rc = garage_ec_check_sums(ec, buf, expect, lens.data(), stride, n, 1, bad, GARAGE_EC_MEM_HOST, nullptr);
            if (rc != GARAGE_EC_OK) return rc;
            for (size_t i = 0; i < n; i++) {
                if (!state[i]) continue;
                nchecked++;
                if (state[i] == 3 || (state[i] == 1 && !bad[i])) continue;
                nbad++;
                quarantine(node, hashes[c0 + i]);
            }
        }
        scrub_checked += nchecked;
        scrub_corrupt += nbad;
        if (checked) *checked = nchecked;
        if (corrupt) *corrupt = nbad;
        return GARAGE_BM_OK;
    }

    // ---- native closed-loop load generator (tools/bm_bench.py drives it): `threads` client threads,
    // each PUTs (mode 0) or GETs (mode 1) `per_thread` blocks of `block_len` bytes.  Blocks are the
    // splitmix64 stream (seed, thread, i); hashing them is the S3 layer's job (put.rs:448) and
    // happens before the clock starts.
    int bench(int threads, int per_thread, uint32_t block_len, int mode, uint64_t seed, double *gib_per_s, uint64_t *errors)
    {
        if (threads < 1 || per_thread < 1 || block_len < 1 || shard_len_of(block_len) > slot_stride) return GARAGE_EC_E_INVALID;
        const size_t nb = (size_t)threads * per_thread;
        std::vector<uint8_t> data;
        std::vector<Hash> hashes(nb);
        const size_t words = ((size_t)block_len + 7) / 8;
        if (mode == 0) data.resize(nb * words * 8);
        auto gen = [&](size_t b, uint8_t *dst) {
            uint64_t *w = reinterpret_cast<uint64_t *>(dst);
            for (size_t i = 0; i < words; i++) {
                uint64_t z = seed + (b * words + i + 1) * 0x9E3779B97F4A7C15ull;
                z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
                z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
                w[i] = z ^ (z >> 31);
            }
        };
        {
            std::vector<std::thread> th;
            for (int t = 0; t < threads; t++)
                th.emplace_back([&, t] {
                    std::vector<uint8_t> tmp(words * 8);
                    for (int i = 0; i < per_thread; i++) {
                        const size_t b = (size_t)t * per_thread + i;
                        uint8_t *dst = mode == 0 ? data.data() + b * words * 8 : tmp.data();
                        gen(b, dst);
                        garage_ec_blake2sum(dst, block_len, hashes[b].data());
                    }
                });
            for (auto &x : th) x.join();
        }
        if (mode == 0 && !warmed.exchange(true)) {
            // first use of this manager: one block through every dispatcher (streams, lane buffers, kernels)
            std::vector<uint8_t> wblk(words * 8);
            gen(nb, wblk.data());
            Hash wh;
            garage_ec_blake2sum(wblk.data(), block_len, wh.data());
            std::vector<std::thread> wt;
            for (int t = 0; t < 3 * kWorkers; t++)
                wt.emplace_back([&] {
                    try {
                        rpc_put_block(wh, wblk.data(), block_len);
                    } catch (...) {
                    }
                });
            for (auto &x : wt) x.join();
        }
        if (mode == 0 && nodes[0]->dir.empty())  // the stores' memory is in place before the clock starts (see ShardArena)
            ShardArena::instance().reserve(shard_len_of(block_len), nb * (size_t)tot);
        std::atomic<uint64_t> errs{0};
        std::atomic<int> ready{0};
        std::atomic<bool> go{false};
        std::vector<std::thread> th;
        for (int t = 0; t < threads; t++)
            th.emplace_back([&, t] {
                garage_ec_bind_thread(ec);
                std::vector<uint8_t> out(mode == 1 ? block_len : 0);
                ready++;
                while (!go.load(std::memory_order_acquire)) std::this_thread::yield();
                for (int i = 0; i < per_thread; i++) {
                    const size_t b = (size_t)t * per_thread + i;
                    int rc;
                    try {
                        if (mode == 0) {
                            rc = rpc_put_block(hashes[b], data.data() + b * words * 8, block_len);
                        } else {
                            size_t n = 0;
                            rc = rpc_get_block(hashes[b], out.data(), out.size(), &n);
                            if (rc == GARAGE_BM_OK && n != block_len) rc = GARAGE_BM_E_CORRUPT_DATA;
                        }
                    } catch (...) {
                        rc = GARAGE_EC_E_NOMEM;
                    }
                    if (rc != GARAGE_BM_OK) errs++;
                }
            });
        while (ready.load() < threads) std::this_thread::yield();
        const auto t0 = Clock::now();
        go.store(true, std::memory_order_release);
        for (auto &x : th) x.join();
        const double el = std::chrono::duration<double>(Clock::now() - t0).count();
        if (mode == 0 && getenv("GARAGE_BM_TRACE"))
            fprintf(stderr, "[garage_bm] PUT x%zu, %d threads, %.3f s: per block ms  slot-wait %.3f  landing copy %.3f  batch+GPU %.3f  "
                            "store %d shards %.3f\n", nb, threads, el, put_ns_slot.exchange(0) / 1e6 / nb, put_ns_land.exchange(0) / 1e6 / nb,
                    put_ns_wait.exchange(0) / 1e6 / nb, tot, put_ns_store.exchange(0) / 1e6 / nb);
        if (gib_per_s) *gib_per_s = (double)nb * block_len / el / (double)(1ull << 30);
        if (errors) *errors = errs.load();
        return GARAGE_BM_OK;
    }
};

// ================================================================= C API
// Nothing throws across the C boundary (the reference returns Result everywhere,
// src/util/error.rs:14-82): allocation failures and anything unexpected become status codes.
#define BM_GUARD(expr)                       \
    try {                                    \
        return (expr);                       \
    } catch (const std::bad_alloc &) {       \
        return GARAGE_EC_E_NOMEM;            \
    } catch (...) {                          \
        return GARAGE_BM_E_MESSAGE;          \
    }

extern "C" {

void garage_bm_default_config(garage_bm_config *c)
{
    if (!c) return;
    c->data_shards = 10;
    c->parity_shards = 4;
    c->cuda_device = 0;
    c->n_nodes = 14;
    c->block_size = 1u << 20;               // util/config.rs:273-275
    c->block_ram_buffer_max = 256ull << 20;  // util/config.rs:276-278
    c->batch_max_blocks = 64;
    c->batch_linger_us = 100;  // 300 us cost 30 % of the closed-loop PUT rate at 32 callers (r02_summary.md)
    c->data_dir = nullptr;
    c->shard_sum_kind = GARAGE_EC_SUM_ADLER8;
    c->verify_content_hash = 1;
    c->data_fsync = 0;             // util/config.rs data_fsync default
    c->block_gc_delay_ms = 600000;  // BLOCK_GC_DELAY, manager.rs:49-52
}

static int bm_create(garage_bm **out, const garage_bm_config *cfg)
{
    *out = nullptr;
    const int k = cfg->data_shards, m = cfg->parity_shards;
    if (k < 1 || m < 1 || k > GARAGE_EC_MAX_K || m > GARAGE_EC_MAX_M || cfg->n_nodes < k + m || cfg->n_nodes > 256)
        return GARAGE_EC_E_INVALID;
    if (cfg->shard_sum_kind != GARAGE_EC_SUM_BLAKE2 && cfg->shard_sum_kind != GARAGE_EC_SUM_ADLER8) return GARAGE_EC_E_INVALID;
    std::unique_ptr<garage_bm> bm(new garage_bm());
    bm->cfg = *cfg;
    if (!bm->cfg.block_size) bm->cfg.block_size = 1u << 20;
    bm->k = k;
    bm->m = m;
    bm->tot = k + m;
    bm->sum_kind = cfg->shard_sum_kind;
    bm->slot_stride = garage_ec_stride_for(garage_ec_shard_len(bm->cfg.block_size, k));
    int rc = garage_ec_create(&bm->ec, cfg->cuda_device, k, m, GARAGE_EC_VANDERMONDE);
    if (rc != GARAGE_EC_OK) return rc;  // no GPU => no block manager: there is no CPU fallback
    garage_ec_set_sum_kind(bm->ec, bm->sum_kind);
    if (cfg->n_nodes <= GARAGE_LAYOUT_MAX_NODES) {
        const int n = cfg->n_nodes, tot = k + m;
        std::vector<uint8_t> ring((size_t)GARAGE_NB_PARTITIONS * tot);
        for (int p = 0; p < GARAGE_NB_PARTITIONS; p++)
            for (int i = 0; i < tot; i++) ring[(size_t)p * tot + i] = (uint8_t)((p % n + i) % n);
        std::vector<int32_t> zone(n, 0);
        std::vector<uint64_t> capacity(n, 1);
        if (garage_layout_from_ring(&bm->layout, 1, n, zone.data(), capacity.data(), tot, ring.data()) != GARAGE_LAYOUT_OK)
            bm->layout = nullptr;
    }
    for (int i = 0; i < cfg->n_nodes; i++) {
        bm->nodes.emplace_back(new Node());
        Node &nd = *bm->nodes.back();
        nd.k = k;
        nd.m = m;
        nd.fsync_data = cfg->data_fsync != 0;
        if (cfg->data_dir && cfg->data_dir[0]) {
            nd.dir = std::string(cfg->data_dir) + "/node" + std::to_string(i);
            std::error_code ec;
            std::filesystem::create_directories(nd.dir, ec);
            // restart: what is on disk is what exists (the block_ref table would say the same)
            std::vector<Hash> have;
            nd.store_list(have);
            std::vector<uint8_t> tmp(bm->slot_stride);
            for (const Hash &h : have) {
                ShardMeta mt;
                if (nd.store_read_into(h, tmp.data(), tmp.size(), mt) == kReadOk) bm->refs[h] = mt.block_len;
            }
        }
    }
    bm->ram.reset(new ByteSemaphore(cfg->block_ram_buffer_max ? cfg->block_ram_buffer_max : (256ull << 20)));
    bm->scrub_buf.ctx = bm->ec;
    auto destroy_on_error = [&](int code) {
        garage_bm_destroy(bm.release());
        return code;
    };
    for (int w = 0; w < garage_bm::kWorkers; w++) {
        rc = garage_ec_create(&bm->enc_ctx[w], cfg->cuda_device, k, m, GARAGE_EC_VANDERMONDE);
        if (rc == GARAGE_EC_OK) rc = garage_ec_create(&bm->rec_ctx[w], cfg->cuda_device, k, m, GARAGE_EC_VANDERMONDE);
        if (rc != GARAGE_EC_OK) return destroy_on_error(rc);
        garage_ec_set_sum_kind(bm->enc_ctx[w], bm->sum_kind);
        garage_ec_set_sum_kind(bm->rec_ctx[w], bm->sum_kind);
        // Dispatchers wait for their batch spinning in the driver (default) or sleeping on an event
        // (GARAGE_BM_SLEEP_WAIT=1).  Measured on a 16-CPU box, 32 client threads: 20.0 GiB/s PUT spinning, 16.9
        // sleeping -- the wake-up latency costs more than the three CPUs (profiles/r02_summary.md).
        const int sleep_wait = getenv("GARAGE_BM_SLEEP_WAIT") ? 1 : 0;
        garage_ec_set_wait_mode(bm->enc_ctx[w], sleep_wait);
        garage_ec_set_wait_mode(bm->rec_ctx[w], sleep_wait);
        for (auto &eb : bm->enc_out[w]) eb.ctx = bm->enc_ctx[w];
        // the pinned parity buffers at their final size now, not on the first large batch
        const size_t out_bytes = (size_t)std::max<uint32_t>(cfg->batch_max_blocks, 1) * ((size_t)m * bm->slot_stride + (size_t)(k + m) * 32);
        for (auto &eb : bm->enc_out[w])
            if (!eb.get(out_bytes)) return destroy_on_error(GARAGE_EC_E_NOMEM);
    }
    const size_t nslots = (size_t)std::max<uint32_t>(cfg->batch_max_blocks, 1) * (garage_bm::kWorkers + 1);
    if (!bm->put_slots.init(bm->ec, nslots, bm->cfg.block_size)) return destroy_on_error(GARAGE_EC_E_NOMEM);
    if (!bm->stripe_slots.init(bm->ec, nslots, (size_t)bm->tot * bm->slot_stride)) return destroy_on_error(GARAGE_EC_E_NOMEM);
    // Warm every dispatcher's context now: streams, lane buffers, and the first launch of each kernel (CUDA
    // loads kernels lazily) cost tens of milliseconds that would otherwise land on the first real batches.
    {
        SlotLease blk(bm->put_slots), stripe(bm->stripe_slots);
        const uint32_t wlen = bm->cfg.block_size;
        memset(blk.p, 0x5a, wlen);
        memset(stripe.p, 0, (size_t)bm->tot * bm->slot_stride);
        for (int w = 0; w < garage_bm::kWorkers; w++) {
            const uint8_t *ptrs[1] = {blk.p};
            uint8_t *par = bm->enc_out[w][0].get(1);
            rc = garage_ec_encode_blocks_with_sums(bm->enc_ctx[w], ptrs, &wlen, 1, par, par + (size_t)m * bm->slot_stride, bm->slot_stride);
            if (rc != GARAGE_EC_OK) return destroy_on_error(rc);
            uint8_t present[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M], want[GARAGE_EC_MAX_K + GARAGE_EC_MAX_M] = {0};
            memset(present, 1, sizeof(present));
            present[0] = 0;
            want[0] = 1;
            uint8_t *stripes[1] = {stripe.p};
            const uint32_t slen = (uint32_t)bm->shard_len_of(wlen);
            int32_t st = 0;
            rc = garage_ec_reconstruct_stripes(bm->rec_ctx[w], stripes, present, want, &st, &slen, bm->slot_stride, 1);
            if (rc != GARAGE_EC_OK) return destroy_on_error(rc);
        }
        uint8_t bad1 = 0, exp1[32] = {0};
        const uint32_t slen = (uint32_t)bm->shard_len_of(wlen);
        rc = garage_ec_check_sums(bm->ec, stripe.p, exp1, &slen, bm->slot_stride, 1, 1, &bad1, GARAGE_EC_MEM_HOST, nullptr);
        if (rc != GARAGE_EC_OK) return destroy_on_error(rc);
    }
    garage_bm *raw = bm.get();
    auto bind = [raw] { garage_ec_bind_thread(raw->ec); };
    bm->enc_batcher.reset(new Batcher<EncodeItem>(cfg->batch_max_blocks, cfg->batch_linger_us, garage_bm::kWorkers,
                                                  [raw](int w, std::vector<EncodeItem *> &b) { raw->run_encode(w, b); }, bind));
    bm->rec_batcher.reset(new Batcher<ReconItem>(cfg->batch_max_blocks, cfg->batch_linger_us, garage_bm::kWorkers,
                                                 [raw](int w, std::vector<ReconItem *> &b) { raw->run_reconstruct(w, b); }, bind));
    *out = bm.release();
    return GARAGE_BM_OK;
}

int garage_bm_create(garage_bm **out, const garage_bm_config *cfg)
{
    if (!out || !cfg) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm_create(out, cfg));
}

void garage_bm_destroy(garage_bm *bm)
{
    if (!bm) return;
    bm->enc_batcher.reset();
    bm->rec_batcher.reset();
    garage_ec_ctx *ec = bm->ec;
    garage_ec_ctx *ctxs[2 * garage_bm::kWorkers];
    for (int w = 0; w < garage_bm::kWorkers; w++) {
        for (auto &eb : bm->enc_out[w]) eb.release();  // pinned buffers go before their context
        ctxs[2 * w] = bm->enc_ctx[w];
        ctxs[2 * w + 1] = bm->rec_ctx[w];
    }
    bm->scrub_buf.release();
    bm->put_slots.destroy();
    bm->stripe_slots.destroy();
    delete bm;
    for (garage_ec_ctx *c : ctxs)
        if (c) garage_ec_destroy(c);
    if (ec) garage_ec_destroy(ec);
}

void garage_bm_blake2sum(const uint8_t *data, size_t len, uint8_t hash_out[32]) { garage_ec_blake2sum(data, len, hash_out); }

int garage_bm_rpc_put_block(garage_bm *bm, const uint8_t hash[32], const uint8_t *data, size_t len)
{
    if (!bm || !hash || !data) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm->rpc_put_block(to_hash(hash), data, len));
}

int garage_bm_rpc_get_block(garage_bm *bm, const uint8_t hash[32], uint8_t *out, size_t cap, size_t *out_len)
{
    if (!bm || !hash || !out_len || !out) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm->rpc_get_block(to_hash(hash), out, cap, out_len));
}

int garage_bm_resync_block(garage_bm *bm, int node, const uint8_t hash[32])
{
    if (!bm || !hash || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm->resync_block(node, to_hash(hash)));
}

int garage_bm_block_incref(garage_bm *bm, const uint8_t hash[32])
{
    if (!bm || !hash) return GARAGE_EC_E_INVALID;
    BM_GUARD((bm->block_incref(to_hash(hash)), GARAGE_BM_OK));
}

int garage_bm_block_decref(garage_bm *bm, const uint8_t hash[32])
{
    if (!bm || !hash) return GARAGE_EC_E_INVALID;
    BM_GUARD((bm->block_decref(to_hash(hash)), GARAGE_BM_OK));
}

long long garage_bm_get_block_rc(garage_bm *bm, const uint8_t hash[32])
{
    if (!bm || !hash) return -1;
    BM_GUARD((long long)bm->get_block_rc(to_hash(hash)));
}

int garage_bm_resync_all(garage_bm *bm, int node, int workers, uint64_t *resynced)
{
    if (!bm || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm->resync_all(node, workers, resynced));
}

int garage_bm_repair_enqueue_missing(garage_bm *bm, int node, uint64_t *enqueued)
{
    if (!bm || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm->repair_enqueue_missing(node, enqueued));
}

int garage_bm_scrub(garage_bm *bm, int node, uint64_t *checked, uint64_t *corrupt)
{
    if (!bm || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm->scrub(node, checked, corrupt));
}

int garage_bm_scrub_step(garage_bm *bm, int node, const uint8_t *cursor32, size_t max_shards, uint8_t cursor_out32[32],
                         int *finished, uint64_t *checked, uint64_t *corrupt)
{
    if (!bm || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    try {
        Hash cur, out;
        if (cursor32) cur = to_hash(cursor32);
        int rc = bm->scrub(node, checked, corrupt, cursor32 ? &cur : nullptr, max_shards, &out, finished);
        if (rc == GARAGE_BM_OK && cursor_out32) memcpy(cursor_out32, out.data(), 32);
        return rc;
    } catch (const std::bad_alloc &) {
        return GARAGE_EC_E_NOMEM;
    } catch (...) {
        return GARAGE_BM_E_MESSAGE;
    }
}

int garage_bm_bench(garage_bm *bm, int threads, int blocks_per_thread, uint32_t block_len, int mode, uint64_t seed,
                    double *gib_per_s, uint64_t *errors)
{
    if (!bm || (mode != 0 && mode != 1)) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm->bench(threads, blocks_per_thread, block_len, mode, seed, gib_per_s, errors));
}

int garage_bm_set_node_up(garage_bm *bm, int node, int up)
{
    if (!bm || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    std::lock_guard<std::mutex> lk(bm->nodes[node]->mu);
    bm->nodes[node]->up = up != 0;
    return GARAGE_BM_OK;
}

// fault injection: what = 0 flips a bit of the shard's bytes at byte_off, 1 rewrites the stored
// block_len (+1), 2 rewrites the stored index (+1 mod k+m); the stored tag / header check are left
// alone in every case -- that is the corruption.
static int bm_corrupt(garage_bm *bm, int node, const uint8_t hash[32], size_t byte_off, int what)
{
    Node &nd = *bm->nodes[node];
    std::lock_guard<std::mutex> lk(nd.mu);
    const Hash h = to_hash(hash);
    if (nd.dir.empty()) {
        auto it = nd.shards.find(h);
        if (it == nd.shards.end()) return GARAGE_BM_E_MISSING_BLOCK;
        auto mod = std::make_shared<StoredShard>(*it->second);  // stored shards are immutable: replace by a damaged copy
        if (what == 0) {
            if (mod->bytes.empty()) return GARAGE_BM_E_MISSING_BLOCK;
            mod->bytes[byte_off % mod->bytes.size()] ^= 0x01;
        } else if (what == 1) {
            mod->block_len += 1;
        } else {
            mod->index = (mod->index + 1) % (bm->tot);
        }
        it->second = std::move(mod);
        return GARAGE_BM_OK;
    }
    FILE *f = fopen(nd.path_of(h, ".shard").c_str(), "r+b");
    if (!f) return GARAGE_BM_E_MISSING_BLOCK;
    ShardFileHeader hd;
    int rc = GARAGE_BM_E_MISSING_BLOCK;
    if (fread(&hd, sizeof(hd), 1, f) == 1) {
        long off = -1;
        uint8_t b = 0;
        if (what == 0 && hd.shard_len) off = (long)sizeof(hd) + (long)(byte_off % hd.shard_len);
        else if (what == 1) off = offsetof(ShardFileHeader, block_len);
        else if (what == 2) off = offsetof(ShardFileHeader, index);
        if (off >= 0 && fseek(f, off, SEEK_SET) == 0 && fread(&b, 1, 1, f) == 1) {
            b = what == 0 ? (uint8_t)(b ^ 1) : (uint8_t)(b + 1);
            if (fseek(f, off, SEEK_SET) == 0 && fwrite(&b, 1, 1, f) == 1) rc = GARAGE_BM_OK;
        }
    }
    fclose(f);
    return rc;
}

int garage_bm_corrupt_shard(garage_bm *bm, int node, const uint8_t hash[32], size_t byte_off)
{
    if (!bm || !hash || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm_corrupt(bm, node, hash, byte_off, 0));
}

int garage_bm_corrupt_shard_header(garage_bm *bm, int node, const uint8_t hash[32], int what)
{
    if (!bm || !hash || node < 0 || node >= (int)bm->nodes.size() || (what != 1 && what != 2)) return GARAGE_EC_E_INVALID;
    BM_GUARD(bm_corrupt(bm, node, hash, 0, what));
}

// replace the shard stored on `node` with a VALID shard (correct tag, correct index) of other
// content -- the "stale shard / wrong shard written by an earlier bad resync" case that only the
// whole-block content hash can catch
int garage_bm_plant_stale_shard(garage_bm *bm, int node, const uint8_t hash[32])
{
    if (!bm || !hash || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    try {
        Node &nd = *bm->nodes[node];
        std::lock_guard<std::mutex> lk(nd.mu);
        StoredShard sh;
        const Hash h = to_hash(hash);
        if (!nd.store_get(h, sh) || sh.bytes.empty()) return GARAGE_BM_E_MISSING_BLOCK;
        for (size_t i = 0; i < sh.bytes.size(); i += 97) sh.bytes[i] ^= 0x5a;
        garage_ec_shard_sum_host(sh.sum_kind, sh.bytes.data(), sh.bytes.size(), sh.sum.data());
        return nd.store_put(h, sh, sh.bytes.data(), sh.bytes.size()) ? GARAGE_BM_OK : GARAGE_BM_E_MESSAGE;
    } catch (...) {
        return GARAGE_EC_E_NOMEM;
    }
}

int garage_bm_set_node_readonly(garage_bm *bm, int node, int readonly)
{
    if (!bm || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    Node &nd = *bm->nodes[node];
    std::lock_guard<std::mutex> lk(nd.mu);
    if (nd.dir.empty()) return GARAGE_BM_E_MESSAGE;  // only meaningful for the file store
    // works for root too (which ignores permission bits): the directory is moved aside and a plain
    // FILE takes its name, so every create / open below it fails with ENOTDIR
    const std::string saved = nd.dir + ".moved_aside";
    if (readonly) {
        if (::rename(nd.dir.c_str(), saved.c_str()) != 0) return GARAGE_BM_E_MESSAGE;
        FILE *f = fopen(nd.dir.c_str(), "wb");
        if (f) fclose(f);
        return f ? GARAGE_BM_OK : GARAGE_BM_E_MESSAGE;
    }
    ::remove(nd.dir.c_str());
    return ::rename(saved.c_str(), nd.dir.c_str()) == 0 ? GARAGE_BM_OK : GARAGE_BM_E_MESSAGE;
}

int garage_bm_drop_shard(garage_bm *bm, int node, const uint8_t hash[32])
{
    if (!bm || !hash || node < 0 || node >= (int)bm->nodes.size()) return GARAGE_EC_E_INVALID;
    Node &nd = *bm->nodes[node];
    std::lock_guard<std::mutex> lk(nd.mu);
    if (nd.store_erase(to_hash(hash))) {
        bm->delete_counter++;
        return GARAGE_BM_OK;
    }
    return GARAGE_BM_E_MISSING_BLOCK;
}

int garage_bm_node_shard_index(garage_bm *bm, int node, const uint8_t hash[32])
{
    if (!bm || !hash || node < 0 || node >= (int)bm->nodes.size()) return -1;
    try {
        Node &nd = *bm->nodes[node];
        std::lock_guard<std::mutex> lk(nd.mu);
        StoredShard sh;
        return nd.store_get(to_hash(hash), sh) ? sh.index : -1;
    } catch (...) {
        return -1;
    }
}

int garage_bm_storage_nodes_of(garage_bm *bm, const uint8_t hash[32], int *nodes_out)
{
    if (!bm || !hash || !nodes_out) return GARAGE_EC_E_INVALID;
    bm->storage_nodes_of(to_hash(hash), nodes_out);
    return GARAGE_BM_OK;
}

void garage_bm_get_metrics(garage_bm *bm, garage_bm_metrics *o)
{
    if (!bm || !o) return;
    memset(o, 0, sizeof(*o));
    o->bytes_written = bm->bytes_written;
    o->bytes_read = bm->bytes_read;
    o->corruption_counter = bm->corruption_counter;
    o->resync_counter = bm->resync_counter;
    o->resync_error_counter = bm->resync_error_counter;
    o->resync_recv_counter = bm->resync_recv_counter;
    o->delete_counter = bm->delete_counter;
    o->put_calls = bm->put_calls;
    o->put_batches = bm->enc_batcher ? bm->enc_batcher->batches() : 0;
    o->reconstruct_calls = bm->reconstruct_calls;
    o->reconstruct_batches = bm->rec_batcher ? bm->rec_batcher->batches() : 0;
    o->scrub_shards_checked = bm->scrub_checked;
    o->scrub_corruptions = bm->scrub_corrupt;
    o->encode_call_us = bm->enc_gpu_us;
    o->reconstruct_call_us = bm->rec_gpu_us;
    o->corrupt_data_errors = bm->corrupt_data_errors;
    o->write_errors = bm->write_errors;
    uint64_t ql = 0;
    for (auto &n : bm->nodes) {
        std::lock_guard<std::mutex> lk(n->mu);
        ql += n->resync_queue.size();
    }
    o->resync_queue_length = ql;
}

}  // extern "C"
