// rawfile.cpp — raw-file streaming around the chain (SURVEY.md 8(f) rank 2): the step either side of the
// hot path for file inputs.  Replaces the reference's Reader -> ... -> Writer plumbing for raw files
// (src/input_rawfile.c:188-249: one sf_read_raw of a 16384-frame chunk per loop, src/output_raw_file.c:
// 146-184: 1 MB fwrites out of a ring buffer) with three overlapped stages on pinned memory:
//
//   reader thread   large sequential reads of whole chunk trains into a ring of pinned input buffers
//   caller thread   one chain call per train (H2D / kernels / D2H pipelined inside the chain): iqgpu_chain_process, or
//                   iqgpu_chain_process_multi when several channels share the input (one H2D for all of them)
//   writer thread   one fwrite per train and channel out of a ring of pinned output buffers (K buffers per slot)
//
// Chunk semantics are the reference's: the file is cut into 16384-frame chunks, a short read makes a short
// last chunk, trailing bytes that do not fill a frame are dropped (input_rawfile.c:236), and nothing is
// flushed at end of stream (SURVEY quirk B1).  Only the C ABI of include/iqgpu.h is used.
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/iqgpu.h"
#include "stream_io.hpp"

namespace {

struct Slot {
    std::vector<void*> buf;     // one buffer per channel (the input ring has one)
    std::vector<size_t> bytes;  // valid bytes
    bool last = false;
};

// single-producer single-consumer ring of pinned buffers
struct Ring {
    std::vector<Slot> slots;
    size_t head = 0, tail = 0, count = 0;
    std::mutex mu;
    std::condition_variable cv;
    bool aborted = false;

    Slot* acquire_free()        // producer: next slot to fill (blocks while the ring is full)
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return count < slots.size() || aborted; });
        return aborted ? nullptr : &slots[head];
    }
    void publish()
    {
        std::lock_guard<std::mutex> lk(mu);
        head = (head + 1) % slots.size();
        count++;
        cv.notify_all();
    }
    Slot* acquire_full()        // consumer: oldest filled slot (blocks while the ring is empty)
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return count > 0 || aborted; });
        return (count > 0) ? &slots[tail] : nullptr;
    }
    void release()
    {
        std::lock_guard<std::mutex> lk(mu);
        tail = (tail + 1) % slots.size();
        count--;
        cv.notify_all();
    }
    void abort()
    {
        std::lock_guard<std::mutex> lk(mu);
        aborted = true;
        cv.notify_all();
    }
};

thread_local std::string g_io_err;

}  // namespace

void iqio::set_last_error(const std::string& msg) { g_io_err = msg; }

std::string iqio::channel_prefix(size_t k, size_t n) { return n == 1 ? std::string() : "channel " + std::to_string(k) + ": "; }

int iqio::process_one(iqgpu_chain* const* chains, size_t n_chains, const void* raw_in, size_t n_frames, const uint32_t* chunk_frames,
                      size_t n_chunks, void* const* out, const size_t* out_capacity_bytes, size_t* out_frames,
                      uint32_t* const* per_chunk_out)
{
    if (n_chains != 1) { g_io_err = "one chain expected"; return IQGPU_EINVAL; }
    return iqgpu_chain_process(chains[0], raw_in, n_frames, chunk_frames, n_chunks, out[0], out_capacity_bytes[0], out_frames,
                               per_chunk_out ? per_chunk_out[0] : nullptr);
}

int iqio::Channels::open(const iqgpu_chain_config* cfgs, size_t n, int device, const char* const* out_paths, const char* open_error,
                         std::string& err)
{
    for (size_t k = 0; k < n; k++) {
        iqgpu_chain* c = nullptr;
        const int rc = iqgpu_chain_create(&cfgs[k], device, &c);
        if (rc) { err = channel_prefix(k, n) + iqgpu_last_error(); close(err); return rc; }
        chains.push_back(c);
    }
    if (n > 1) {
        // the refusals of the chain call (different input formats or rates, ...) before any output is created
        std::vector<void*> no_out(n, nullptr);
        std::vector<size_t> no_cap(n, 0), no_frames(n, 0);
        const int rc = process(chains.data(), n, nullptr, 0, nullptr, 0, no_out.data(), no_cap.data(), no_frames.data(), nullptr);
        if (rc) { err = iqgpu_last_error(); close(err); return rc; }
    }
    for (size_t k = 0; k < n; k++) {
        FILE* f = fopen(out_paths[k], "wb");
        if (!f) {
            err = std::string(open_error) + out_paths[k];
            std::string ignored;
            close(ignored);
            for (auto& p : paths) remove(p.c_str());      // nothing is written when one output cannot be
            paths.clear();
            return IQGPU_EINVAL;
        }
        fouts.push_back(f);
        paths.push_back(out_paths[k]);
    }
    return IQGPU_OK;
}

int iqio::Channels::close(std::string& err)
{
    int rc = IQGPU_OK;
    for (FILE* f : fouts)
        if (fclose(f) != 0 && !rc) { rc = IQGPU_EINVAL; err = "write error on the output file"; }
    fouts.clear();
    for (iqgpu_chain* c : chains) iqgpu_chain_destroy(c);
    chains.clear();
    return rc;
}

iqio::Channels::~Channels()
{
    std::string ignored;
    close(ignored);
}

int iqio::rawfile_run(const iqgpu_chain_config* cfgs, size_t n, int device, const char* in_path, const char* const* out_paths,
                      size_t train_chunks, iqgpu_rawfile_stats* stats, ProcessFn process)
{
    if (!cfgs || !in_path || !out_paths) { g_io_err = "null argument"; return IQGPU_EINVAL; }
    if (n == 0) { g_io_err = "n_channels must be at least 1"; return IQGPU_EINVAL; }
    if (stats) memset(stats, 0, n * sizeof(*stats));
    for (size_t k = 0; k < n; k++) {
        if (!out_paths[k]) { g_io_err = channel_prefix(k, n) + "null argument"; return IQGPU_EINVAL; }
        if (!iqgpu_get_bytes_per_sample(cfgs[k].input_format) || !iqgpu_get_bytes_per_sample(cfgs[k].output_format)) {
            g_io_err = channel_prefix(k, n) + "unhandled sample format";
            return IQGPU_EINVAL;
        }
    }
    FILE* fin = fopen(in_path, "rb");
    if (!fin) { g_io_err = std::string("cannot open input file ") + in_path; return IQGPU_EINVAL; }
    Channels ch;
    ch.process = process;
    std::string err;
    int rc = ch.open(cfgs, n, device, out_paths, "cannot open output file ", err);
    if (rc) { fclose(fin); g_io_err = err; return rc; }
    rc = run_stream(ch, cfgs, fin, UINT64_MAX, train_chunks, stats, err);
    fclose(fin);
    const int rc_close = ch.close(err);
    if (!rc) rc = rc_close;
    if (rc) g_io_err = err;
    return rc;
}

extern "C" {

const char* iqgpu_rawfile_last_error(void) { return g_io_err.c_str(); }

int iqgpu_rawfile_run(const iqgpu_chain_config* cfg, int device, const char* in_path, const char* out_path,
                      size_t train_chunks, iqgpu_rawfile_stats* stats)
{
    return iqio::rawfile_run(cfg, 1, device, in_path, &out_path, train_chunks, stats, iqio::process_one);
}

}  // extern "C"

// One pass of an open input stream through existing chains into their open output streams: at most `in_limit_bytes`
// are read from the current position of `fin` (UINT64_MAX = to end of file); the caller owns chains and files.
int iqio::run_stream(const Channels& ch, const iqgpu_chain_config* cfgs, FILE* fin, uint64_t in_limit_bytes, size_t train_chunks,
                     iqgpu_rawfile_stats* stats, std::string& err)
{
    if (train_chunks == 0) train_chunks = 64;      // 1 Mi frames per train: measured best on B200 (profiles/r02_bench_lines.jsonl, file:cfg2)
    const size_t K = ch.chains.size();
    const size_t in_bps = iqgpu_get_bytes_per_sample(cfgs[0].input_format);
    std::vector<size_t> out_bps(K), out_cap(K);
    if (!in_bps) { err = "unhandled sample format"; return IQGPU_EINVAL; }
    int rc = IQGPU_OK;
    const size_t train_frames = train_chunks * (size_t)IQGPU_CHUNK_SAMPLES;
    for (size_t k = 0; k < K; k++) {
        out_bps[k] = iqgpu_get_bytes_per_sample(cfgs[k].output_format);
        if (!out_bps[k]) { err = channel_prefix(k, K) + "unhandled sample format"; return IQGPU_EINVAL; }
        iqgpu_chain_set_option(ch.chains[k], "subtrain_frames", (int64_t)std::min<size_t>(train_frames, (size_t)1 << 24));
        // output capacity of one train: closed form for the worst alignment + one FFT block of slack
        iqgpu_chain_info info{};
        iqgpu_chain_get_info(ch.chains[k], &info);
        const double r = (cfgs[k].no_resample || info.ratio <= 0.f) ? 1.0 : (double)info.ratio;
        const size_t out_cap_frames = (size_t)((double)train_frames * (r > 1.0 ? r : 1.0)) + 4 * IQGPU_CHUNK_SAMPLES + 2 * (size_t)info.filter_block_size + 4096;
        out_cap[k] = out_cap_frames * out_bps[k];
    }

    Ring rin, rout;
    rin.slots.resize(3);
    rout.slots.resize(3);
    bool alloc_ok = true;
    for (auto& s : rin.slots) {
        s.buf.assign(1, iqgpu_host_alloc(train_frames * in_bps));
        s.bytes.assign(1, 0);
        alloc_ok &= s.buf[0] != nullptr;
    }
    for (auto& s : rout.slots) {
        s.buf.assign(K, nullptr);
        s.bytes.assign(K, 0);
        for (size_t k = 0; k < K; k++) { s.buf[k] = iqgpu_host_alloc(out_cap[k]); alloc_ok &= s.buf[k] != nullptr; }
    }
    auto cleanup = [&]() {
        for (auto& s : rin.slots) for (void* b : s.buf) iqgpu_host_free(b);
        for (auto& s : rout.slots) for (void* b : s.buf) iqgpu_host_free(b);
    };
    if (!alloc_ok) { err = "pinned host allocation failed (no CUDA device?)"; cleanup(); return IQGPU_ENOMEM; }

    std::string reader_err, writer_err;
    std::vector<uint64_t> bytes_written(K, 0);
    uint64_t remaining = in_limit_bytes;    // touched by the reader thread only
    // A regular file is read with several pread()s in flight per train (one thread's copy out of the page cache moves
    // ~2 GB/s — less than a tenth of what the chain takes over PCIe; SURVEY 8(f) rank 2); anything else (a pipe) with fread.
    struct stat sb;
    const int fd = fileno(fin);
    const bool regular = fd >= 0 && fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode);
    off_t file_pos = regular ? ftello(fin) : 0;
    const unsigned n_read_threads = regular ? std::max(1u, std::min(8u, std::thread::hardware_concurrency() / 2)) : 1;
    auto parallel_read = [&](char* dst, size_t want, bool& io_error) -> size_t {
        const uint64_t left_in_file = (uint64_t)sb.st_size > (uint64_t)file_pos ? (uint64_t)sb.st_size - (uint64_t)file_pos : 0;
        want = (size_t)std::min<uint64_t>(want, left_in_file);
        if (!want) return 0;
        const size_t slice = ((want + n_read_threads - 1) / n_read_threads + 4095) & ~(size_t)4095;
        std::vector<std::thread> th;
        std::vector<char> bad(n_read_threads, 0);
        for (unsigned k = 0; k < n_read_threads; k++) {
            const size_t lo = (size_t)k * slice;
            if (lo >= want) break;
            const size_t len = std::min(slice, want - lo);
            th.emplace_back([&, k, lo, len] {
                size_t done = 0;
                while (done < len) {
                    const ssize_t r = pread(fd, dst + lo + done, len - done, file_pos + (off_t)(lo + done));
                    if (r <= 0) { bad[k] = 1; return; }
                    done += (size_t)r;
                }
            });
        }
        for (auto& t : th) t.join();
        for (char b : bad) io_error |= b != 0;
        file_pos += (off_t)want;
        return want;
    };
    std::thread reader([&] {
        for (;;) {
            Slot* s = rin.acquire_free();
            if (!s) return;
            const size_t full = train_frames * in_bps;
            const size_t want = (size_t)std::min<uint64_t>(full, remaining);
            bool io_error = false;
            const size_t got = !want ? 0 : (regular ? parallel_read(static_cast<char*>(s->buf[0]), want, io_error) : fread(s->buf[0], 1, want, fin));
            if (io_error || (got < want && !regular && ferror(fin))) { reader_err = "read error on the input file"; rin.abort(); return; }
            remaining -= got;
            s->bytes[0] = got - got % in_bps;   // a trailing partial frame is dropped (input_rawfile.c:236)
            s->last = got < full;
            rin.publish();
            if (s->last) return;
        }
    });
    std::thread writer([&] {
        for (;;) {
            Slot* s = rout.acquire_full();
            if (!s) return;
            for (size_t k = 0; k < K; k++) {
                if (s->bytes[k] && fwrite(s->buf[k], 1, s->bytes[k], ch.fouts[k]) != s->bytes[k]) {
                    writer_err = channel_prefix(k, K) + "write error on the output file";
                    rout.abort(); rin.abort();
                    return;
                }
                bytes_written[k] += s->bytes[k];
            }
            const bool last = s->last;
            rout.release();
            if (last) return;
        }
    });

    uint64_t frames_in = 0, trains = 0;
    std::vector<uint64_t> frames_out(K, 0);
    std::vector<size_t> produced(K, 0);
    rc = IQGPU_OK;
    for (;;) {
        Slot* in = rin.acquire_full();
        if (!in) { rc = IQGPU_EINVAL; break; }
        Slot* out = rout.acquire_free();
        if (!out) { rc = IQGPU_EINVAL; break; }
        const size_t n = in->bytes[0] / in_bps;
        std::fill(produced.begin(), produced.end(), 0);
        if (n) {
            rc = ch.process(ch.chains.data(), K, in->buf[0], n, nullptr, 0, out->buf.data(), out_cap.data(), produced.data(), nullptr);
            if (rc) { err = iqgpu_last_error(); break; }
        }
        frames_in += n; trains++;
        for (size_t k = 0; k < K; k++) { frames_out[k] += produced[k]; out->bytes[k] = produced[k] * out_bps[k]; }
        out->last = in->last;
        const bool last = in->last;
        rin.release();
        rout.publish();
        if (last) break;
    }
    if (rc) { rin.abort(); rout.abort(); }
    reader.join();
    writer.join();
    // an I/O thread that failed aborted the rings, which is what stopped the loop above: report its message
    if (!reader_err.empty()) { err = reader_err; rc = IQGPU_EINVAL; }
    if (!writer_err.empty()) { err = writer_err; rc = IQGPU_EINVAL; }
    if (stats)
        for (size_t k = 0; k < K; k++) {
            stats[k].frames_in = frames_in; stats[k].frames_out = frames_out[k];
            stats[k].bytes_written = bytes_written[k]; stats[k].trains = trains;
        }
    cleanup();
    return rc;
}
