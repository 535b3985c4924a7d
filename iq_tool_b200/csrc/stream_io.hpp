// stream_io.hpp — the reader / chain / writer pass shared by the raw-file and WAV-container entry points
// (rawfile.cpp, wavfile.cpp, channels.cpp).  Host code only; uses the C ABI of include/iqgpu.h.
#pragma once
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/iqgpu.h"

namespace iqio {

// The chain call of a pass: iqgpu_chain_process_multi, or for one channel process_one (iqgpu_chain_process, its K = 1
// case).  rawfile.cpp and wavfile.cpp reach the chain only through this pointer and the single-chain calls, so that
// they link against a test double of those (tests/native/stream_stub.cpp).
using ProcessFn = int (*)(iqgpu_chain* const* chains, size_t n_chains, const void* raw_in, size_t n_frames,
                          const uint32_t* chunk_frames, size_t n_chunks, void* const* out, const size_t* out_capacity_bytes,
                          size_t* out_frames, uint32_t* const* per_chunk_out);
int process_one(iqgpu_chain* const* chains, size_t n_chains, const void* raw_in, size_t n_frames, const uint32_t* chunk_frames,
                size_t n_chunks, void* const* out, const size_t* out_capacity_bytes, size_t* out_frames,
                uint32_t* const* per_chunk_out);

// The chains and output files of a run with one or more channels over one input.
struct Channels {
    ProcessFn process = process_one;
    std::vector<iqgpu_chain*> chains;
    std::vector<FILE*> fouts;
    std::vector<std::string> paths;
    // builds one chain per config on `device`, checks with a zero-frame call that they can share one input, then opens
    // every output for writing.  On failure nothing stays open, the outputs opened so far are removed, and `err` says
    // why (`open_error` + the path when an output cannot be opened).
    int open(const iqgpu_chain_config* cfgs, size_t n, int device, const char* const* out_paths, const char* open_error,
             std::string& err);
    // closes the outputs (IQGPU_EINVAL if a close fails: the data did not reach the file) and destroys the chains
    int close(std::string& err);
    ~Channels();
};

// "channel k: " in front of a message about one channel of several; nothing with one channel
std::string channel_prefix(size_t k, size_t n);

// Streams at most `in_limit_bytes` from the current position of `fin` through every chain of `ch` (one chain call per
// train) into its output file: three overlapped stages on pinned rings, see rawfile.cpp.  cfgs[k] is the configuration
// chain k was built from; stats (optional) receives one record per channel.
int run_stream(const Channels& ch, const iqgpu_chain_config* cfgs, FILE* fin, uint64_t in_limit_bytes, size_t train_chunks,
               iqgpu_rawfile_stats* stats, std::string& err);

// The whole raw-file and WAV / RF64 runs behind iqgpu_rawfile_run(_channels) and iqgpu_wavfile_run(_channels).
int rawfile_run(const iqgpu_chain_config* cfgs, size_t n, int device, const char* in_path, const char* const* out_paths,
                size_t train_chunks, iqgpu_rawfile_stats* stats, ProcessFn process);
int wavfile_run(const iqgpu_chain_config* cfgs, size_t n, int device, const char* in_path, int in_container,
                const char* const* out_paths, const int* out_containers, const float* center_target_hz, size_t train_chunks,
                iqgpu_rawfile_stats* stats, iqgpu_wav_info* in_info, ProcessFn process);

// sets the calling thread's message behind iqgpu_rawfile_last_error()
void set_last_error(const std::string& msg);

}  // namespace iqio
