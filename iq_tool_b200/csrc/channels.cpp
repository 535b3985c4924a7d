// channels.cpp — file runs with several channels over one input: the raw-file and WAV / RF64 passes of rawfile.cpp and
// wavfile.cpp with iqgpu_chain_process_multi as their chain call, so that the capture is read and copied to the device
// once for all channels.  Kept apart from those two files, which reach the chain only through the single-chain calls.
#include "../../include/iqgpu.h"
#include "stream_io.hpp"

extern "C" {

int iqgpu_rawfile_run_channels(const iqgpu_chain_config* cfgs, size_t n_channels, int device, const char* in_path,
                               const char* const* out_paths, size_t train_chunks, iqgpu_rawfile_stats* stats)
{
    return iqio::rawfile_run(cfgs, n_channels, device, in_path, out_paths, train_chunks, stats, iqgpu_chain_process_multi);
}

int iqgpu_wavfile_run_channels(const iqgpu_chain_config* cfgs, size_t n_channels, int device, const char* in_path, int in_container,
                               const char* const* out_paths, const int* out_containers, const float* center_target_hz,
                               size_t train_chunks, iqgpu_rawfile_stats* stats, iqgpu_wav_info* in_info)
{
    return iqio::wavfile_run(cfgs, n_channels, device, in_path, in_container, out_paths, out_containers, center_target_hz,
                             train_chunks, stats, in_info, iqgpu_chain_process_multi);
}

}  // extern "C"
