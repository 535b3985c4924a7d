// Host-only check of the owner types' failure rule (iq_tool_b200/csrc/cuda_owned.hpp): a grow() that cannot be satisfied
// returns the error and leaves the array empty, never a capacity without memory behind it.  With a device the failing
// request replaces real memory first; without one every request fails the same way.
//   nvcc -std=c++17 -I iq_tool_b200/csrc -o cuda_owned_check tests/native/cuda_owned_check.cu
#include <cstdio>

#include "cuda_owned.hpp"
using namespace iqgpu;

static int bad = 0;
#define REQUIRE(cond) do { if (!(cond)) { bad++; printf("  VIOLATED: %s (line %d)\n", #cond, __LINE__); } } while (0)

template <typename A>
static void check(const char* name, bool device)
{
    A a;
    auto drain = [] { return cudaSuccess; };
    if (device) {
        REQUIRE(a.grow(256, 256, drain) == cudaSuccess && a.data() && a.size() == 256);
        auto* p = a.data();
        REQUIRE(a.grow(100, 4096, drain) == cudaSuccess && a.data() == p && a.size() == 256);     // fits: no-op
    }
    // 2^62 bytes: more than any allocator can hand out, refused without touching memory
    const size_t huge = ((size_t)1 << 62) / sizeof(*a.data());
    const cudaError_t e = a.grow(huge, huge, drain);
    REQUIRE(e != cudaSuccess);
    REQUIRE(a.data() == nullptr);
    REQUIRE(a.size() == 0);
    if (device) REQUIRE(a.grow(16, 16, drain) == cudaSuccess && a.data() && a.size() == 16);
    // a drain that fails: the same rule
    REQUIRE(a.grow(1024, 1024, [] { return cudaErrorNotReady; }) == cudaErrorNotReady && a.data() == nullptr && a.size() == 0);
    printf("%s: impossible grow -> %s, empty afterwards\n", name, cudaGetErrorName(e));
}

int main()
{
    int ndev = 0;
    const bool device = cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0;
    cudaGetLastError();
    printf("device: %s\n", device ? "yes" : "no");
    check<DeviceArray<float2>>("DeviceArray", device);
    check<PinnedArray<float2>>("PinnedArray", device);
    printf(bad ? "FAILED\n" : "OK\n");
    return bad ? 1 : 0;
}
