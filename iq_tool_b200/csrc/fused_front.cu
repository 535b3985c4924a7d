// fused_front.cu — the fused "front" of the chain for decimating configurations:
//
//   raw ints --convert--> [DC block] --> [I/Q apply] --> [LUT-NCO mix]            (K1)
//            --> S halfband decimators --> 256-arm polyphase arbitrary resampler  (K2)
//            --> cf32 at the output rate
//
// replacing pre_processor_apply_chain (reference src/pre_processor.c:10-55, minus the optional
// pre-resample filter) + resampler_execute (src/resampler.c:49 -> liquid msresamp_crcf_execute)
// in ONE pass over HBM: 4 B/sample in (cs16), 8*r B/sample out.
//
// The kernel is the warp-streaming one of fused_front2.cuh, instantiated here.  This file matches
// the cascade to one of its compiled plans (S = 0..W2_MAXS halfband stages, semi-lengths
// 3...3,5,10; any other cascade runs the stage-by-stage kernels), sizes and launches it, and runs
// the DC pre-pass.
// Frames older than the call (previous call / sub-train) come from a small cf32 "tail" of the
// pre-processed stream kept in HBM, so nothing depends on how the host cuts the stream into calls.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <vector>

#include "cuda_owned.hpp"
#include "device_common.cuh"
#include "fused_front2.cuh"
#include "kernels.hpp"

namespace iqgpu {

struct FusedFront {
    DeviceArray<float2> d_tail[2];
    int tail_cur = 0;
    // DC pre-pass products, double buffered so that the (HBM-bound) pre-pass of the next sub-train can
    // run on a second stream underneath the (issue-bound) front kernel of the current one
    DeviceArray<double2> d_dc_table[2], d_dc_sums[2];
    DeviceArray<double> d_dc_ws[2];
    bool dc_ready[2] = {false, false};  // slot holds the table of the sub-train about to be launched
    int num_sms = 148;
    int format = 0;
    // the compiled plan of the warp-streaming kernel (fused_front2.cuh) that matches the cascade
    int v2_S = 0, v2_warps = 0, v2_sup = 1, v2_warm_sup = 0, v2_warp_f2 = 0;
    size_t v2_smem = 0;
    float v2_taps[W2_MAX_TAPS] = {0};
    float v2_zeta = 1.f;
    uint32_t v2_step = 0;
    int H_tail = 0;                     // cf32 tail length of the plan
    DeviceArray<float2> d_bank_image;   // polyphase bank in the v2 shared-memory layout (w2_bank_row)
    DeviceArray<float2> d_bank_image_q; // ... and in the layout of the four-output variant (w2_qbank_chunk, rotation arb_tz)
    int arb_tz = 0, arb_b2 = 0, arb_b3 = 0, arb_skew_sh = 31;
    bool arb_quad_ok = false;
    // local DC state (fused_front2.cuh, DC == 2): per-warp records, per-stretch corrections, row gains of the polyphase stage
    DeviceArray<W2DcStretch> d_dc_stretch;
    DeviceArray<W2DcCorr> d_dc_corr;
    DeviceArray<float> d_dc_G;
    float dc_G_for_c = -1.f;            // pole the gains were computed for
    double dc_atot = 1.0;
    std::vector<float> h_bank;          // host copy of the 256 x 14 polyphase bank
    // polyphase stage variant (one or two outputs per lane: same bits, different shared-memory access pattern).  Which one is
    // faster depends on the rate of the arbitrary stage (bank conflicts of the window loads), so the first launch that is
    // large enough times both on its own data — the kernel is idempotent — and the choice sticks.
    int arb_pairs = -1;
    uint32_t lut_dtheta = 0;            // NCO table swizzle chosen for this phase increment
    unsigned lut_sh = 4, lut_mask = 0, lut_rot_sh = 4, lut_rot_c = 0;
    bool lut_picked = false;
};

// ---- v2 plan table ---------------------------------------------------------------------------
template <int S> static bool v2_plan_matches(const ResamplerDesc& r)
{
    if ((int)r.S != S) return false;
    for (int d = 0; d < S; d++)
        if ((int)r.m_exec[d] != W2Plan<S>::m(d)) return false;
    return true;
}
template <int S> static void v2_fill(FusedFront* f)
{
    f->v2_S = S;
    f->v2_sup = W2Plan<S>::sup;
    f->v2_warp_f2 = W2Plan<S>::warp_f2;
    const long long warm_ticks = (W2Plan<S>::halo_frames() + W2_T0 - 1) / W2_T0;
    f->v2_warm_sup = (int)((warm_ticks + W2Plan<S>::sup - 1) / W2Plan<S>::sup);
    f->H_tail = (f->v2_warm_sup + 1) * W2Plan<S>::sup * W2_T0;
}
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder()
{
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q{};
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
// the raw cs16 capture of one call as rows of 128 bytes; a tick is a {32 x u32, 16 rows} box, 128-byte swizzle
static bool encode_raw_map(CUtensorMap* map, const void* raw, size_t n_frames)
{
    EncodeTiledFn enc = tensor_map_encoder();
    const cuuint64_t rows = (cuuint64_t)(n_frames * 4 / 128);
    if (!enc || rows < 16) return false;
    const cuuint64_t dims[2] = {32, rows};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {32, 16};
    const cuuint32_t estr[2] = {1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(raw), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static bool v2_setup(FusedFront* f, const ResamplerDesc& r, bool nco)
{
    bool ok = false;
#define V2_TRY(SS) if (!ok && v2_plan_matches<SS>(r)) { v2_fill<SS>(f); ok = true; }
    V2_TRY(0) V2_TRY(1) V2_TRY(2) V2_TRY(3) V2_TRY(4) V2_TRY(5) V2_TRY(6)
#undef V2_TRY
    if (!ok) return false;
    const bool cs16 = f->format == IQGPU_FMT_CS16 || f->format == IQGPU_FMT_SC16Q11;
    // cs16 kernels: a 2 KiB raw tick buffer per warp in front of everything else, 1 KiB aligned (up to 1 KiB of slack)
    const size_t fixed = (size_t)W2_BANK_F2 * sizeof(float2) + (nco ? 1024 * sizeof(float2) : 0) + (cs16 ? 1024 : 0);
    const size_t per_warp = (size_t)f->v2_warp_f2 * sizeof(float2) + (cs16 ? (size_t)W2_RAW_TICK_BYTES : 0);
    const size_t avail = 227 * 1024 - 256;       // 227 KiB per block is static + dynamic: the barriers (168 bytes) stay clear
    int warps = (int)((avail - fixed) / per_warp);
    if (warps > W2_MAX_WARPS) warps = W2_MAX_WARPS;
    if (warps < 4) return false;
    f->v2_warps = warps;
    f->v2_smem = fixed + (size_t)warps * per_warp;
    int k = 0;
    for (unsigned d = 0; d < r.S; d++)
        for (unsigned j = 0; j < 2 * r.m_exec[d]; j++) f->v2_taps[k++] = r.h1_exec[d][j];
    f->v2_zeta = r.zeta;
    f->v2_step = r.step;
    return true;
}

bool fused_supported(int format, const ResamplerDesc& r)
{
    switch (format) {
        case IQGPU_FMT_CS16: case IQGPU_FMT_SC16Q11: case IQGPU_FMT_CU16: case IQGPU_FMT_CS8: case IQGPU_FMT_CU8:
        case IQGPU_FMT_CF32: break;
        default: return false;
    }
    return v2_plan_matches<0>(r) || v2_plan_matches<1>(r) || v2_plan_matches<2>(r) || v2_plan_matches<3>(r) ||
           v2_plan_matches<4>(r) || v2_plan_matches<5>(r) || v2_plan_matches<6>(r);
}

FusedFront* fused_create(int format, const ResamplerDesc& r, bool nco, const float* d_bank, int num_sms, std::string& err)
{
    std::unique_ptr<FusedFront> f(new FusedFront());
    f->format = format;
    f->num_sms = num_sms;
    if (!v2_setup(f.get(), r, nco)) { err = "fused front: no compiled plan fits this cascade"; return nullptr; }
    if (f->d_tail[0].alloc(f->H_tail) != cudaSuccess || f->d_tail[1].alloc(f->H_tail) != cudaSuccess) {
        err = "fused front: device allocation failed";
        return nullptr;
    }
    // lay the bank out the way the kernel reads it, so one TMA bulk copy stages it per CTA
    std::vector<float> hb(256 * 14);
    std::vector<float2> img(W2_BANK_F2, make_float2(0.f, 0.f));
    if (cudaMemcpy(hb.data(), d_bank, hb.size() * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess ||
        f->d_bank_image.alloc(img.size()) != cudaSuccess) {
        err = "fused front: bank image allocation failed";
        return nullptr;
    }
    f->h_bank = hb;
    for (int idx = 0; idx < 256; idx++)
        for (int i = 0; i < 7; i++) img[w2_bank_row(idx) + i] = make_float2(hb[idx * 14 + 2 * i], hb[idx * 14 + 2 * i + 1]);
    if (cudaMemcpy(f->d_bank_image.data(), img.data(), img.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) {
        err = "fused front: bank image upload failed";
        return nullptr;
    }
    // four-output variant: rows of 16 floats, rotated / chunk-permuted for this rate (fused_front2.cuh)
    f->arb_b2 = (int)((2ull * r.step) >> 24);
    f->arb_b3 = (int)((3ull * r.step) >> 24);
    f->arb_quad_ok = ((f->arb_b2 == 2 && (f->arb_b3 == 3 || f->arb_b3 == 4)) || (f->arb_b2 == 3 && (f->arb_b3 == 4 || f->arb_b3 == 5)));
    if (f->arb_quad_ok) {
        f->arb_tz = (int)w2_pick_qbank_tz(r.step);
        f->arb_skew_sh = 31;
        if (f->v2_S <= 2)       // W2Plan<S>::quad_skew: only the shallow plans have room for a skewed level
            f->arb_skew_sh = w2_pick_flat_skew(r.step);
        std::vector<float> q((size_t)W2_BANK_F2 * 2, 0.f);
        for (unsigned idx = 0; idx < 256; idx++)
            for (unsigned j = 0; j < 4; j++)
                for (unsigned t = 0; t < 4; t++)
                    if (4 * j + t < 14) q[w2_qbank_chunk(idx, (unsigned)f->arb_tz, j) + t] = hb[idx * 14 + 4 * j + t];
        if (f->d_bank_image_q.alloc(q.size() / 2) != cudaSuccess ||
            cudaMemcpy(f->d_bank_image_q.data(), q.data(), q.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
            err = "fused front: bank image upload failed";
            return nullptr;
        }
    }
    return f.release();
}

void fused_destroy(FusedFront* f) { delete f; }

cudaError_t fused_reset(FusedFront* f, cudaStream_t st)
{
    f->tail_cur = 0;
    f->dc_ready[0] = f->dc_ready[1] = false;
    cudaError_t e = cudaMemsetAsync(f->d_tail[0].data(), 0, (size_t)f->H_tail * sizeof(float2), st);
    if (e != cudaSuccess) return e;
    return cudaMemsetAsync(f->d_tail[1].data(), 0, (size_t)f->H_tail * sizeof(float2), st);
}

uint32_t fused_halo_frames(const FusedFront* f)
{
    return (uint32_t)(f->v2_warm_sup * f->v2_sup * W2_T0);
}

// DC blocker state v just before absolute frame `pos` of the sub-train that fused_launch() last ran from frame n0 with table
// slot `slot` (device pointer into the tick table), or nullptr when the launch kept no table entry for that frame (local DC
// state, frame not on a tick boundary)
const double2* fused_dc_state_at(const FusedFront* f, int slot, int64_t n0, int64_t pos)
{
    if (slot < 0 || slot > 1 || !f->d_dc_table[slot].data() || pos < n0) return nullptr;
    const int64_t A0 = (n0 / W2_T0) * W2_T0;
    if ((pos - A0) % W2_T0) return nullptr;
    const size_t idx = (size_t)((pos - A0) / W2_T0);
    return idx < f->d_dc_table[slot].size() ? f->d_dc_table[slot].data() + idx : nullptr;
}

__global__ void dc_rewind_kernel(double2* carry, double c, long long k)
{
    // v(A0) such that k zero frames later the state equals the carried v(n0)
    const double f = pow(c, -(double)k);
    *carry = make_double2(carry->x * f, carry->y * f);
}

// DC pre-pass on the virtual range [A0, N1): frames below n0 read as zero, the carry is rewound to A0
static cudaError_t fused_dc_prepass(FusedFront* f, int slot, const void* raw, long long n0, long long N1, const PreParams& pre,
                                    double2* d_carry, long long A0, cudaStream_t st)
{
    const size_t nv = (size_t)(N1 - A0);
    const size_t n_runs = (nv + 511) / 512;          // one table entry per 512-frame tick
    // rare (first use / larger sub-train): nothing may still read the old buffers
    auto drain = [] { return cudaDeviceSynchronize(); };
    const size_t cap = n_runs * 2 + 16;
    cudaError_t e = f->d_dc_table[slot].grow(n_runs + 2, cap, drain);
    if (e == cudaSuccess) e = f->d_dc_sums[slot].grow(n_runs + 2, cap, drain);
    // the scan's workspace covers the table
    const size_t ws = dc_scan_workspace_doubles(f->d_dc_table[slot].size());
    if (e == cudaSuccess) e = f->d_dc_ws[slot].grow(ws, ws, drain);
    if (e != cudaSuccess) return e;
    const size_t bps = (pre.format == IQGPU_FMT_CS8 || pre.format == IQGPU_FMT_CU8) ? 2 : (pre.format == IQGPU_FMT_CF32 ? 8 : 4);
    const long long back = n0 - A0;
    const char* vraw = reinterpret_cast<const char*>(raw) - back * (long long)bps;
    if (back) dc_rewind_kernel<<<1, 1, 0, st>>>(d_carry, (double)pre.dc_c, back);
    e = launch_dc_tick_sums(vraw, nv, (size_t)back, pre, f->d_dc_sums[slot].data(), st);
    if (e != cudaSuccess) return e;
    return launch_dc_scan(f->d_dc_sums[slot].data(), n_runs, 512, nv, pre.dc_c, d_carry, f->d_dc_table[slot].data(),
                          f->d_dc_ws[slot].data(), st, 512);
}

// DC pre-pass of the sub-train [n0, n0+n) into table slot `slot`, on stream `st` (which may differ from the
// stream of the front kernel: the caller orders them with events).  fused_launch() then skips its own pre-pass.
// local DC state + closed-form correction instead of the pre-pass: the blocker must be followed directly by the (real-tap,
// linear, time-invariant) cascade — no I/Q apply and no table NCO in between
static bool v2_dc_local(const PreParams& pre)
{
    return pre.dc_enable && !pre.nco_enable && !pre.iq_enable && !getenv("IQGPU_DC_TABLE");
}

// gains of the cascade for the sequence c^n (see fused_front2.cuh): Atot over the halfband stages, G per polyphase row
static cudaError_t v2_dc_gains(FusedFront* f, float c, cudaStream_t st)
{
    if (f->dc_G_for_c == c && f->d_dc_G.data()) return cudaSuccess;
    double mu = (double)c, atot = 1.0;
    int k = 0;
    for (int d = 0; d < f->v2_S; d++) {
        const int m = (d == f->v2_S - 1) ? 10 : ((d == f->v2_S - 2) ? 5 : 3);
        double a = pow(mu, (double)(1 - 2 * m));
        for (int j = 0; j < 2 * m; j++) a += (double)f->v2_taps[k + j] * pow(mu, 2.0 * (double)(j + 1 - 2 * m));
        k += 2 * m;
        atot *= a;
        mu *= mu;
    }
    f->dc_atot = atot * (f->v2_S > 0 ? (double)f->v2_zeta : 1.0);
    std::vector<float> G(256);
    for (int idx = 0; idx < 256; idx++) {
        double g = 0.0;
        for (int i = 0; i < 14; i++) g += (double)f->h_bank[idx * 14 + i] * pow(mu, (double)(i - 13));
        G[idx] = (float)g;
    }
    cudaError_t e = cudaSuccess;
    if (!f->d_dc_G.data()) e = f->d_dc_G.alloc(256);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(st);           // first use / new pole only
    if (e != cudaSuccess) return e;
    e = cudaMemcpy(f->d_dc_G.data(), G.data(), 256 * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) f->dc_G_for_c = c;
    return e;
}

cudaError_t fused_prepare_dc(FusedFront* f, int slot, const void* raw, int64_t n0, size_t n, const PreParams& pre,
                             double2* d_dc_carry, uint32_t* launches, cudaStream_t st)
{
    if (n == 0 || !pre.dc_enable) return cudaSuccess;
    if (v2_dc_local(pre)) return cudaSuccess;        // no pre-pass in this mode
    const long long A0 = (n0 / W2_T0) * W2_T0;
    cudaError_t e = fused_dc_prepass(f, slot, raw, n0, n0 + (long long)n, pre, d_dc_carry, A0, st);
    if (e != cudaSuccess) return e;
    f->dc_ready[slot] = true;
    if (launches) *launches += 2;
    return cudaSuccess;
}

template <int S>
static cudaError_t launch_v2_s(const FusedFront* f, const Fused2Args& A, int grid, int dc, bool cs16, cudaStream_t st)
{
    const int threads = f->v2_warps * 32;
    const size_t smem = f->v2_smem;
#define V2_LAUNCH(DCF, C16)                                                                                        \
    do {                                                                                                           \
        cudaError_t e_ = cudaFuncSetAttribute(fused_front2_kernel<S, DCF, C16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e_ != cudaSuccess) return e_;                                                                          \
        fused_front2_kernel<S, DCF, C16><<<grid, threads, smem, st>>>(A, f->v2_warps);                              \
    } while (0)
    if (dc == 2)      { if (cs16) V2_LAUNCH(2, true); else V2_LAUNCH(2, false); }
    else if (dc == 1) { if (cs16) V2_LAUNCH(1, true); else V2_LAUNCH(1, false); }
    else              { if (cs16) V2_LAUNCH(0, true); else V2_LAUNCH(0, false); }
#undef V2_LAUNCH
    return cudaGetLastError();
}

cudaError_t fused_launch(FusedFront* f, const void* raw, int64_t n0, size_t n, const PreParams& pre, double2* d_dc_carry,
                         int64_t O0, size_t n_out, float2* y, uint32_t* launches, int dc_slot, cudaStream_t st, DcFold* fold)
{
    if (fold) fold->corr = nullptr;
    if (n == 0) return cudaSuccess;
    if (dc_slot < 0 || dc_slot > 1) dc_slot = 0;
    Fused2Args A{};
    A.raw = raw; A.n0 = n0; A.N1 = n0 + (long long)n;
    A.tail_in = f->d_tail[f->tail_cur].data();
    A.tail_out = f->d_tail[f->tail_cur ^ 1].data();
    A.H_tail = f->H_tail;
    A.pre = pre;
    A.dc = make_dc_dev16(pre.dc_enable ? pre.dc_c : 0.f, pre.dc_a);
    A.A0 = (n0 / W2_T0) * W2_T0;                 // the tick that contains n0 starts the DC table
    A.bank_image = f->d_bank_image.data();
    A.O0 = O0; A.O1 = O0 + (long long)n_out; A.y = y;
    A.step = f->v2_step; A.zeta = f->v2_zeta;
    A.lut_sh = 4; A.lut_mask = 0;
    A.arb_skew_sh = 31;
    if (pre.nco_enable) {
        if (f->lut_dtheta != pre.nco_dtheta || !f->lut_picked) {
            w2_pick_lut_swizzle(pre.nco_dtheta, f->lut_sh, f->lut_mask);
            f->lut_rot_c = 0;
            if (pre.format == IQGPU_FMT_CS16 || pre.format == IQGPU_FMT_SC16Q11) w2_pick_lut_rotation(pre.nco_dtheta, f->lut_sh, f->lut_mask, f->lut_rot_sh, f->lut_rot_c);
            if (getenv("IQGPU_VERBOSE"))
                fprintf(stderr, "iqgpu: NCO table layout: fold sh %u mask %u, rotation sh %u c %u\n", f->lut_sh, f->lut_mask, f->lut_rot_sh, f->lut_rot_c);
            f->lut_dtheta = pre.nco_dtheta; f->lut_picked = true;
        }
        A.lut_sh = f->lut_sh; A.lut_mask = f->lut_mask;
        A.lut_rot_sh = f->lut_rot_sh; A.lut_rot_c = f->lut_rot_c;
    }
    memcpy(A.taps, f->v2_taps, sizeof(A.taps));
    const long long sup_frames = (long long)f->v2_sup * W2_T0;
    A.sup_first = n0 / sup_frames;
    A.sup_last = (A.N1 - 1) / sup_frames;
    A.warm_sup = f->v2_warm_sup;
    const long long nsup = A.sup_last - A.sup_first + 1;
    const long long total_warps = (long long)f->num_sms * f->v2_warps;
    long long per = (nsup + total_warps - 1) / total_warps;
    // do not let the warm-up dominate: at least 6 warm-up lengths of own work per warp
    const long long min_per = std::max<long long>(1, 6LL * f->v2_warm_sup);
    if (per < min_per) per = min_per;
    A.sup_per_warp = (int)per;
    const long long warps_needed = (nsup + per - 1) / per;
    const int grid = (int)((warps_needed + f->v2_warps - 1) / f->v2_warps);
    A.raw_aligned = ((reinterpret_cast<size_t>(raw) & 15) == 0) && (n0 % 4 == 0);
    // ticks start at absolute multiples of 512 frames: they are whole 128-byte rows of this call's buffer iff n0 is a multiple of 32
    A.raw_tma = 0;
    if ((pre.format == IQGPU_FMT_CS16 || pre.format == IQGPU_FMT_SC16Q11) && A.raw_aligned && n0 % 32 == 0)
        A.raw_tma = encode_raw_map(&A.raw_map, raw, n) ? 1 : 0;
    cudaError_t e;
    if ((long long)n < f->H_tail) {
        const size_t keep = (size_t)f->H_tail - n;
        e = cudaMemcpyAsync(f->d_tail[f->tail_cur ^ 1].data(), f->d_tail[f->tail_cur].data() + n, keep * sizeof(float2),
                            cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return e;
    }
    const bool dc_local = v2_dc_local(pre);
    W2DcGeom geo{};
    if (dc_local) {
        e = v2_dc_gains(f, pre.dc_c, st);
        if (e != cudaSuccess) return e;
        auto drain = [st] { return cudaStreamSynchronize(st); };
        e = f->d_dc_stretch.grow((size_t)warps_needed, (size_t)warps_needed + 64, drain);
        if (e == cudaSuccess) e = f->d_dc_corr.grow((size_t)warps_needed, (size_t)warps_needed + 64, drain);
        if (e != cudaSuccess) return e;
        const double c = (double)pre.dc_c;
        A.dc_carry = d_dc_carry;
        A.dc_stretch = f->d_dc_stretch.data();
        A.dc_lnc = log(c);
        A.dc_c512 = pow(c, 512.0);
        geo.n_stretch = (int)warps_needed;
        geo.B0 = A.sup_first * sup_frames;
        geo.L_full = per * sup_frames;
        if (geo.L_full + (long long)f->v2_warm_sup * sup_frames >= (1LL << 31)) return cudaErrorInvalidValue;   // dc_fold_add: int
        geo.L_last = (A.sup_last - (A.sup_first + (warps_needed - 1) * per) + 1) * sup_frames;
        geo.warm_frames = (long long)f->v2_warm_sup * sup_frames;
        geo.pad_frames = (A.sup_last + 1) * sup_frames - A.N1;
        geo.lnc = A.dc_lnc; geo.alpha = (double)pre.dc_a; geo.atot = f->dc_atot;
    } else if (pre.dc_enable) {
        if (!f->dc_ready[dc_slot]) {
            e = fused_dc_prepass(f, dc_slot, raw, n0, A.N1, pre, d_dc_carry, A.A0, st);
            if (e != cudaSuccess) return e;
            if (launches) *launches += 2;
        }
        f->dc_ready[dc_slot] = false;
        A.dc_table = f->d_dc_table[dc_slot].data();
        A.dc_table_shift = 9;
    }
    const int dc = dc_local ? 2 : (pre.dc_enable ? 1 : 0);
    const bool cs16 = pre.format == IQGPU_FMT_CS16 || pre.format == IQGPU_FMT_SC16Q11;
    auto go = [&](const Fused2Args& a) -> cudaError_t {
        switch (f->v2_S) {
            case 0: return launch_v2_s<0>(f, a, grid, dc, cs16, st);
            case 1: return launch_v2_s<1>(f, a, grid, dc, cs16, st);
            case 2: return launch_v2_s<2>(f, a, grid, dc, cs16, st);
            case 3: return launch_v2_s<3>(f, a, grid, dc, cs16, st);
            case 4: return launch_v2_s<4>(f, a, grid, dc, cs16, st);
            case 5: return launch_v2_s<5>(f, a, grid, dc, cs16, st);
            case 6: return launch_v2_s<6>(f, a, grid, dc, cs16, st);
            default: return cudaErrorInvalidValue;
        }
    };
    A.arb_tz = f->arb_tz; A.arb_b2 = f->arb_b2; A.arb_b3 = f->arb_b3;
    auto set_mode = [&](int m) {
        A.arb_pairs = m;
        A.bank_image = (m == 2) ? f->d_bank_image_q.data() : f->d_bank_image.data();
        A.arb_skew_sh = (m == 2) ? f->arb_skew_sh : 31;
    };
    if (const char* force = getenv("IQGPU_ARB_PAIRS")) {
        f->arb_pairs = std::max(0, std::min(2, atoi(force)));
        if (f->arb_pairs == 2 && !f->arb_quad_ok) f->arb_pairs = 1;
    }
    if (f->arb_pairs < 0 && n >= ((size_t)1 << 22)) {
        // time the variants on this launch (same inputs, same outputs: every run overwrites the last with equal bits)
        const int nmodes = f->arb_quad_ok ? 3 : 2;
        Event ev[4];
        for (auto& x : ev) create(x, cudaEventDefault);
        float ms[3] = {0.f, 0.f, 0.f};
        set_mode(1); e = go(A);                          // untimed: caches, clocks, TMA descriptors warm for all candidates
        cudaEventRecord(ev[0], st);
        for (int m = 0; m < nmodes && e == cudaSuccess; m++) {
            set_mode(m); e = go(A);
            cudaEventRecord(ev[m + 1], st);
        }
        if (e == cudaSuccess) e = cudaEventSynchronize(ev[nmodes]);
        if (e == cudaSuccess) {
            int best = 0;
            for (int m = 0; m < nmodes; m++) {
                cudaEventElapsedTime(&ms[m], ev[m], ev[m + 1]);
                if (ms[m] < 0.98f * ms[best]) best = m;
            }
            f->arb_pairs = best;
            if (getenv("IQGPU_VERBOSE"))
                fprintf(stderr, "iqgpu: polyphase stage: one output per lane %.3f ms, two %.3f ms, four %.3f ms -> mode %d (tz %d, B2 %d, B3 %d, skew %d)\n",
                        ms[0], ms[1], ms[2], best, f->arb_tz, f->arb_b2, f->arb_b3, f->arb_skew_sh);
        }
        if (launches) *launches += (uint32_t)nmodes;
        if (e == cudaSuccess && A.arb_pairs != f->arb_pairs) { set_mode(f->arb_pairs); e = go(A); if (launches) *launches += 1; }
    } else {
        set_mode(f->arb_pairs > 0 ? f->arb_pairs : 0);
        e = go(A);
    }
    if (launches) *launches += 1;
    if (dc_local && e == cudaSuccess) {
        w2_dc_scan_kernel<<<1, 1024, 0, st>>>(f->d_dc_stretch.data(), geo, f->d_dc_corr.data(), d_dc_carry);
        // a consumer that adds the term to the resampled stream itself leaves only the cf32 tail to this pass
        const long long O1c = fold ? A.O0 : A.O1;
        if (fold) *fold = DcFold{f->d_dc_corr.data(), f->d_dc_G.data(), geo, A.O0, A.step, f->v2_S};
        const long long work = (O1c - A.O0) + f->H_tail;
        const int cgrid = (int)std::min<long long>((work + 255) / 256, 148LL * 16);
        w2_dc_correct_kernel<<<std::max(cgrid, 1), 256, 0, st>>>(y, A.O0, O1c, A.step, f->v2_S, geo, f->d_dc_corr.data(),
                                                               f->d_dc_G.data(), f->d_tail[f->tail_cur ^ 1].data(), A.N1 - f->H_tail,
                                                               A.n0, A.N1);
        e = cudaGetLastError();
        if (launches) *launches += 2;
    }
    f->tail_cur ^= 1;
    return e;
}

// the closed-form term, in memory, for the samples [first, first + count) of the launch `fold` describes
cudaError_t fused_dc_correct_range(const DcFold& fold, float2* y, size_t first, size_t count, cudaStream_t st)
{
    if (!fold.corr || count == 0) return cudaSuccess;
    const long long Oa = fold.O0 + (long long)first;
    const int cgrid = (int)std::min<size_t>((count + 255) / 256, (size_t)148 * 16);
    w2_dc_correct_kernel<<<std::max(cgrid, 1), 256, 0, st>>>(y + first, Oa, Oa + (long long)count, fold.step, fold.S, fold.geo,
                                                           fold.corr, fold.G, nullptr, 0, 0, 0);
    return cudaGetLastError();
}

}  // namespace iqgpu
