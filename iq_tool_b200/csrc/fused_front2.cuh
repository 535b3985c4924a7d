// fused_front2.cuh — the "warp-streaming" fused front kernel (v2; host side in fused_front.cu):
// convert -> [DC] -> [I/Q] -> [NCO] -> S halfband decimators -> 256-arm polyphase stage, reference
// src/pre_processor.c:10-55 + src/resampler.c:49.  Its shape answers what ncu showed about the
// block-synchronous kernel it replaced (profiles/r01a_fused_front_full_cfg2.md): that kernel was
// instruction-issue bound (54 % issue active, 15 % FMA pipe, 7 % DRAM) with most issue slots going
// to address arithmetic, run-time plan lookups and block barriers.
//
//   * Every WARP owns a contiguous run of the stream and a private set of level FIFOs in shared
//     memory; nothing is shared between warps except read-only tables, so the kernel has no
//     __syncthreads in its steady state (only __syncwarp between producer and consumer phases).
//   * The plan (stage count S, semi-lengths m, tile sizes, padded layouts) is a template
//     parameter: every shared-memory offset is an immediate, halfband taps are read straight from
//     the kernel-parameter constant bank as FFMA operands.
//   * A tick is 512 raw frames per warp; a lane owns 16 consecutive frames (4 x LDG.128 for
//     cs16), so the DC blocker's weighted prefix needs one warp scan per 512 frames instead of
//     four, and stage d gives every lane R = 8, 4, 2, 1 consecutive outputs (register tiles fed
//     by LDS.128 from group-padded planes, bank-conflict free).  Stages deeper than 3 run every
//     2^(d-3) ticks on 32 outputs.
//   * Accumulation order is the reference's (oldest tap first), so results are bit-identical to
//     the stage-by-stage kernels; all indices are absolute, so results do not depend on how the
//     host cuts the stream into calls.
#pragma once
#include <cuda.h>          // CUtensorMap (type only: the encoder is fetched through cudaGetDriverEntryPoint)
#include "device_common.cuh"
#include "kernels.hpp"

namespace iqgpu {

constexpr int W2_T0 = 512;          // raw frames per warp tick
#ifndef W2_CAP_DEF
#define W2_CAP_DEF 0                // 0: per-plan default (W2Plan::CAP)
#endif
#ifndef W2_REG0_M5_DEF
#define W2_REG0_M5_DEF 1            // S == 2: first stage (semi-length 5) from registers
#endif
#ifndef W2_REG1_DEF
#define W2_REG1_DEF 1               // second halfband stage from registers too (S >= 4)
#endif
#ifndef W2_MAX_WARPS_DEF
#define W2_MAX_WARPS_DEF 20
#endif
constexpr int W2_MAX_WARPS = W2_MAX_WARPS_DEF;   // warps per CTA (one CTA per SM): bounded by 64K registers / (32 x registers per thread)
constexpr int W2_ARB_HIST = 16;     // >= 13 decimated samples of look-back
// polyphase bank image in shared memory: row `idx` (14 taps = 7 float2) starts at float2 offset
// 9*idx + (idx >> 2).  The odd stride plus the slow skew keeps the 16 lanes of a half-warp, whose
// rows advance by a configuration-dependent step, spread over the 16 LDS.64 bank pairs (a plain
// stride degenerates to 16-way conflicts when the step has a factor of 8; measured on cfg1:
// profiles/r01c_fused_front2_full_cfg1.md).  The image is laid out by the host and pulled in with
// one TMA bulk copy (cp.async.bulk) per CTA.
// NCO table {sign*sin, cos}[1024] in shared memory, XOR-swizzled: lanes look up phases that advance by a
// configuration-dependent stride (16 frames apart), which on a plain table piles a half-warp onto a few
// bank pairs (6-way on cfg5); folding index bits 4..7 into the bank bits spreads any stride.
// Which fold (none, or index bits sh..sh+3 with sh = 4, 5, 6) is best depends on the phase increment, so the
// host simulates the half-warp access pattern for the actual increment and picks one (w2_pick_lut_swizzle).
__host__ __device__ constexpr unsigned w2_lut_slot(unsigned idx, unsigned sh, unsigned mask) { return idx ^ ((idx >> sh) & mask); }
// Second family, for increments at which no XOR fold gets below two-way conflicts (cfg5: lanes 26.67 entries apart,
// 2.2 wavefronts per half warp after the best fold, 1.6 here): the entries of every row of 16 are ROTATED by a multiple of
// a higher index field, slot = row | ((idx + c (idx >> sh)) mod 16) — a permutation of the table for any c.
__host__ __device__ constexpr unsigned w2_lut_slot_rot(unsigned idx, unsigned sh, unsigned c)
{
    return (idx & ~15u) | ((idx + c * (idx >> sh)) & 15u);
}
template <typename SLOT>
__host__ static inline double w2_lut_cost(uint32_t dtheta, SLOT slot)
{
    double cost = 0;
    for (uint32_t trial = 0; trial < 64; trial++) {
        const uint32_t th0 = trial * 0x9e3779b9u;          // arbitrary start phases
        for (int half = 0; half < 2; half++) {
            int hits[16] = {0};
            unsigned seen_idx[16];
            int deg = 0;
            for (int l = 0; l < 16; l++) {
                const uint32_t th = th0 + (uint32_t)((half * 16 + l) * 16) * dtheta;
                const unsigned idx = ((th + (1u << 21)) >> 22) & 0x3ffu;
                seen_idx[l] = idx;
                bool dup = false;                          // identical addresses broadcast
                for (int m = 0; m < l; m++) dup |= (seen_idx[m] == idx);
                if (dup) continue;
                const unsigned b = slot(idx) & 15u;
                if (++hits[b] > deg) deg = hits[b];
            }
            cost += deg;
        }
    }
    return cost;
}
// rotation (c != 0) only when it beats the best fold by 10 %: it costs one more instruction per look-up
__host__ static inline void w2_pick_lut_rotation(uint32_t dtheta, unsigned xor_sh, unsigned xor_mask, unsigned& rot_sh, unsigned& rot_c)
{
    const double base = w2_lut_cost(dtheta, [&](unsigned i) { return w2_lut_slot(i, xor_sh, xor_mask); });
    double best = base * 0.9;
    rot_sh = 4; rot_c = 0;
    for (unsigned sh = 3; sh <= 7; sh++)
        for (unsigned c = 1; c < 16; c++) {
            const double k = w2_lut_cost(dtheta, [&](unsigned i) { return w2_lut_slot_rot(i, sh, c); });
            if (k < best - 1e-9) { best = k; rot_sh = sh; rot_c = c; }
        }
}
__host__ static inline void w2_pick_lut_swizzle(uint32_t dtheta, unsigned& sh, unsigned& mask)
{
    const unsigned cand_sh[4] = {4, 4, 5, 6}, cand_mask[4] = {0, 15, 15, 15};
    double best = 1e30;
    sh = 4; mask = 0;
    for (int c = 0; c < 4; c++) {
        double cost = 0;
        for (uint32_t trial = 0; trial < 64; trial++) {
            const uint32_t th0 = trial * 0x9e3779b9u;          // arbitrary start phases
            for (int half = 0; half < 2; half++) {
                int hits[16] = {0};
                unsigned seen_idx[16];
                int deg = 0;
                for (int l = 0; l < 16; l++) {
                    const uint32_t th = th0 + (uint32_t)((half * 16 + l) * 16) * dtheta;
                    const unsigned idx = ((th + (1u << 21)) >> 22) & 0x3ffu;
                    seen_idx[l] = idx;
                    bool dup = false;                          // identical addresses broadcast
                    for (int m = 0; m < l; m++) dup |= (seen_idx[m] == idx);
                    if (dup) continue;
                    const unsigned b = w2_lut_slot(idx, cand_sh[c], cand_mask[c]) & 15u;
                    if (++hits[b] > deg) deg = hits[b];
                }
                cost += deg;
            }
        }
        if (cost < best - 1e-9) { best = cost; sh = cand_sh[c]; mask = cand_mask[c]; }
    }
}
__host__ __device__ constexpr int w2_flat_phys(int e, int sh) { return e + ((e >> sh) << 1); }
__host__ __device__ constexpr int w2_ilog2(int v) { int l = 0; while ((1 << (l + 1)) <= v) l++; return l; }
constexpr int W2_BANK_F2 = 2368;    // float2 entries of the image (9*255 + 63 + 7 = 2365, padded to 16 B)
// (two leading float2 of zeros: the second output of a lane reads its taps through a pointer shifted back by up to two floats)
__host__ __device__ constexpr int w2_bank_row(int idx) { return 9 * idx + (idx >> 2) + 2; }
constexpr int W2_MAX_TAPS = 72;     // sum of 2m over the cascade (6*4 + 10 + 20 = 54 for S = 6)

// compile-time plan of a cascade of S halfband stages; semi-lengths by execution depth are
// 3,...,3,5,10 (liquid msresamp2 at As = 60 dB, SURVEY App. A7) — checked against the run-time
// design in fused2_supported().
template <int S>
struct W2Plan {
    __host__ __device__ static constexpr int m(int d) { return (d == S - 1) ? 10 : ((d == S - 2) ? 5 : 3); }
    // Stage d makes 256 >> d outputs per tick.  Deep stages would leave a lane with one output per run (21 shared-memory
    // loads for one output at m = 10: the kernel is bound by the LSU data pipe), so they wait for several ticks and run
    // on CAP outputs at a time: R = CAP/32 consecutive outputs per lane share one register window.
    static constexpr int CAP = W2_CAP_DEF ? W2_CAP_DEF : ((S <= 4) ? 128 : 64);
    __host__ __device__ static constexpr int nat(int d) { return 256 >> d; }
    __host__ __device__ static constexpr int out(int d) { return nat(d) > CAP ? nat(d) : CAP; }   // outputs of stage d per run
    __host__ __device__ static constexpr int R(int d) { return out(d) / 32; }                 // consecutive outputs per lane
    __host__ __device__ static constexpr int PAD(int d) { return R(d) >= 4 ? 2 : (R(d) == 2 ? 1 : 0); }
    __host__ __device__ static constexpr int Hh(int d) { return ((2 * m(d) - 1 + R(d) - 1) / R(d)) * R(d); }   // history entries per plane
    __host__ __device__ static constexpr int entries(int d) { return Hh(d) + out(d); }
    __host__ __device__ static constexpr int phys(int d, int p) { return p + PAD(d) * (p / R(d)); }
    // A level whose producer needs two runs per consumer run (both capped: ratio(d - 1) == 2) is written by lane PAIRS per
    // padded group, which puts two lanes of every quarter (R = 4: STS.128) or three of every half warp (R = 2: STS.64) on a
    // bank group another lane already uses (profiles/r02i_fused_front2_full_cfg2.md: 12 of 228 LSU wavefronts per tick).
    // Those lanes store their O entry first and their E entry second (w2_stage_store); that is conflict free when the O
    // plane starts 8 (mod 16) entries after the E plane, which is what the extra padding here arranges.
    __host__ __device__ static constexpr bool pair_fed(int d)
    {
        return d >= 1 && d < S && (2 * out(d) / out(d - 1) == 2) && (R(d) == 4 || R(d) == 2);
    }
    __host__ __device__ static constexpr int plane_size(int d)
    {
        int n = (phys(d, entries(d)) + 3) & ~1;
        if (pair_fed(d)) while (n % 16 != 8) n += 2;
        return n;
    }
    // first stage straight from the lane's registers (neighbour entries by warp shuffle): cascades whose first
    // stage has semi-length 3, i.e. S >= 3.  Level 0 then keeps only an 8-entry history instead of its planes.
    static constexpr bool reg0 = (S >= 3) || (S == 2 && W2_REG0_M5_DEF);     // S == 2: first stage of semi-length 5
    // ... and the second one as well when it also has semi-length 3 (S >= 4): the lane's 8 first-stage outputs are 4 (E, O)
    // pairs of level 1, the inputs of its own 4 second-stage outputs; older entries come from the two lanes below
    static constexpr bool reg1 = W2_REG1_DEF && (S >= 4);
    // (a register stage keeps only the hand-over history of its last lanes: 8 entries at semi-length 3, 14 at 5)
    __host__ __device__ static constexpr int level_size(int d)
    {
        return ((d == 0 && reg0) || (d == 1 && reg1)) ? (m(d) == 3 ? 8 : 16) : 2 * plane_size(d);
    }
    __host__ __device__ static constexpr int e_off(int d)
    {
        int o = 0;
        for (int i = 0; i < d; i++) o += level_size(i);
        return o;
    }
    __host__ __device__ static constexpr int o_off(int d) { return e_off(d) + plane_size(d); }
    __host__ __device__ static constexpr int taps_off(int d)
    {
        int o = 0;
        for (int i = 0; i < d; i++) o += 2 * m(i);
        return o;
    }
    static constexpr int flat_new = (S == 0) ? W2_T0 : out(S - 1);        // new polyphase inputs per arb run
    static constexpr int flat_off = e_off(S);
    // + 8: the four-output polyphase variant reads up to 6 entries beyond the newest one (they meet zero taps; the slack is
    // zeroed once and never written, so the products are exact zeros)
    // (+ 1/8 on top: room for the skew of the four-output variant, 2 entries per 16)
    // The skewed level exists for the shallow cascades, where the polyphase stage is most of the kernel (S <= 2: one output
    // per lane spends 60 % of cfg1's LSU wavefronts there); deeper cascades take the four-output variant on the plain level
    // (+ 64 bytes per warp: S = 4 keeps its 20 warps, the 220 bytes of the skew room would cost the 20th)
    static constexpr bool quad = true;
    static constexpr bool quad_skew = (S <= 2);
    static constexpr int flat_lin = W2_ARB_HIST + flat_new + (quad ? 8 : 0);
    static constexpr int flat_size = quad_skew ? ((flat_lin + flat_lin / 8 + 2 + 1) & ~1) : ((flat_lin + 3) & ~1);
    static constexpr int warp_f2 = flat_off + flat_size;                 // float2 per warp
    __host__ __device__ static constexpr int period(int d) { return nat(d) >= CAP ? 1 : CAP / nat(d); }   // stage d runs every `period` ticks
    // runs of stage d per run of stage d+1 (1: every run feeds one consumer run; 2: the consumer waits for two)
    __host__ __device__ static constexpr int ratio(int d) { return 2 * out(d + 1) / out(d); }
    static constexpr int sup = (S == 0) ? 1 : period(S - 1);             // ticks per super-tick (period of the last stage)
    __host__ __device__ static constexpr long long halo_frames()
    {
        long long h = 0;
        for (int d = 0; d < S; d++) h += (long long)(4 * m(d)) << d;
        return h + ((long long)W2_ARB_HIST << S);
    }
};

struct W2DcStretch { double2 v_emit, v_end; };   // local v at the first frame of the warp's emit range / after its last tick

struct Fused2Args {
    const void* raw;
    long long n0, N1;                   // absolute index range of raw
    const float2* tail_in;
    float2* tail_out;
    int H_tail;
    PreParams pre;
    DcDev16 dc;
    const double2* dc_table;            // v at absolute multiples of 2^dc_table_shift frames, starting at A0
    int dc_table_shift;                 // 9: per-tick table (dc_tick_sums pre-pass)
    long long A0;
    // DC == 2 ("local" DC state, no pre-pass): every warp carries v through its own stretch from zero (the warp that holds
    // n0 from the carried state) and reports v at the start and the end of its emit range; the term it misses is a
    // decaying exponential, an eigenfunction of the linear cascade, added afterwards in closed form (w2_dc_correct_kernel)
    const double2* dc_carry;            // device: v just before frame n0
    W2DcStretch* dc_stretch;            // one record per warp of the launch
    double dc_c512, dc_lnc;             // c^512 and ln c in double (c = the float pole)
    const float2* bank_image;           // device, W2_BANK_F2 float2 in the w2_bank_row layout
    long long O0, O1;
    ArbBase arb_pos;                    // polyphase position of O0 (kernels.hpp): k and row of every output o >= O0
    float2* y;
    long long sup_first, sup_last;      // absolute super-tick range of the call
    int sup_per_warp, warm_sup;
    int raw_aligned;
    uint32_t step;
    float zeta;
    unsigned lut_sh, lut_mask;          // NCO table swizzle (w2_lut_slot)
    unsigned lut_rot_sh, lut_rot_c;     // lut_rot_c != 0: the rotation family instead (w2_lut_slot_rot)
    int arb_pairs;                      // polyphase stage: one output per lane (0), two (1) or four (2); same bits, picked by timing
    int arb_tz, arb_b2, arb_b3;         // four-output variant: row rotation of the bank image; floor(2/rate), floor(3/rate)
    // skew of the polyphase input level: entry e sits at e + 2 * (e >> arb_skew_sh) (31: none).  The four-output variant's
    // window loads start 4 / rate entries apart from lane to lane; at rates where three such strides come to ~16 entries
    // (cfg1: 16.13) the lanes of a half warp pile onto three bank groups — two entries of padding per 16 (or 32) spread them
    int arb_skew_sh;
    float taps[W2_MAX_TAPS];            // h1 by execution depth, concatenated (constant-bank FFMA operands)
    // raw staging by TMA (cs16): the capture seen as rows of 128 bytes (32 frames); a tick is a box of 16 rows that one
    // cp.async.bulk.tensor per warp drops into the warp's 2 KiB buffer with the 128-byte swizzle, so that the lanes' 64-byte
    // runs (16 consecutive frames each) come out with four conflict-free LDS.128 — instead of four LDG.128 whose 32 lanes
    // touch 16 different cache lines each (64 LSU wavefronts per tick, a quarter of the kernel's LSU traffic in
    // profiles/r01j_fused_front2_full_cfg2.md)
    int raw_tma;                        // 0: the map is not valid (unaligned call): ticks load with LDG
    alignas(64) CUtensorMap raw_map;
};
constexpr int W2_RAW_TICK_BYTES = W2_T0 * 4;     // cs16 tick

// ------------------------------------------------------------------------------------------------
// TMA bulk copy global -> shared with mbarrier completion (cp.async.bulk, sm_90+/sm_100a)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t w2_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void w2_mbar_init(uint64_t* bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(w2_smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void w2_tma_load(void* smem_dst, const void* gmem_src, unsigned bytes, uint64_t* bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(w2_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(w2_smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(w2_smem_u32(bar)) : "memory");
}
// one tick of raw cs16 frames: box {32 x u32, 16 rows} at row `row` of the capture -> 2 KiB of shared memory (128B swizzle)
__device__ __forceinline__ void w2_tma_load_tick(void* smem_dst, const CUtensorMap* map, int row, uint64_t* bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(w2_smem_u32(bar)), "r"(W2_RAW_TICK_BYTES) : "memory");
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(w2_smem_u32(smem_dst)), "l"(map), "r"(0), "r"(row), "r"(w2_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void w2_mbar_wait(uint64_t* bar, unsigned parity)
{
    uint32_t ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(w2_smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}

// ------------------------------------------------------------------------------------------------
// raw loaders (16 consecutive frames of one lane)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float w2_scale(int fmt, float gain)
{
    switch (fmt) {
        case IQGPU_FMT_CS16: case IQGPU_FMT_CU16: return gain * (1.0f / 32768.0f);
        case IQGPU_FMT_SC16Q11: return gain * (1.0f / 2048.0f);
        case IQGPU_FMT_CS8: case IQGPU_FMT_CU8: return gain * (1.0f / 128.0f);
        default: return gain;
    }
}
__device__ __forceinline__ float2 w2_load_frame(int fmt, const void* __restrict__ raw, size_t i, float sc, float gain)
{
    switch (fmt) {
        case IQGPU_FMT_CS16: case IQGPU_FMT_SC16Q11: return load_frame<IQGPU_FMT_CS16>(raw, i, sc, gain);
        case IQGPU_FMT_CU16: return load_frame<IQGPU_FMT_CU16>(raw, i, sc, gain);
        case IQGPU_FMT_CS8: return load_frame<IQGPU_FMT_CS8>(raw, i, sc, gain);
        case IQGPU_FMT_CU8: return load_frame<IQGPU_FMT_CU8>(raw, i, sc, gain);
        default: return load_frame<IQGPU_FMT_CF32>(raw, i, sc, gain);
    }
}
__device__ __forceinline__ void w2_load_quad(int fmt, const void* __restrict__ raw, size_t i, float sc, float gain, float2 (&x)[4])
{
    const size_t big = ~(size_t)0 >> 1;
    switch (fmt) {
        case IQGPU_FMT_CS16: case IQGPU_FMT_SC16Q11: load_quad<IQGPU_FMT_CS16>(raw, i, big, sc, gain, true, x); break;
        case IQGPU_FMT_CS8: load_quad<IQGPU_FMT_CS8>(raw, i, big, sc, gain, true, x); break;
        case IQGPU_FMT_CU8: load_quad<IQGPU_FMT_CU8>(raw, i, big, sc, gain, true, x); break;
        case IQGPU_FMT_CF32: load_quad<IQGPU_FMT_CF32>(raw, i, big, sc, gain, true, x); break;
        default:
#pragma unroll
            for (int k = 0; k < 4; k++) x[k] = w2_load_frame(fmt, raw, i + k, sc, gain);
    }
}

// raw frames of one tick and one lane (cs16 fast path): four 16-byte chunks
struct W2Raw { uint4 q[4]; };
struct W2True { static constexpr bool value = true; };
struct W2False { static constexpr bool value = false; };

// ------------------------------------------------------------------------------------------------
// P0: one tick (512 frames) of the pre-processor chain into level 0 (or the flat level when S == 0)
// ------------------------------------------------------------------------------------------------
template <int S, int DC, bool CS16>
__device__ __forceinline__ void w2_p0(const Fused2Args& A, float2* __restrict__ wsm, const float2* __restrict__ lut2,
                                      long long tick_start, int lane, const W2Raw& pre, f32x2_t (&x)[16], double2& vloc,
                                      bool write_tail, bool active, bool fast)
{
    // active: the tick holds frames of this call; fast: all of them come from this call's raw buffer with aligned vector
    // loads and none belongs to the cf32 tail (both decided by the caller from per-warp tick ranges)
    using P = W2Plan<S>;
    const PreParams& p = A.pre;
    const int fmt = CS16 ? IQGPU_FMT_CS16 : p.format;
    const float sc = CS16 ? p.gain * ((p.format == IQGPU_FMT_SC16Q11) ? (1.0f / 2048.0f) : (1.0f / 32768.0f)) : w2_scale(fmt, p.gain);
    const long long a0 = tick_start + lane * 16;               // first frame of this lane
    // the lane's 16 frames as packed {re, im} pairs (FMUL2 / FFMA2: one issue slot per complex sample)
    if (fast && CS16) {
        // sample_convert.c:136-141: x / 32768 * gain (exact power-of-two scale folded into sc)
        const f32x2_t sc2 = pk2(sc, sc);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const unsigned w[4] = {pre.q[j].x, pre.q[j].y, pre.q[j].z, pre.q[j].w};
#pragma unroll
            for (int k = 0; k < 4; k++)
                x[4 * j + k] = mul2(pk2((float)(short)(w[k] & 0xffffu), (float)(short)(w[k] >> 16)), sc2);
        }
    } else if (fast) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            float2 q[4];
            w2_load_quad(fmt, A.raw, (size_t)(a0 - A.n0) + 4 * j, sc, p.gain, q);
#pragma unroll
            for (int k = 0; k < 4; k++) x[4 * j + k] = pk2(q[k]);
        }
    } else if (active) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const long long i = a0 + k;
            x[k] = (i >= A.n0 && i < A.N1) ? pk2(w2_load_frame(fmt, A.raw, (size_t)(i - A.n0), sc, p.gain)) : 0ull;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = 0ull;
    }
    if (DC == 2 && !active) { vloc.x *= A.dc_c512; vloc.y *= A.dc_c512; }     // a tick of zeros
    if (active) {
        if (DC) {
            // DC blocker (dc_block.c:76 -> liquid iirfilt): v[n] = x[n] + c v[n-1], y[n] = x[n] - (1-c) v[n-1].
            // lane-local weighted sum, one warp scan per tick, state at the tick start from the table
            const double2 vt = (DC == 2) ? vloc : A.dc_table[(tick_start - A.A0) >> A.dc_table_shift];
            // v just before the lane's frame k is c^k w0 + P(k-1), P = the lane-local running sum, so
            //   y[k] = (x[k] - a P(k-1)) - (a c^k) w0 :
            // the first term hangs off the lane-local chain and is independent of the warp scan that delivers w0;
            // once w0 is known the 16 corrections are independent FMAs (no second serial chain).
            const f32x2_t cc = pk2(A.dc.c, A.dc.c), na = pk2(-A.dc.a, -A.dc.a);
            f32x2_t pr = x[0];
#pragma unroll
            for (int k = 1; k < 16; k++) {
                const f32x2_t t = fma2(na, pr, x[k]);
                pr = fma2(pr, cc, x[k]);
                x[k] = t;
            }
#pragma unroll
            for (int s = 0; s < 5; s++) {
                const int dist = 1 << s;
                const f32x2_t q = __shfl_up_sync(0xffffffffu, pr, dist);
                pr = fma2s((lane >= dist) ? A.dc.w[s] : 0.f, q, pr);        // (+ 0 * q: pr unchanged; q is finite)
            }
            f32x2_t e = __shfl_up_sync(0xffffffffu, pr, 1);
            if (lane == 0) e = 0ull;
            if (DC == 2) {      // carry the state to the next tick: v' = c^512 v + (weighted sum of the tick)
                const float2 tot = unpk2(__shfl_sync(0xffffffffu, pr, 31));
                vloc.x = fma(A.dc_c512, vloc.x, (double)tot.x);
                vloc.y = fma(A.dc_c512, vloc.y, (double)tot.y);
            }
            const float lp = A.dc.lanepow[lane];
            const f32x2_t w0 = fma2s(lp, pk2((float)vt.x, (float)vt.y), e);   // v just before the lane's first frame
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = fma2s(A.dc.nac[k], w0, x[k]);
        }
        if (p.iq_enable) {   // iq_correct.c:307-313
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const float2 v = unpk2(x[k]);
                x[k] = pk2(__fmul_rn(v.x, p.iq_magp1), __fadd_rn(v.y, __fmul_rn(p.iq_phase, v.x)));
            }
        }
        if (p.nco_enable) {  // liquid LIQUID_NCO: 32-bit phase, 1024-entry table, nearest entry
            uint32_t th = p.nco_theta0 + (uint32_t)(a0 - A.n0) * p.nco_dtheta;
            // one loop per table layout (the choice is uniform: a branch around the loop, not a select per look-up)
            auto mix = [&](auto rot_c) {
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const unsigned li = ((th + (1u << 21)) >> 22) & 0x3ffu;
                const float2 sc2 = lut2[decltype(rot_c)::value ? w2_lut_slot_rot(li, A.lut_rot_sh, A.lut_rot_c)
                                                               : w2_lut_slot(li, A.lut_sh, A.lut_mask)];   // {sign*sin, cos}
                // (v.x c - v.y s, v.x s + v.y c) with every product and every sum rounded on its own (liquid's complex
                // multiply): the products as two packed multiplies — {v.x, v.y} * c and {v.y, v.x} * {-s, s}, whose swap
                // and sign are operand modifiers of FMUL2 — the sums as SCALAR adds: ptxas 12.9 contracts a packed
                // mul.rn.f32x2 into a packed add or fma that consumes it (one rounding instead of two), never into add.rn.f32
                const float2 v = unpk2(x[k]);
                const float2 t1 = unpk2(mul2(x[k], pk2(sc2.y, sc2.y)));
                const float2 t2 = unpk2(mul2(pk2(v.y, v.x), pk2(-sc2.x, sc2.x)));
                x[k] = pk2(__fadd_rn(t1.x, t2.x), __fadd_rn(t1.y, t2.y));
                th += p.nco_dtheta;
            }
            };
            // (the second copy of the loop exists in the cs16 kernels only: on the cu8 / table-DC kernel of cfg4 it cost 8 %
            // of the kernel whichever copy ran — session r3b; the host never picks a rotation for other formats)
            if (CS16 && A.lut_rot_c) mix(W2True{}); else mix(W2False{});
        }
    }
    if (!fast) {
        if (a0 < A.n0) {      // frames of an earlier call: already pre-processed, kept in the tail
#pragma unroll
            for (int k = 0; k < 16; k++) {
                if (a0 + k < A.n0) {
                    const long long j = a0 + k - (A.n0 - A.H_tail);
                    x[k] = (j >= 0) ? pk2(A.tail_in[j]) : 0ull;
                }
            }
        }
        if (write_tail && a0 + 16 > A.N1 - A.H_tail && a0 < A.N1) {
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const long long j = a0 + k - (A.N1 - A.H_tail);
                if (j >= 0 && a0 + k < A.N1) A.tail_out[j] = unpk2(x[k]);
            }
        }
    }
    if (P::reg0) return;            // the first halfband stage reads x[] straight from registers (w2_stage0_reg)
    if (S == 0) {
        ulonglong2* f = reinterpret_cast<ulonglong2*>(wsm + P::flat_off + w2_flat_phys(W2_ARB_HIST + 16 * lane, A.arb_skew_sh));
#pragma unroll
        for (int j = 0; j < 8; j++) f[j] = make_ulonglong2(x[2 * j], x[2 * j + 1]);
    } else {
        // level 0 planes: lane owns plane entries Hh + 8*lane .. +7 = one padded group of 8
        constexpr int c0 = P::Hh(0);
        float2* E = wsm + P::e_off(0) + (8 + P::PAD(0)) * lane;
        float2* O = wsm + P::o_off(0) + (8 + P::PAD(0)) * lane;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int ph = P::phys(0, c0 + 2 * j);
            *reinterpret_cast<ulonglong2*>(E + ph) = make_ulonglong2(x[4 * j], x[4 * j + 2]);
            *reinterpret_cast<ulonglong2*>(O + ph) = make_ulonglong2(x[4 * j + 1], x[4 * j + 3]);
        }
    }
}

// write the R outputs of stage D (lane owns outputs R*lane .. R*lane+R-1 of the run) to the next level's planes,
// or to the flat polyphase input when D is the last stage
template <int S, int D>
__device__ __forceinline__ void w2_stage_store(float2* __restrict__ wsm, int lane, int half, const f32x2_t (&v)[W2Plan<S>::R(D)],
                                               int skew_sh = 31)
{
    using P = W2Plan<S>;
    constexpr int R = P::R(D);
    if constexpr (D + 1 == S && R == 8) {
        // 64 contiguous bytes per lane: four STS.128 in lane order would put the 8 lanes of a quarter warp on two bank groups
        // (4-way conflict, 48 excess wavefronts per tick on cfg1).  Every lane starts with a different chunk instead — chunk
        // (j + rot) & 3 in instruction j, rot = (lane >> 1) & 3 — which covers all eight groups; the rotation of the register
        // chunks is a two-level select.
        if (!P::quad_skew) skew_sh = 31;
        float2* f = wsm + P::flat_off + w2_flat_phys(W2_ARB_HIST + R * lane, skew_sh);
        const unsigned rot = (skew_sh == 31) ? (((unsigned)lane >> 1) & 3u) : 0u;      // a skewed level is conflict free as it is
        const bool r1 = rot & 1u, r2 = rot & 2u;
        f32x2_t a[8], b[8];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            a[2 * c] = r1 ? v[(2 * c + 2) & 7] : v[2 * c];
            a[2 * c + 1] = r1 ? v[(2 * c + 3) & 7] : v[2 * c + 1];
        }
#pragma unroll
        for (int c = 0; c < 4; c++) {
            b[2 * c] = r2 ? a[(2 * c + 4) & 7] : a[2 * c];
            b[2 * c + 1] = r2 ? a[(2 * c + 5) & 7] : a[2 * c + 1];
        }
#pragma unroll
        for (int j = 0; j < 4; j++)
            *reinterpret_cast<ulonglong2*>(f + 2 * (((unsigned)j + rot) & 3u)) = make_ulonglong2(b[2 * j], b[2 * j + 1]);
    } else if constexpr (D + 1 == S && R == 4) {
        // 32 contiguous bytes per lane: two STS.128 in lane order put the 8 lanes of a quarter warp on four bank groups
        // (8 wavefronts instead of 4 per instruction, profiles/r03e_fused_front2_full_cfg3.md); lanes 4..7 of every eight
        // store their second chunk first
        if (!P::quad_skew) skew_sh = 31;
        float2* f = wsm + P::flat_off + w2_flat_phys(W2_ARB_HIST + R * lane, skew_sh);
        const bool rot = (skew_sh == 31) && (((unsigned)lane >> 2) & 1u);
        *reinterpret_cast<ulonglong2*>(f + (rot ? 2 : 0)) = make_ulonglong2(rot ? v[2] : v[0], rot ? v[3] : v[1]);
        *reinterpret_cast<ulonglong2*>(f + (rot ? 0 : 2)) = make_ulonglong2(rot ? v[0] : v[2], rot ? v[1] : v[3]);
    } else if constexpr (D + 1 == S) {
        if (!P::quad_skew) skew_sh = 31;
        float2* f = wsm + P::flat_off + w2_flat_phys(W2_ARB_HIST + R * lane, skew_sh);
        if (R >= 2) {
#pragma unroll
            for (int r = 0; r < R; r += 2) *reinterpret_cast<ulonglong2*>(f + r) = make_ulonglong2(v[r], v[r + 1]);
        } else *reinterpret_cast<f32x2_t*>(f) = v[0];
    } else if constexpr (P::ratio(D) == 1) {
        // the lane's R/2 (E, O) pairs are exactly one register group of the consumer
        constexpr int R2 = R / 2, HN = P::Hh(D + 1), PN = P::PAD(D + 1);
        static_assert(R2 == P::R(D + 1), "one producer lane feeds one consumer group");
        float2* nE = wsm + P::e_off(D + 1) + (R2 + PN) * lane;
        float2* nO = wsm + P::o_off(D + 1) + (R2 + PN) * lane;
        if (R2 >= 4 || (R2 == 2 && PN == 2)) {
#pragma unroll
            for (int i = 0; i < R2; i += 2) {
                const int ph = P::phys(D + 1, HN + i);
                *reinterpret_cast<ulonglong2*>(nE + ph) = make_ulonglong2(v[2 * i], v[2 * i + 2]);
                *reinterpret_cast<ulonglong2*>(nO + ph) = make_ulonglong2(v[2 * i + 1], v[2 * i + 3]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < R2; i++) {
                const int ph = P::phys(D + 1, HN + i);
                *reinterpret_cast<f32x2_t*>(nE + ph) = v[2 * i];
                *reinterpret_cast<f32x2_t*>(nO + ph) = v[2 * i + 1];
            }
        }
    } else {
        // the consumer takes two runs of this stage (`half` = which one this is): the lane's R/2 pairs are the lower
        // (even lane) or upper (odd lane) half of consumer group half*16 + lane/2
        constexpr int R2 = R / 2, RN = P::R(D + 1), HN = P::Hh(D + 1), PN = P::PAD(D + 1);
        static_assert(P::ratio(D) == 2 && RN == 2 * R2 && R >= 2, "capped stages keep their tile size");
        const int p0 = HN + half * (P::out(D) / 2) + R2 * lane;        // plane index of the lane's first pair
        const int ph0 = p0 + PN * (p0 / RN);
        float2* nE = wsm + P::e_off(D + 1) + ph0;
        float2* nO = wsm + P::o_off(D + 1) + ph0;
        if constexpr (R2 == 2 && PN == 2 && P::pair_fed(D + 1)) {
            // lanes 1, 9, 17, 25 would share a bank group with lanes 6, 14, ...: they store O first, E second (plane_size)
            const bool sw = (lane & 7) == 1;
            float2* pa = sw ? nO : nE;
            float2* pb = sw ? nE : nO;
            *reinterpret_cast<ulonglong2*>(pa) = make_ulonglong2(sw ? v[1] : v[0], sw ? v[3] : v[2]);
            *reinterpret_cast<ulonglong2*>(pb) = make_ulonglong2(sw ? v[0] : v[1], sw ? v[2] : v[3]);
        } else if constexpr (R2 == 1 && PN == 1 && P::pair_fed(D + 1)) {
            const unsigned l15 = (unsigned)lane & 15u;
            const bool sw = (l15 == 11u) || (l15 == 13u) || (l15 == 15u);
            *reinterpret_cast<f32x2_t*>(sw ? nO : nE) = sw ? v[1] : v[0];
            *reinterpret_cast<f32x2_t*>(sw ? nE : nO) = sw ? v[0] : v[1];
        } else if (R2 >= 2 && PN == 2) {
#pragma unroll
            for (int i = 0; i < R2; i += 2) {
                *reinterpret_cast<ulonglong2*>(nE + i) = make_ulonglong2(v[2 * i], v[2 * i + 2]);
                *reinterpret_cast<ulonglong2*>(nO + i) = make_ulonglong2(v[2 * i + 1], v[2 * i + 3]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < R2; i++) {
                *reinterpret_cast<f32x2_t*>(nE + i) = v[2 * i];
                *reinterpret_cast<f32x2_t*>(nO + i) = v[2 * i + 1];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// first halfband stage (semi-length 3) straight from registers.  The lane's 16 frames are 8 (E, O) pairs of
// level 0, i.e. exactly the inputs of its own 8 outputs; the 5 older E entries and 3 older O entries an output
// window reaches back to belong to the lane below and come by warp shuffle, lane 0 takes them from a 64-byte
// history that lane 31 left in shared memory one tick earlier.  This replaces the level-0 planes (a 4 KiB
// store + a 5 KiB load per tick and warp) by 16 shuffles; the arithmetic and its order are those of w2_stage.
// ------------------------------------------------------------------------------------------------
// the same for a first stage of semi-length 5 (S == 2): 9 older E entries (8 from the lane below, 1 from the lane below
// that) and 5 older O entries; lanes 0 and 1 take theirs from the 112-byte history lanes 31 and 30 left one tick earlier
// p ? a : b on both halves of a packed pair (two SELs, no moves)
__device__ __forceinline__ f32x2_t w2_sel(bool p, f32x2_t a, f32x2_t b)
{
    const unsigned lo = p ? (unsigned)a : (unsigned)b;
    const unsigned hi = p ? (unsigned)(a >> 32) : (unsigned)(b >> 32);
    return ((unsigned long long)hi << 32) | lo;
}

template <int S>
__device__ __forceinline__ void w2_stage0_reg_m5(const Fused2Args& A, float2* __restrict__ wsm, int lane, const f32x2_t (&x)[16],
                                                 f32x2_t (&v)[8])
{
    using P = W2Plan<S>;
    static_assert(P::m(0) == 5 && P::R(0) == 8, "semi-length 5, 8 outputs per lane");
    f32x2_t ent[17], oc[8];
    ent[0] = __shfl_up_sync(0xffffffffu, x[14], 2);                                         // E[q0-9]
#pragma unroll
    for (int k = 0; k < 8; k++) ent[1 + k] = __shfl_up_sync(0xffffffffu, x[2 * k], 1);      // E[q0-8 .. q0-1]
#pragma unroll
    for (int k = 0; k < 5; k++) oc[k] = __shfl_up_sync(0xffffffffu, x[7 + 2 * k], 1);       // O[q0-5 .. q0-1]
    // history (f32x2 entries): [0..7] lane 31's E[0..7], [8..12] lane 31's O[3..7], [13] lane 30's E[7]
    ulonglong2* hist = reinterpret_cast<ulonglong2*>(wsm + P::e_off(0));
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; k++) { const ulonglong2 h = hist[k]; ent[1 + 2 * k] = h.x; ent[2 + 2 * k] = h.y; }
        const ulonglong2 h4 = hist[4], h5 = hist[5], h6 = hist[6];
        oc[0] = h4.x; oc[1] = h4.y; oc[2] = h5.x; oc[3] = h5.y; oc[4] = h6.x; ent[0] = h6.y;
    }
    if (lane == 1) ent[0] = reinterpret_cast<const f32x2_t*>(hist)[7];                     // lane 31's E[7] of the last tick
    __syncwarp();
    if (lane == 31) {
#pragma unroll
        for (int k = 0; k < 4; k++) hist[k] = make_ulonglong2(x[4 * k], x[4 * k + 2]);
        hist[4] = make_ulonglong2(x[7], x[9]);
        hist[5] = make_ulonglong2(x[11], x[13]);
        reinterpret_cast<f32x2_t*>(hist)[12] = x[15];
    }
    if (lane == 30) reinterpret_cast<f32x2_t*>(hist)[13] = x[14];
#pragma unroll
    for (int k = 0; k < 8; k++) ent[9 + k] = x[2 * k];
#pragma unroll
    for (int k = 0; k < 3; k++) oc[5 + k] = x[2 * k + 1];
    f32x2_t acc[8];
#pragma unroll
    for (int r = 0; r < 8; r++) acc[r] = 0ull;
#pragma unroll
    for (int j = 0; j < 10; j++) {
        const float h = A.taps[P::taps_off(0) + j];
        const f32x2_t hh = pk2(h, h);
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = fma2(hh, ent[r + j], acc[r]);
    }
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = add2(oc[r], acc[r]);
    w2_stage_store<S, 0>(wsm, lane, 0, v, A.arb_skew_sh);
}

template <int S>
__device__ __forceinline__ void w2_stage0_reg(const Fused2Args& A, float2* __restrict__ wsm, int lane, const f32x2_t (&x)[16],
                                              f32x2_t (&v)[8])
{
    using P = W2Plan<S>;
    if constexpr (P::m(0) == 5) { w2_stage0_reg_m5<S>(A, wsm, lane, x, v); return; }
    else {
    static_assert(P::m(0) == 3 && P::R(0) == 8, "register first stage: semi-length 3, 8 outputs per lane");
    f32x2_t ent[13], oc[8];
    ulonglong2* hist = reinterpret_cast<ulonglong2*>(wsm + P::e_off(0));                    // level-0 planes are unused
    {
        // every lane reads the history (one broadcast wavefront per load, as a load by lane 0 alone would cost) and lane 0
        // keeps it through a select: the predicated form cost four register moves per entry (profiles/r02i: 71 of 658
        // instructions per tick were moves)
        const ulonglong2 h0 = hist[0], h1 = hist[1], h2 = hist[2], h3 = hist[3];
        const bool l0 = lane == 0;
        ent[0] = w2_sel(l0, h0.x, __shfl_up_sync(0xffffffffu, x[6], 1));                    // E[q0-5 .. q0-1]
        ent[1] = w2_sel(l0, h0.y, __shfl_up_sync(0xffffffffu, x[8], 1));
        ent[2] = w2_sel(l0, h1.x, __shfl_up_sync(0xffffffffu, x[10], 1));
        ent[3] = w2_sel(l0, h1.y, __shfl_up_sync(0xffffffffu, x[12], 1));
        ent[4] = w2_sel(l0, h2.x, __shfl_up_sync(0xffffffffu, x[14], 1));
        oc[0] = w2_sel(l0, h2.y, __shfl_up_sync(0xffffffffu, x[11], 1));                    // O[q0-3 .. q0-1]
        oc[1] = w2_sel(l0, h3.x, __shfl_up_sync(0xffffffffu, x[13], 1));
        oc[2] = w2_sel(l0, h3.y, __shfl_up_sync(0xffffffffu, x[15], 1));
    }
    __syncwarp();
    if (lane == 31) {
        hist[0] = make_ulonglong2(x[6], x[8]);
        hist[1] = make_ulonglong2(x[10], x[12]);
        hist[2] = make_ulonglong2(x[14], x[11]);
        hist[3] = make_ulonglong2(x[13], x[15]);
    }
#pragma unroll
    for (int k = 0; k < 8; k++) ent[5 + k] = x[2 * k];
#pragma unroll
    for (int k = 0; k < 5; k++) oc[3 + k] = x[2 * k + 1];
    f32x2_t acc[8];
#pragma unroll
    for (int r = 0; r < 8; r++) acc[r] = 0ull;
#pragma unroll
    for (int j = 0; j < 6; j++) {
        const float h = A.taps[P::taps_off(0) + j];
        const f32x2_t hh = pk2(h, h);
#pragma unroll
        for (int r = 0; r < 8; r++) acc[r] = fma2(hh, ent[r + j], acc[r]);
    }
#pragma unroll
    for (int r = 0; r < 8; r++) v[r] = add2(oc[r], acc[r]);
    if (!P::reg1) w2_stage_store<S, 0>(wsm, lane, 0, v, A.arb_skew_sh);
    }
}

// second halfband stage (semi-length 3, 4 outputs per lane) from the first stage's outputs in registers:
//   E1[j] = v[2j], O1[j] = v[2j+1] (j < 4) are the lane's level-1 pairs; an output window reaches back 5 E entries (4 from
//   the lane below, 1 from the lane below that) and 3 O entries (lane below).  Lanes 0 and 1 take theirs from the 64-byte
//   history lanes 31 and 30 left one tick earlier.  Replaces the level-1 planes by 16 shuffles.
template <int S>
__device__ __forceinline__ void w2_stage1_reg(const Fused2Args& A, float2* __restrict__ wsm, int lane, int half, const f32x2_t (&v)[8])
{
    using P = W2Plan<S>;
    static_assert(P::m(1) == 3 && P::R(1) == 4, "register second stage: semi-length 3, 4 outputs per lane");
    f32x2_t ent[9], oc[4];
    ulonglong2* hist = reinterpret_cast<ulonglong2*>(wsm + P::e_off(1));                    // level-1 planes are unused
    // history: [0..3] = lane 31's E1[0..3], [4..6] = lane 31's O1[1..3], [7] = lane 30's E1[3]
    {
        const ulonglong2 h0 = hist[0], h1 = hist[1], h2 = hist[2], h3 = hist[3];            // broadcast loads, selects (w2_stage0_reg)
        const bool l0 = lane == 0, l1 = lane == 1;
        // E1[q0-5]: lane 0 takes lane 30's E1[3], lane 1 lane 31's E1[3] of the last tick
        ent[0] = w2_sel(l0, h3.y, w2_sel(l1, h1.y, __shfl_up_sync(0xffffffffu, v[6], 2)));
        ent[1] = w2_sel(l0, h0.x, __shfl_up_sync(0xffffffffu, v[0], 1));                    // E1[q0-4 .. q0-1]
        ent[2] = w2_sel(l0, h0.y, __shfl_up_sync(0xffffffffu, v[2], 1));
        ent[3] = w2_sel(l0, h1.x, __shfl_up_sync(0xffffffffu, v[4], 1));
        ent[4] = w2_sel(l0, h1.y, __shfl_up_sync(0xffffffffu, v[6], 1));
        oc[0] = w2_sel(l0, h2.x, __shfl_up_sync(0xffffffffu, v[3], 1));                     // O1[q0-3 .. q0-1]
        oc[1] = w2_sel(l0, h2.y, __shfl_up_sync(0xffffffffu, v[5], 1));
        oc[2] = w2_sel(l0, h3.x, __shfl_up_sync(0xffffffffu, v[7], 1));
    }
    __syncwarp();
    if (lane == 31) {
        hist[0] = make_ulonglong2(v[0], v[2]);
        hist[1] = make_ulonglong2(v[4], v[6]);
        hist[2] = make_ulonglong2(v[3], v[5]);
        reinterpret_cast<f32x2_t*>(hist)[6] = v[7];
    }
    if (lane == 30) reinterpret_cast<f32x2_t*>(hist)[7] = v[6];
#pragma unroll
    for (int k = 0; k < 4; k++) ent[5 + k] = v[2 * k];
    oc[3] = v[1];
    f32x2_t acc[4];
#pragma unroll
    for (int r = 0; r < 4; r++) acc[r] = 0ull;
#pragma unroll
    for (int j = 0; j < 6; j++) {
        const float h = A.taps[P::taps_off(1) + j];
        const f32x2_t hh = pk2(h, h);
#pragma unroll
        for (int r = 0; r < 4; r++) acc[r] = fma2(hh, ent[r + j], acc[r]);
    }
    f32x2_t y[4];
#pragma unroll
    for (int r = 0; r < 4; r++) y[r] = add2(oc[r], acc[r]);
    w2_stage_store<S, 1>(wsm, lane, half, y, A.arb_skew_sh);
}

// ------------------------------------------------------------------------------------------------
// one halfband decimator run (liquid resamp2_crcf_decim_execute):
//   y[q] = ( O[q-m] + sum_{j<2m} h1[j] E[q-2m+1+j] ) * scale       (plane-local indices)
// lane owns outputs q0 = R*lane .. q0+R-1.
// ------------------------------------------------------------------------------------------------
template <int S, int D>
__device__ __forceinline__ void w2_stage(const Fused2Args& A, float2* __restrict__ wsm, int lane, int half)
{
    using P = W2Plan<S>;
    constexpr int M = P::m(D), R = P::R(D), HH = P::Hh(D), PADD = P::PAD(D);
    constexpr int NE = 2 * M + R - 1;                 // E entries a lane reads
    constexpr int CE = HH - (2 * M - 1);              // plane index (before + R*lane) of the first one
    constexpr int CO = HH - M;                        // plane index of O[q0 - m]
    constexpr bool VEC = (R >= 4);                    // padded layouts keep even-aligned pairs 16-byte aligned
    const float2* __restrict__ E = wsm + P::e_off(D) + (R + PADD) * lane;
    const float2* __restrict__ O = wsm + P::o_off(D) + (R + PADD) * lane;
    // samples are kept as packed {re, im} pairs: every tap multiplies both halves, so one FFMA2 does the
    // work of two FFMAs (bit-identical: each half is an IEEE fma)
    f32x2_t ent[NE], oc[R];
    // even-aligned pairs of a padded plane are 16-byte aligned: one LDS.128 per pair
#pragma unroll
    for (int e = 0; e < NE; e++) {
        const int c = CE + e;
        const bool first = VEC && (c % 2 == 0) && (e + 1 < NE);
        const bool second = VEC && (c % 2 != 0) && (e >= 1);
        if (first) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(E + P::phys(D, c));
            ent[e] = v.x;
            ent[e + 1] = v.y;
        } else if (!second) ent[e] = *reinterpret_cast<const f32x2_t*>(E + P::phys(D, c));
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int c = CO + r;
        const bool first = VEC && (c % 2 == 0) && (r + 1 < R);
        const bool second = VEC && (c % 2 != 0) && (r >= 1);
        if (first) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(O + P::phys(D, c));
            oc[r] = v.x;
            oc[r + 1] = v.y;
        } else if (!second) oc[r] = *reinterpret_cast<const f32x2_t*>(O + P::phys(D, c));
    }
    f32x2_t acc[R];
#pragma unroll
    for (int r = 0; r < R; r++) acc[r] = 0ull;
#pragma unroll
    for (int j = 0; j < 2 * M; j++) {
        const float h = A.taps[P::taps_off(D) + j];
        const f32x2_t hh = pk2(h, h);
#pragma unroll
        for (int r = 0; r < R; r++) acc[r] = fma2(hh, ent[r + j], acc[r]);
    }
    f32x2_t v[R];
    const f32x2_t zz = pk2(A.zeta, A.zeta);
#pragma unroll
    for (int r = 0; r < R; r++) {
        if (D + 1 == S) v[r] = mul2(add2(oc[r], acc[r]), zz);
        else v[r] = add2(oc[r], acc[r]);
    }
    w2_stage_store<S, D>(wsm, lane, half, v, A.arb_skew_sh);
}

// move the last Hh entries of both planes of level D to the history slots (all lanes call).  The loads are
// issued together with the stage's own loads (the tail is not touched by the stage), the stores after the
// stage's __syncwarp, so the copy adds no exposed shared-memory round trip.
template <int S, int D>
struct W2Slide {
    using P = W2Plan<S>;
    static constexpr int HH = P::Hh(D), N = P::out(D);
    static_assert(2 * HH <= 64, "history too long for the two-round slide");
    f32x2_t t = 0ull, t2 = 0ull;
    f32x2_t *pl, *pl2;
    int i, i2;
    bool act, act2;
    __device__ __forceinline__ W2Slide(float2* __restrict__ wsm, int lane)
    {
        pl = reinterpret_cast<f32x2_t*>(wsm + ((lane < HH) ? P::e_off(D) : P::o_off(D)));
        i = (lane < HH) ? lane : lane - HH;
        act = lane < 2 * HH;
        pl2 = reinterpret_cast<f32x2_t*>(wsm + ((lane + 32 < HH) ? P::e_off(D) : P::o_off(D)));
        i2 = (lane + 32 < HH) ? lane + 32 : lane + 32 - HH;
        act2 = (2 * HH > 32) && (lane + 32 < 2 * HH);
        if (act) t = pl[P::phys(D, i + N)];
        if (act2) t2 = pl2[P::phys(D, i2 + N)];
    }
    __device__ __forceinline__ void store() const
    {
        if (act) pl[P::phys(D, i)] = t;
        if (act2) pl2[P::phys(D, i2)] = t2;
    }
};

// ------------------------------------------------------------------------------------------------
// polyphase stage, FOUR consecutive outputs per lane (arb_pairs == 2).  The stage is bound by the LSU data pipe (97 % of its
// wavefront peak on cfg1, profiles/r02a_fused_front2_cfg1.md): one output per lane loads 14 window entries (LDS.64 whose lanes
// are 1.3 .. 1.7 entries apart: 2 x the ideal wavefronts) and 14 taps (7 LDS.64 from rows a configuration-dependent stride
// apart: another 2 x).  Here the windows of outputs o .. o+3 start k_q - k_0 = 0, {1,2}, {B2, B2+1}, {B3, B3+1} entries apart
// (rate in [0.5, 1)), so ONE register window of 15 + B3 entries serves all four, and the rows come as four LDS.128 each from
// an image in which row r sits at rotr8(r, tz) with its four 16-byte chunks XOR-permuted — tz chosen on the host so that the
// eight lanes of a quarter warp, whose rows advance by (4 step >> 16) mod 256, fall into eight different bank groups.
// Output q reads its taps shifted by e_q = (k_q - k_0) - Bq in {0, 1} through a select (T[j] = e ? f[j-1] : f[j]; the taps
// that fall outside the row are exact zeros, the non-zero terms keep the reference's order: same bits as one output per lane).
// ------------------------------------------------------------------------------------------------
constexpr int W2_QBANK_ROW_F = 16;            // floats per row of the image: 14 taps + 2 zeros
__host__ __device__ constexpr unsigned w2_qbank_rot(unsigned r, unsigned tz) { return ((r >> tz) | (r << (8u - tz))) & 255u; }
// float offset of logical chunk j (4 floats) of row r
__host__ __device__ constexpr unsigned w2_qbank_chunk(unsigned r, unsigned tz, unsigned j)
{
    return 16u * w2_qbank_rot(r, tz) + 4u * (j ^ ((w2_qbank_rot(r, tz) >> 1) & 3u));
}
__host__ static inline unsigned w2_pick_qbank_tz(uint32_t step)
{
    unsigned best_tz = 0;
    double best = 1e30;
    for (unsigned tz = 0; tz < 8; tz++) {
        double cost = 0;
        for (unsigned trial = 0; trial < 256; trial++) {
            const unsigned long long o0 = 4ull * (trial * 977ull + 13ull);
            for (int quarter = 0; quarter < 4; quarter++)
                for (int q = 0; q < 4; q++)
                    for (unsigned j = 0; j < 4; j++) {
                        int hits[8] = {0};
                        unsigned seen[8];
                        int deg = 0;
                        for (int l = 0; l < 8; l++) {
                            const unsigned long long o = o0 + 4ull * (unsigned)(8 * quarter + l) + (unsigned)q;
                            const unsigned r = (unsigned)((o * step) >> 16) & 255u;
                            const unsigned off = w2_qbank_chunk(r, tz, j);
                            seen[l] = off;
                            bool dup = false;
                            for (int m = 0; m < l; m++) dup |= (seen[m] == off);
                            if (dup) continue;
                            const unsigned slot = (off >> 2) & 7u;
                            if (++hits[slot] > deg) deg = hits[slot];
                        }
                        cost += deg;
                    }
        }
        if (cost < best - 1e-9) { best = cost; best_tz = tz; }
    }
    return best_tz;
}

// shared-memory wavefronts of the four-output variant's window loads (LDS.64, half warps of 16 lanes) for a given skew
__host__ static inline double w2_window_cost(uint32_t step, int sh)
{
    double cost = 0;
    for (unsigned trial = 0; trial < 128; trial++) {
        const unsigned long long o0 = 4ull * (trial * 7919ull + 5ull);
        const long long kbase = (long long)((o0 * step) >> 24);
        for (int half = 0; half < 2; half++) {
            int cnt[32] = {0};
            int deg = 0;
            for (int l = 0; l < 16; l++) {
                const unsigned long long o = o0 + 4ull * (unsigned)(16 * half + l);
                const int e = (int)((long long)((o * step) >> 24) - kbase) + 3;
                const int ph = w2_flat_phys(e, sh);
                for (int w = 0; w < 2; w++) { const int b = (2 * ph + w) & 31; if (++cnt[b] > deg) deg = cnt[b]; }
            }
            cost += deg;
        }
    }
    return cost;
}
__host__ static inline int w2_pick_flat_skew(uint32_t step)
{
    const int cand[3] = {31, 4, 5};
    int best = 31;
    double bc = 1e30;
    for (int c = 0; c < 3; c++) {
        const double k = w2_window_cost(step, cand[c]);
        if (k < bc * 0.97) { bc = k; best = cand[c]; }       // a skew has to pay for its address arithmetic
    }
    return best;
}

template <int B2, int B3, bool SKEW>
__device__ __forceinline__ void w2_arb_quad(const Fused2Args& A, const float2* __restrict__ flat, const float2* __restrict__ sbank,
                                            long long kA, long long oa, long long ob, int lane)
{
    const unsigned long long step = A.step;
    const unsigned tz = (unsigned)A.arb_tz;
    const float* __restrict__ bank = reinterpret_cast<const float*>(sbank);
    constexpr int NU = 15 + B3;                         // window entries: output 3 reaches index B3 + 1 + 13
    const long long kA_rel = kA - A.arb_pos.k_base;
    for (long long o = oa + 4 * lane; o < ob; o += 128) {
        // relative to the launch's base (ArbBase): P0..P3 never wrap, so the steps e1..e3 are right wherever o * step would
        const unsigned long long P0 = (unsigned long long)o * step - A.arb_pos.p_base, P1 = P0 + step, P2 = P1 + step, P3 = P2 + step;
        const long long k0 = (long long)(P0 >> 24);
        const int rel = (int)(k0 - kA_rel);
        const bool e1 = ((long long)(P1 >> 24) - k0) != 1;
        const bool e2 = ((long long)(P2 >> 24) - k0) != B2;
        const bool e3 = ((long long)(P3 >> 24) - k0) != B3;
        const f32x2_t* __restrict__ w = reinterpret_cast<const f32x2_t*>(flat);
        const int e0 = rel + (W2_ARB_HIST - 13);
        f32x2_t u[NU];
        if constexpr (SKEW) {
            const int ssh = A.arb_skew_sh;
#pragma unroll
            for (int j = 0; j < NU; j++) u[j] = w[w2_flat_phys(e0 + j, ssh)];
            // (two thresholds on one base register instead of a shift and an add per load, and a separate loop for
            // ssh == 31, measured SLOWER: cfg1 0.437 -> 0.469 ms, session r2y — the selects cost what the shifts did and
            // the second copy of the loop cost registers)
        } else {                                            // plain level: one base register, immediate offsets
#pragma unroll
            for (int j = 0; j < NU; j++) u[j] = w[e0 + j];
        }
        f32x2_t s[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const unsigned long long Pq = (q == 0) ? P0 : (q == 1 ? P1 : (q == 2 ? P2 : P3));
            const unsigned r = (unsigned)(Pq >> 16) & 255u;
            const unsigned pr = w2_qbank_rot(r, tz);
            const float* __restrict__ row = bank + 16u * pr;
            const unsigned sw = (pr >> 1) & 3u;
            float f[17];
            f[0] = 0.f;                                     // f[1 + i] = tap i; f[15], f[16] = the row's zero padding
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float4 c = *reinterpret_cast<const float4*>(row + 4u * ((unsigned)j ^ sw));
                f[1 + 4 * j] = c.x; f[2 + 4 * j] = c.y; f[3 + 4 * j] = c.z; f[4 + 4 * j] = c.w;
            }
            f32x2_t acc = 0ull;
            if (q == 0) {
#pragma unroll
                for (int i = 0; i < 14; i++) acc = fma2s(f[1 + i], u[i], acc);
            } else {
                const bool e = (q == 1) ? e1 : (q == 2 ? e2 : e3);
                const int base = (q == 1) ? 1 : (q == 2 ? B2 : B3);
#pragma unroll
                for (int j = 0; j < 15; j++) acc = fma2s(e ? f[j] : f[j + 1], u[base + j], acc);   // tap j - e of the row
            }
            s[q] = acc;
        }
#pragma unroll
        for (int q = 0; q < 4; q++)
            if (o + q < ob) *reinterpret_cast<f32x2_t*>(A.y + (o + q - A.O0)) = s[q];
    }
}

// ------------------------------------------------------------------------------------------------
// polyphase arbitrary-rate stage (liquid resamp_crcf, fixed-point phase) on the new flat entries
//   output o: P = o*step, k = P >> 24, bank row = (P >> 16) & 255, y = sum_{i<14} row[i] * x[k-13+i]
// ------------------------------------------------------------------------------------------------
// o_cur = first output whose push index is >= kA (carried from run to run: one exact 64-bit
// division per warp at start, then a float estimate + integer fix-up per run).
template <int S>
__device__ __forceinline__ void w2_arb(const Fused2Args& A, const float2* __restrict__ flat, const float2* __restrict__ sbank,
                                       long long kA, long long& o_cur, int lane)
{
    using P = W2Plan<S>;
    const unsigned long long step = A.step;
    const unsigned long long kb = (unsigned long long)kA + P::flat_new;
    // outputs of this run: o >= o_cur with o*step < kb << 24.  Both products may wrap mod 2^64; their true difference lies
    // in (0, (flat_new+2) << 24], so the difference mod 2^64 is exact.
    const unsigned long long Dn = (kb << 24) - (unsigned long long)o_cur * step;
    // cnt = ceil(Dn / step): float estimate of the quotient (Dn < 2^34, step in [2^24, 2^25]: off by at most one),
    // then an exact remainder fix-up without loops
    unsigned cnt = (unsigned)__fdividef((float)Dn, (float)step);
    long long rem = (long long)Dn - (long long)((unsigned long long)cnt * step);
    if (rem < 0) { cnt--; rem += (long long)step; }
    if (rem >= (long long)step) { cnt++; rem -= (long long)step; }
    cnt += (rem > 0) ? 1u : 0u;
    long long oa = o_cur, ob = o_cur + cnt;
    o_cur = ob;
    if (oa < A.O0) oa = A.O0;
    if (ob > A.O1) ob = A.O1;
    if (P::quad && A.arb_pairs == 2) {
        if (A.arb_b2 == 2) {
            if (A.arb_b3 == 3) w2_arb_quad<2, 3, P::quad_skew>(A, flat, sbank, kA, oa, ob, lane);
            else w2_arb_quad<2, 4, P::quad_skew>(A, flat, sbank, kA, oa, ob, lane);
        } else {
            if (A.arb_b3 == 4) w2_arb_quad<3, 4, P::quad_skew>(A, flat, sbank, kA, oa, ob, lane);
            else w2_arb_quad<3, 5, P::quad_skew>(A, flat, sbank, kA, oa, ob, lane);
        }
        return;
    }
    // o * step relative to the launch's base (ArbBase, o >= oa >= O0): exact k and row at any stream position
    const long long kA_rel = kA - A.arb_pos.k_base;
    const unsigned long long p_base = A.arb_pos.p_base;
    if (!A.arb_pairs) {
    for (long long o = oa + lane; o < ob; o += 32) {
        const unsigned long long Pp = (unsigned long long)o * step - p_base;
        const int rel = (int)((long long)(Pp >> 24) - kA_rel);
        const unsigned idx = (unsigned)(Pp >> 16) & 0xffu;
        const float2* __restrict__ w = flat + rel + (W2_ARB_HIST - 13);
        const float2* __restrict__ b = sbank + w2_bank_row((int)idx);
        f32x2_t sacc = 0ull;
#pragma unroll
        for (int i = 0; i < 7; i++) {
            const float2 h = b[i];
            const f32x2_t v0 = *reinterpret_cast<const f32x2_t*>(w + 2 * i), v1 = *reinterpret_cast<const f32x2_t*>(w + 2 * i + 1);
            sacc = fma2s(h.x, v0, sacc);
            sacc = fma2s(h.y, v1, sacc);
        }
        *reinterpret_cast<f32x2_t*>(A.y + (o - A.O0)) = sacc;
    }
        return;
    }
    // A lane makes TWO consecutive outputs o, o+1.  Their windows x[k-13 .. k] start d = k(o+1) - k(o) = 1 or 2 entries apart
    // (the rate of the arbitrary stage lies in [0.5, 1)), so 16 window entries serve both instead of 28; the second
    // output reads its row from two floats in front of it (rows are separated by >= 4 floats of zeros) and shifts it by d,
    // which lines its taps up with the shared window: taps that fall outside the row are exact zeros, the order of the
    // non-zero terms is that of a single output, hence the same bits.
    for (long long o = oa + 2 * lane; o < ob; o += 64) {
        const unsigned long long P0 = (unsigned long long)o * step - p_base, P1 = P0 + step;
        const int rel = (int)((long long)(P0 >> 24) - kA_rel);
        const int d = (int)((P1 >> 24) - (P0 >> 24));
        const f32x2_t* __restrict__ w = reinterpret_cast<const f32x2_t*>(flat + rel + (W2_ARB_HIST - 13));
        const float2* __restrict__ b0 = sbank + w2_bank_row((int)((unsigned)(P0 >> 16) & 0xffu));
        // row of the second output from one float2 (two zeros) in front of it: 8 LDS.64 with the conflict-free pattern of
        // the first row; the shift by d floats is a select between neighbours
        const float2* __restrict__ b1 = sbank + w2_bank_row((int)((unsigned)(P1 >> 16) & 0xffu)) - 1;
        f32x2_t u[16];
#pragma unroll
        for (int j = 0; j < 16; j++) u[j] = w[j];
        f32x2_t s0 = 0ull, s1 = 0ull;
#pragma unroll
        for (int i = 0; i < 7; i++) {
            const float2 h = b0[i];
            s0 = fma2s(h.x, u[2 * i], s0);
            s0 = fma2s(h.y, u[2 * i + 1], s0);
        }
        float f1[17];
#pragma unroll
        for (int i = 0; i < 8; i++) { const float2 h = b1[i]; f1[2 * i] = h.x; f1[2 * i + 1] = h.y; }
        f1[16] = 0.f;
        const bool d2 = (d == 2);
#pragma unroll
        for (int j = 0; j < 16; j++) s1 = fma2s(d2 ? f1[j] : f1[j + 1], u[j], s1);     // tap j - d of the row (zero outside it)
        *reinterpret_cast<f32x2_t*>(A.y + (o - A.O0)) = s0;
        if (o + 1 < ob) *reinterpret_cast<f32x2_t*>(A.y + (o + 1 - A.O0)) = s1;
    }
}

template <int S, int D>
struct W2Cascade {
    // run stage D (and everything below it) for tick `t` (absolute tick index)
    static __device__ __forceinline__ void run(const Fused2Args& A, float2* __restrict__ wsm, long long t, int lane, bool& arb_due)
    {
        using P = W2Plan<S>;
        constexpr int PER = P::period(D);
        if (PER > 1 && ((t & (PER - 1)) != (PER - 1))) { arb_due = false; return; }
        // which of the consumer's two feeding runs this is (stages whose consumer waits for two runs)
        int half = 0;
        if constexpr (D + 1 < S) {
            if (P::ratio(D) == 2) half = (int)((t >> w2_ilog2(PER)) & 1);     // arithmetic shift: t may be negative during warm-up
        }
        const W2Slide<S, D> slide(wsm, lane);
        w2_stage<S, D>(A, wsm, lane, half);
        __syncwarp();
        slide.store();
        __syncwarp();
        if constexpr (D + 1 < S) W2Cascade<S, D + 1>::run(A, wsm, t, lane, arb_due);
    }
};

template <int S, int DC, bool CS16>
__global__ void __launch_bounds__(W2_MAX_WARPS * 32, 1) fused_front2_kernel(const __grid_constant__ Fused2Args A, int warps_per_cta)
{
    using P = W2Plan<S>;
    extern __shared__ __align__(16) float2 sm2_base[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // shared tables: polyphase bank image (TMA bulk copy), NCO table {sign*sin, cos}[1024]
    __shared__ __align__(8) uint64_t tma_bar;
    __shared__ __align__(8) uint64_t raw_bar[W2_MAX_WARPS];
    // per-warp raw tick buffers first (the 128-byte swizzle repeats every 1 KiB: 1 KiB-aligned), cs16 kernels only
    unsigned char* dyn = reinterpret_cast<unsigned char*>(sm2_base);
    unsigned char* rawbuf = nullptr;
    if (CS16) {
        const unsigned a = w2_smem_u32(dyn);
        dyn += ((a + 1023u) & ~1023u) - a;
        rawbuf = dyn + warp * W2_RAW_TICK_BYTES;
        dyn += warps_per_cta * W2_RAW_TICK_BYTES;
    }
    float2* sm2 = reinterpret_cast<float2*>(dyn);
    float2* sbank = sm2;
    float2* lut2 = sm2 + W2_BANK_F2;
    float2* wsm = lut2 + (A.pre.nco_enable ? 1024 : 0) + warp * P::warp_f2;
    if (tid == 0) w2_mbar_init(&tma_bar, 1);
    if (CS16 && lane == 0) w2_mbar_init(&raw_bar[warp], 1);
    __syncthreads();
    if (tid == 0) w2_tma_load(sbank, A.bank_image, W2_BANK_F2 * sizeof(float2), &tma_bar);
    if (A.pre.nco_enable)
        for (int i = tid; i < 1024; i += blockDim.x)
            lut2[A.lut_rot_c ? w2_lut_slot_rot((unsigned)i, A.lut_rot_sh, A.lut_rot_c) : w2_lut_slot((unsigned)i, A.lut_sh, A.lut_mask)] = make_float2(A.pre.nco_table[i] * A.pre.nco_sign, A.pre.nco_table[(i + 256) & 1023]);
    for (int i = lane; i < P::warp_f2; i += 32) wsm[i] = make_float2(0.f, 0.f);
    w2_mbar_wait(&tma_bar, 0);
    __syncthreads();

    const long long gw = (long long)blockIdx.x * warps_per_cta + warp;
    const long long seg_first = A.sup_first + gw * A.sup_per_warp;       // in super-ticks
    if (seg_first > A.sup_last) return;
    long long seg_last = seg_first + A.sup_per_warp - 1;
    if (seg_last > A.sup_last) seg_last = A.sup_last;
    float2* flat = wsm + P::flat_off;

    const long long t_begin = (seg_first - A.warm_sup) * P::sup, t_emit = seg_first * P::sup, t_end = (seg_last + 1) * P::sup;
    // first output of the first emitting run, o_cur = ceil(k_emit 2^24 / step), carried from run to run afterwards; as an
    // offset from O0: D = k_emit 2^24 - O0 step = (k_emit - k_base) 2^24 - (O0 step mod 2^24), within the call (any sign)
    long long o_cur;
    {
        const long long k_emit = (t_emit * W2_T0) >> S;
        const long long step = (long long)A.step;
        const long long D = ((k_emit - A.arb_pos.k_base) << 24) - (long long)(((unsigned long long)A.O0 * A.step) & 0xffffffull);
        o_cur = A.O0 + (D >= 0 ? (D + step - 1) / step : -((-D) / step));
    }
    double2 vloc = make_double2(0.0, 0.0);
    if (DC == 2 && gw == 0) {
        // the warp that holds n0 starts from the carried state, rewound through the (zero) frames in front of n0
        const double2 cv = *A.dc_carry;
        const double f = exp(-(double)(A.n0 - t_begin * W2_T0) * A.dc_lnc);
        vloc = make_double2(cv.x * f, cv.y * f);
    }
    // Per-tick bookkeeping in 32-bit tick numbers relative to t_begin (the 64-bit range tests of every tick were 8 % of the
    // kernel's instructions in profiles/r02f_fused_front2_cfg2.md): ticks [fast_lo, fast_hi) are "fast", [act_lo, act_hi) hold
    // frames of this call, emission starts at emit_r.
    const int n_ticks = (int)(t_end - t_begin), emit_r = (int)(t_emit - t_begin);
    int fast_lo = 0, fast_hi = 0, act_lo, act_hi;
    {
        const long long lo = (A.n0 + W2_T0 - 1) / W2_T0, hi = (A.N1 - A.H_tail) / W2_T0;      // tick_start >= n0, tick end <= N1 - H_tail
        if (A.raw_aligned && hi > lo) {
            fast_lo = (int)max(0LL, min((long long)n_ticks, lo - t_begin));
            fast_hi = (int)max(0LL, min((long long)n_ticks, hi - t_begin));
        }
        const long long alo = A.n0 / W2_T0, ahi = (A.N1 + W2_T0 - 1) / W2_T0;                 // tick end > n0, tick_start < N1
        act_lo = (int)max(0LL, min((long long)n_ticks, alo - t_begin));
        act_hi = (int)max(0LL, min((long long)n_ticks, ahi - t_begin));
    }
    const unsigned fast_len = (unsigned)max(0, fast_hi - fast_lo), act_len = (unsigned)max(0, act_hi - act_lo);
    // raw frames of a fast cs16 tick: staged one tick ahead by TMA (A.raw_tma) into the warp's buffer
    const bool use_tma = CS16 && A.raw_tma;
    bool staged = false;                    // a TMA load for the tick about to run is in flight / has landed (warp-uniform)
    unsigned raw_phase = 0;
    const int row0 = (int)((t_begin * W2_T0 - A.n0) >> 5);       // 128-byte row of tick 0 (meaningful for fast ticks only)
    if (use_tma && (unsigned)(0 - fast_lo) < fast_len) {
        if (lane == 0) w2_tma_load_tick(rawbuf, &A.raw_map, row0, &raw_bar[warp]);
        staged = true;
    }
    // the lane's four 16-byte chunks of its 64-byte run: chunk u = 4*lane + j sits in row u >> 3 at 16-byte slot (u & 7) ^ (row & 7)
    const unsigned raw_row = w2_smem_u32(rawbuf) + 128u * (unsigned)(lane >> 1);
    const unsigned raw_sw = (unsigned)(lane >> 1) & 7u, raw_c0 = 4u * (unsigned)(lane & 1);
    long long t = t_begin;
    // The body exists twice: ticks of the fast range (nearly all of them) run a copy in which `fast` and `active` are
    // compile-time true, i.e. without the range tests, the tail handling and the zero-fill of the general copy.
    auto tick = [&](auto fast_c, int tr) {
        constexpr bool FAST = decltype(fast_c)::value;
        const long long tick_start = t * W2_T0;
        const bool fast = FAST, active = FAST || ((unsigned)(tr - act_lo) < act_len);
        W2Raw cur;
        if (CS16) {
            if (staged) {
                w2_mbar_wait(&raw_bar[warp], raw_phase);
                raw_phase ^= 1u;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const unsigned addr = raw_row + 16u * ((raw_c0 + (unsigned)j) ^ raw_sw);
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(cur.q[j].x), "=r"(cur.q[j].y), "=r"(cur.q[j].z), "=r"(cur.q[j].w) : "r"(addr));
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) cur.q[j] = make_uint4(0u, 0u, 0u, 0u);
                if (fast) {                                       // unaligned call: plain loads, no look-ahead
                    const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(A.raw) + (tick_start - A.n0 + lane * 16) * 4);
#pragma unroll
                    for (int j = 0; j < 4; j++) cur.q[j] = __ldg(src + j);
                }
            }
        }
        if (DC == 2 && tr == emit_r && lane == 0) A.dc_stretch[gw].v_emit = vloc;
        f32x2_t x[16];
        // local DC: the frames of a warm-up tick belong to the emit range of the warp below, which stores them in the tail
        // with ITS state (warp 0's warm-up frames precede n0: copies of the old tail)
        w2_p0<S, DC, CS16>(A, wsm, lut2, tick_start, lane, cur, x, vloc, DC != 2 || tr >= emit_r || gw == 0, active, fast);
        if (use_tma) {
            // every lane has consumed its chunks (the conversions in w2_p0 depend on them): the buffer may be refilled
            __syncwarp();
            staged = (unsigned)(tr + 1 - fast_lo) < fast_len;     // (fast_hi <= n_ticks: never beyond the warp's last tick)
            if (staged && lane == 0) w2_tma_load_tick(rawbuf, &A.raw_map, row0 + 16 * (tr + 1), &raw_bar[warp]);
        }
        bool arb_due = true;
        if constexpr (P::reg0) {
            f32x2_t v0[8];
            w2_stage0_reg<S>(A, wsm, lane, x, v0);
            if constexpr (P::reg1) {
                // stage 1 runs every tick; its consumer may wait for two of its runs (capped plans)
                const int half = (P::ratio(1) == 2) ? (int)(t & 1) : 0;
                w2_stage1_reg<S>(A, wsm, lane, half, v0);
                __syncwarp();
                W2Cascade<S, 2>::run(A, wsm, t, lane, arb_due);
            } else {
                __syncwarp();
                W2Cascade<S, 1>::run(A, wsm, t, lane, arb_due);
            }
        } else {
            __syncwarp();
            if constexpr (S > 0) W2Cascade<S, 0>::run(A, wsm, t, lane, arb_due);
        }
        if (arb_due) {
            // the new flat entries are the last stage's outputs of this run: absolute decimated index
            const long long kA = ((tick_start + W2_T0) >> S) - P::flat_new;
            if (tr >= emit_r) w2_arb<S>(A, flat, sbank, kA, o_cur, lane);
            __syncwarp();
            float2 h = make_float2(0.f, 0.f);
            const int ssh = P::quad_skew ? A.arb_skew_sh : 31;
            if (lane < W2_ARB_HIST) h = flat[w2_flat_phys(lane + P::flat_new, ssh)];
            __syncwarp();
            if (lane < W2_ARB_HIST) flat[w2_flat_phys(lane, ssh)] = h;
            __syncwarp();
        }
    };
    for (int tr = 0; tr < n_ticks; tr++, t++) {
        if ((unsigned)(tr - fast_lo) < fast_len) tick(W2True{}, tr);
        else tick(W2False{}, tr);
    }
    if (DC == 2 && lane == 0) A.dc_stretch[gw].v_end = vloc;
}

// ------------------------------------------------------------------------------------------------
// Local DC state (DC == 2): what the warps could not know.
// Warp w ran its stretch (warm-up from frame s_w = B_w - warm, emit range [B_w, B_w + L_w)) with v = 0 in front of s_w,
// while the true state there is V0_w.  The blocker is linear, so every frame it produced lacks -a V0_w c^(n - s_w): a
// decaying exponential.  Each halfband decimator maps kappa mu^n to kappa A(mu) (mu^2)^q and the polyphase stage maps
// kappa mu^k to kappa mu^k_o G[row_o], so the cascade output lacks  -a V0_w Atot c^(2^S k_o - s_w) G[row_o]  (Atot and the
// 256 row gains G are computed once on the host in double from the actual taps).  V0_w follows from the records the
// warps left: v(B_w+1) = a_w v(B_w) + (v_end_w - a_w v_emit_w), a_w = c^L_w — an affine scan over a few thousand stretches.
// ------------------------------------------------------------------------------------------------
// (W2DcCorr, W2DcGeom: kernels.hpp)

__global__ void __launch_bounds__(1024) w2_dc_scan_kernel(const W2DcStretch* __restrict__ rec, W2DcGeom g,
                                                          W2DcCorr* __restrict__ corr, double2* __restrict__ carry)
{
    __shared__ double sA[1024], sBx[1024], sBy[1024];
    const int t = threadIdx.x, n = g.n_stretch;
    const int G = (n - 1 + 1023) / 1024;                         // stretches 1 .. n-1 in groups of G per thread
    const int w0 = 1 + t * G, w1 = min(n, w0 + G);
    const double a_full = exp((double)g.L_full * g.lnc), a_last = exp((double)g.L_last * g.lnc);
    double A = 1.0, Bx = 0.0, By = 0.0;                          // composite map of this thread's stretches
    for (int w = w0; w < w1; w++) {
        const double a = (w == n - 1) ? a_last : a_full;
        const W2DcStretch r = rec[w];
        const double bx = r.v_end.x - a * r.v_emit.x, by = r.v_end.y - a * r.v_emit.y;
        A = a * A; Bx = a * Bx + bx; By = a * By + by;
    }
    sA[t] = A; sBx[t] = Bx; sBy[t] = By;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {                         // inclusive scan of the maps (earlier map applied first)
        double pa = 1.0, pbx = 0.0, pby = 0.0;
        if (t >= d) { pa = sA[t - d]; pbx = sBx[t - d]; pby = sBy[t - d]; }
        __syncthreads();
        if (t >= d) { sBx[t] = sA[t] * pbx + sBx[t]; sBy[t] = sA[t] * pby + sBy[t]; sA[t] = sA[t] * pa; }
        __syncthreads();
    }
    const double2 v1 = rec[0].v_end;                             // stretch 0 ran from the carried state: exact
    double vx = v1.x, vy = v1.y;
    if (t > 0) { vx = sA[t - 1] * v1.x + sBx[t - 1]; vy = sA[t - 1] * v1.y + sBy[t - 1]; }
    const double unwarm = exp(-(double)g.warm_frames * g.lnc);
    if (t == 0) corr[0] = W2DcCorr{make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
    for (int w = w0; w < w1; w++) {
        const double a = (w == n - 1) ? a_last : a_full;
        const W2DcStretch r = rec[w];
        const double v0x = (vx - r.v_emit.x) * unwarm, v0y = (vy - r.v_emit.y) * unwarm;
        W2DcCorr c;
        c.c_pre = make_float2((float)(-g.alpha * v0x), (float)(-g.alpha * v0y));
        c.c_out = make_float2((float)(-g.alpha * v0x * g.atot), (float)(-g.alpha * v0y * g.atot));
        corr[w] = c;
        vx = a * vx + (r.v_end.x - a * r.v_emit.x);
        vy = a * vy + (r.v_end.y - a * r.v_emit.y);
    }
    // the state just before N1: the last tick ran pad_frames of zeros beyond it
    const bool owns_last = (n == 1) ? (t == 0) : (w0 < w1 && w1 == n);
    if (owns_last) {
        const double un = exp(-(double)g.pad_frames * g.lnc);
        *carry = make_double2(vx * un, vy * un);
    }
}

// adds the missing term to the outputs [O0, O1) of the launch and to the frames of the cf32 tail it wrote
__global__ void __launch_bounds__(256) w2_dc_correct_kernel(float2* __restrict__ y, long long O0, long long O1, uint32_t step, int S,
                                                            W2DcGeom g, const W2DcCorr* __restrict__ corr, const float* __restrict__ G,
                                                            float2* __restrict__ tail, long long tail_first, long long n0, long long N1)
{
    __shared__ float sG[256];
    sG[threadIdx.x] = G[threadIdx.x];
    __syncthreads();
    const float lnc = (float)g.lnc;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long n_out = O1 - O0;
    const long long t_lo = (tail_first > n0) ? tail_first : n0;
    const long long n_tail = (N1 > t_lo) ? (N1 - t_lo) : 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_out + n_tail; i += stride) {
        if (i < n_out) {
            const unsigned long long Dp = (unsigned long long)(O0 + i) * step - g.pos.p_base;
            const long long nk = dc_fold_frame(Dp, g, S);
            const long long w = (nk - g.B0) / g.L_full;
            if (w <= 0) continue;
            y[i] = dc_fold_add(y[i], Dp, nk, w, g, lnc, corr[w], sG);
        } else {
            const long long n = t_lo + (i - n_out);
            const long long w = (n - g.B0) / g.L_full;
            if (w <= 0) continue;
            const W2DcCorr c = corr[w];
            const float e = expf(lnc * (float)(n - (g.B0 + w * g.L_full - g.warm_frames)));
            float2 v = tail[n - tail_first];
            v.x = fmaf(c.c_pre.x, e, v.x); v.y = fmaf(c.c_pre.y, e, v.y);
            tail[n - tail_first] = v;
        }
    }
}

}  // namespace iqgpu
