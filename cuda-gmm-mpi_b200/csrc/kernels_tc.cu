// kernels_tc.cu — tcgen05 (UTCHMMA) kernels of the EM hot path for sm_100a.
//
// M-step (mstep_N + mstep_means + mstep_covariance1 of the reference,
// gaussian_kernel.cu:522-677) as ONE tensor-core contraction over the events:
//
//     S^T[f][k] = sum_n  phi_f(z_n) * g[k][n]        z = (x - shift) * inv_scale
//
// with the per-event feature vector phi = [1, z_d, z_i z_j (i>=j)] (F = 1+D+D(D+1)/2
// rows, shared by all clusters) as the A operand and the responsibilities as the
// B operand; FP32 accumulation in TMEM.
//
// Operand arithmetic (round 2).  The FP32 accumulation in TMEM truncates toward zero (tc_probe T2/T7) — but it
// is EXACT as long as every partial sum is a multiple of one quantum and fits 24 bits (tc_probe T8).  The
// operands are therefore split into a FIXED-POINT leading part and a small remainder:
//     phi_f = ph + pl,   ph = q_f * round(phi_f / q_f),   |ph| <= 2^11 q_f     (q_f: power of two per feature row,
//                                                                              from the data's largest |z_d|)
//     g     = gh + gl,   gh = 2^-6 * round(2^6 g)   (0 .. 64 quanta)
// (both by a magic-number add: no conversion round trip), and the products go to two accumulators per
// 128-row feature tile:
//     columns [0, 64):    sum ph * gh                 — every product a multiple of q_f 2^-6, at most 2^17 quanta;
//                                                       128 events per chain: <= 2^24 quanta: NO rounding at all
//     columns [64, 128):  sum ph * gl + pl * gs       — gs = g rounded once to FP16 (11 bits RELATIVE): with gh alone
//                                                       the dropped pl * gl would be O(pl / phi) of every event whose
//                                                       g is below the quantum (measured: 1.6e-4 on covariances);
//                                                       ~1 % of the magnitude, its truncation bias (~1e-6 relative to
//                                                       itself) is 1e-8 of the statistic
// The raw-moment cancellation |mu - shift|^2 / sigma^2 ~ 100 that amplified the old split's systematic error
// (1.5e-3 on responsibilities after 100 EM iterations) now multiplies unbiased rounding noise only.
// With B = [gh ; gl] stacked as ONE N = 128 operand, ph x [gh ; gl] is a single MMA at the tensor pipe's math
// rate (64 cycles; N = 64 runs at 49.8, operand-fetch bound) that fills both column groups; pl x gs (N = 64)
// adds into the second group: 114 instead of 149 cycles per (tile, k-step) and 14 instead of 18 KB of operand
// fetch.
//
// Dataflow per CTA (persistent over a contiguous range of events, 512 threads):
//   warp 0      TMA producer: tile [D][32 events] of the pre-standardised SoA copy z and raw
//               responsibility tile [64 clusters][32 events] (2-D tensor maps, SWIZZLE_128B for
//               the latter, zero fill out of bounds)
//   warps 4-11  operand builders (two warpgroups on alternate tiles): form the products, split
//               them, write the UMMA operand images (SWIZZLE_NONE core-matrix layout)
//   warp 1      MMA issuer: per 32 events and feature tile 2 x (M=128, N=128, K=16) + 2 x (M=128, N=64, K=16)
//   warps 12-15 flush: accumulators are SINGLE-buffered (3 tiles x 128 columns at D = 24); each feature tile
//               is drained every 128 events, the three tiles staggered by one sub-tile so that a drain
//               (TMEM -> registers, FP32 round-to-nearest adds into 192 register-resident partial sums per
//               thread) overlaps the MMAs of the other tiles.  The partial sums stay in registers for the whole
//               CTA range and are written ONCE (no scratch zeroing, no atomics: round 1 moved 1.7 GB of
//               RED.ADD.F64 traffic per launch).
// A second tiny kernel reduces the per-CTA partials in double and un-scales.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_fp16.h>
#if defined(__F16C__) && defined(__AVX__)
#include <immintrin.h>
#endif
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "host_math.h"
#include "kernels_tc.cuh"
#include "tc_ptx.cuh"

namespace gmm {

using namespace ptx;

#define TC_CUDA_TRY(expr)                                                                     \
    do {                                                                                      \
        cudaError_t e_ = (expr);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(GMM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));    \
    } while (0)

// ---------------------------------------------------------------------------
// M-step kernel configuration
// ---------------------------------------------------------------------------
constexpr int kTE = 32;          // events per sub-tile (MMA K extent per operand part)
constexpr int kNCL = 64;         // clusters per CTA pass
constexpr int kNST = 3;          // operand stages
constexpr int kNRAW = 4;         // raw (TMA) stages
constexpr int kChunkSub = 4;     // sub-tiles per chain of the exact column group: 128 events (the bit budget below)
constexpr int kChunkSub2 = 16;   // sub-tiles per chain of the remainder column group (no exactness to protect: drained 4x less often)
constexpr int kMThreads = 512;
// Bit budget of the exact accumulator: 11 (ph, every integer up to 2048 is an FP16 value) + 6 (gh) + 7 (128 events) = 24.
// The split favours phi: the remainder pl is rounded to FP16 RELATIVE to itself, so its (unbiased) rounding noise scales
// with the quantum of ph — on covariance entries 6e-6 per call with 9 + 8 bits, 1.2e-6 with 11 + 6 (scripts/emu_mstep.py).
constexpr int kPhiBits = 11;     // |ph| <= 2^11 quanta
constexpr float kGammaScale = 1024.0f;               // responsibilities are scaled by 2^10 in the operand
constexpr float kGammaMagic = 1.5f * 134217728.0f;   // 1.5 * 2^27: ulp = 16 = 2^-6 in the scaled units

// Row layout of the feature operand.  The four warps of a builder warpgroup run ONE instruction stream (round 1 / early
// round 2 unrolled a different quarter of the feature list per warp: 50 KB of SASS against a 32 KB L1.5 instruction cache,
// a third of the builders' stall samples were instruction fetch): warp p loads the event's coordinates ROTATED by p*D/4
// dimensions (a run-time shared-memory address) and evaluates the same canonical list of RPP rows on them —
//     r = 0                      1
//     r = 1 + a          (a < S) z'_a
//     r = 1 + S + a      (a < S) z'_a^2
//     r = 1 + 2S + a*D/2 + (d-1) (a < S, 1 <= d <= D/2)   z'_a * z'_{(a+d) mod D}
// with z'_t = z_{(t + pS) mod D}, S = D/4.  The rotations of the canonical pairs cover every unordered pair of
// dimensions once, except the D/2 antipodal pairs (d = D/2), which two warps produce (one copy is ignored), and the
// constant row (kept from warp 0).  Warp p writes operand rows [p*CPP*8, p*CPP*8 + RPP); tc_row_map() gives the packed
// statistic each row feeds.
template <int D> struct MCfg {
    static_assert(D % 4 == 0, "tensor M-step: D must be a multiple of 4");
    static constexpr int F = 1 + D + D * (D + 1) / 2;
    static constexpr int S = D / 4;                       // rotation step between the four builder warps
    static constexpr int RPP = 1 + 2 * S + S * (D / 2);   // canonical rows per warp
    static constexpr int CPP = (RPP + 7) / 8;             // 16-byte chunks per warp
    static constexpr int NCHUNK = 4 * CPP;                // chunks written per event
    static constexpr int MT = (NCHUNK * 8 + 127) / 128;   // M tiles of 128 feature rows
    static constexpr int PHI_PART = MT * 128 * kTE * 2;   // bytes of one part (leading or remainder)
    static constexpr int PHI_STAGE = 2 * PHI_PART;
    static constexpr int G_PART = kNCL * kTE * 2;
    static constexpr int G_STAGE = 3 * G_PART;            // [gh (64 rows) ; gl (64 rows)] = ONE K-major N = 128 image, then gs
    static constexpr int RAWX = D * kTE * 4;              // [D][32 events] from the SoA copy
    static constexpr int RAWG = kNCL * kTE * 4;
    static constexpr int OFF_PHI = 0;
    static constexpr int OFF_G = OFF_PHI + kNST * PHI_STAGE;
    static constexpr int OFF_RAWX = OFF_G + kNST * G_STAGE;
    static constexpr int OFF_RAWG = OFF_RAWX + kNRAW * RAWX;
    static constexpr int OFF_BAR = OFF_RAWG + kNRAW * RAWG;
    static constexpr int SMEM_BYTES = OFF_BAR + 512;
    static constexpr int TMEM_COLS = MT * 128;            // per feature tile: [ph gh | ph gl + pl gh]
    static_assert(OFF_RAWG % 1024 == 0 && RAWG % 1024 == 0, "SWIZZLE_128B TMA destinations need 1024-byte alignment");
    static_assert(MT <= 3, "accumulator tiles");
};

// Rounding constants: (v + magic) - magic = q * round(v / q) with magic = 1.5 * 2^23 * q.  One quantum for the
// coordinate rows and one for the product rows (bound = the largest |z_d| of the data over ALL dimensions, rounded up
// to a power of two: after the standardisation the dimensions have the same scale).
struct MMagic { float lin, prod; };

__host__ __device__ constexpr int tri_row(int t) {        // t = i(i+1)/2 + j, j <= i  ->  i
    int i = 0;
    while ((i + 1) * (i + 2) / 2 <= t) i++;
    return i;
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

// Leading part / remainder of canonical row r for the (rotated) event z (r is a compile-time constant after
// unrolling).  Products: both parts come from the EXACT product (fused multiply-adds), rounded once each.
template <int D>
__device__ __forceinline__ void feature_split(const float (&z)[D], int r, const MMagic& mg, float& h, float& l) {
    using C = MCfg<D>;
    if (r == 0) { h = 1.0f; l = 0.0f; }
    else if (r <= C::S) {
        const float v = z[r - 1];
        h = __fsub_rn(__fadd_rn(v, mg.lin), mg.lin);
        l = __fsub_rn(v, h);
    } else if (r < C::RPP) {
        int a, b;
        if (r <= 2 * C::S) { a = r - 1 - C::S; b = a; }
        else { const int t = r - 1 - 2 * C::S; a = t / (D / 2); b = (a + 1 + t % (D / 2)) % D; }
        h = __fsub_rn(__fmaf_rn(z[a], z[b], mg.prod), mg.prod);
        l = __fmaf_rn(z[a], z[b], -h);
    } else { h = 0.0f; l = 0.0f; }
}

// Builds the CPP 16-byte chunks of one event for builder warp `part` and stores both parts into the MN-major operand image:
//   byte(row, e) = (row/8)*512 + (e/8)*128 + (e%8)*16 + (row%8)*2        (LBO = 128, SBO = 512)
template <int D>
__device__ __forceinline__ void build_phi_chunks(const float (&z)[D], const MMagic& mg, uint8_t* hi_base, uint8_t* lo_base, int e, int part) {
    using C = MCfg<D>;
    const int eoff = part * (C::CPP * 512) + (e >> 3) * 128 + (e & 7) * 16;
#pragma unroll
    for (int c = 0; c < C::CPP; c++) {
        float hi[8], lo[8];
#pragma unroll
        for (int u = 0; u < 8; u++) feature_split<D>(z, c * 8 + u, mg, hi[u], lo[u]);
        uint4 h, l;
        h.x = pack_half2(hi[0], hi[1]); h.y = pack_half2(hi[2], hi[3]); h.z = pack_half2(hi[4], hi[5]); h.w = pack_half2(hi[6], hi[7]);   // exact: <= 2048 quanta
        l.x = pack_half2(lo[0], lo[1]); l.y = pack_half2(lo[2], lo[3]); l.z = pack_half2(lo[4], lo[5]); l.w = pack_half2(lo[6], lo[7]);
        *reinterpret_cast<uint4*>(hi_base + c * 512 + eoff) = h;
        *reinterpret_cast<uint4*>(lo_base + c * 512 + eoff) = l;
    }
}

// Packed statistic (index into a cluster's F values, -1 = ignored copy) and the two dimensions (-1 = none) behind
// operand row `row`; host side of the layout above.
struct RowInfo { int f, i, j; };
static RowInfo tc_row_info(int D, int row) {
    const int S = D / 4, RPP = 1 + 2 * S + S * (D / 2), CPP = (RPP + 7) / 8;
    const int p = row / (CPP * 8), r = row % (CPP * 8);
    RowInfo o{-1, -1, -1};
    if (p >= 4 || r >= RPP) return o;
    if (r == 0) { if (p == 0) o.f = 0; return o; }
    if (r <= S) { o.i = (r - 1 + p * S) % D; o.f = 1 + o.i; return o; }
    int a, b;
    if (r <= 2 * S) { a = r - 1 - S; b = a; }
    else { const int t = r - 1 - 2 * S; a = t / (D / 2); b = (a + 1 + t % (D / 2)) % D; }
    const int ta = (a + p * S) % D, tb = (b + p * S) % D;
    if (a != b && (b - a + D) % D == D / 2 && ta >= D / 2) return o;       // antipodal pair: the copy with the smaller first index counts
    o.i = ta > tb ? ta : tb;
    o.j = ta > tb ? tb : ta;
    o.f = feat2(D, o.i, o.j);
    return o;
}

// Feature tile `mt` is drained after sub-tile i when its 128-event chain ends there: the chains of the tiles are
// staggered by one sub-tile each, so that only one tile is being drained at a time (single-buffered accumulators).
// The remainder column group rides along and is drained (and restarted) only at every fourth of those points.
__device__ __forceinline__ bool chain_ends(int i, int mt, int nsub) { return ((i + mt) % kChunkSub) == kChunkSub - 1 || i == nsub - 1; }
__device__ __forceinline__ bool chain_starts(int i, int mt) { return i == 0 || ((i + mt) % kChunkSub) == 0; }
__device__ __forceinline__ bool chain2_ends(int i, int mt, int nsub) { return ((i + mt) % kChunkSub2) == kChunkSub2 - 1 || i == nsub - 1; }
__device__ __forceinline__ bool chain2_starts(int i, int mt) { return i == 0 || ((i + mt) % kChunkSub2) == 0; }

template <int D>
__global__ void __launch_bounds__(kMThreads, 1)
mstep_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_g, int n,
                float* __restrict__ scratch, int events_per_cta, const __grid_constant__ MMagic magic) {
    using C = MCfg<D>;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);
    uint64_t* raw_full = bars;                 // [kNRAW]
    uint64_t* raw_empty = bars + kNRAW;        // [kNRAW]
    uint64_t* op_full = bars + 2 * kNRAW;      // [kNST]
    uint64_t* op_empty = op_full + kNST;       // [kNST]
    uint64_t* acc_full = op_empty + kNST;      // [MT]  chain of feature tile mt complete (tcgen05.commit)
    uint64_t* acc_empty = acc_full + 3;        // [MT]  tile mt drained (4 flush warps)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 3);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e_begin = blockIdx.x * events_per_cta;
    const int e_end = min(n, e_begin + events_per_cta);
    const int nsub = (e_end - e_begin + kTE - 1) / kTE;
    const int k0 = blockIdx.y * kNCL;

    // ---- one-time setup ----
    for (int i = threadIdx.x * 16; i < C::OFF_RAWX; i += kMThreads * 16) *reinterpret_cast<uint4*>(smem + i) = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < kNRAW; s++) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 4); }
        for (int s = 0; s < kNST; s++) { mbar_init(&op_full[s], 4); mbar_init(&op_empty[s], 1); }
        for (int s = 0; s < 3; s++) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], 4); }
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc<512>(tmem_slot);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    // register re-partition between the warpgroups (64K registers per SM):
    //   WG0 (TMA / MMA / alloc) 40, WG1-2 (builders) 112, WG3 (flush accumulators) 240
    if (warp < 4) {
      asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
      if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            for (int i = 0; i < nsub; i++) {
                const int st = i % kNRAW, ph = (i / kNRAW) & 1;
                mbar_wait_parked(&raw_empty[st], ph ^ 1, 500);
                mbar_arrive_expect_tx(&raw_full[st], kTE * D * 4 + C::RAWG);
                const int e0 = e_begin + i * kTE;
                tma_load_2d(smem + C::OFF_RAWX + st * C::RAWX, &tm_x, e0, 0, &raw_full[st]);
                tma_load_2d(smem + C::OFF_RAWG + st * C::RAWG, &tm_g, e0, k0, &raw_full[st]);
            }
        }
      } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (elect_one()) {
            constexpr uint32_t idesc128 = make_idesc_f16(128, 2 * kNCL, /*A MN-major*/ true, /*B MN-major*/ false);
            constexpr uint32_t idesc64 = make_idesc_f16(128, kNCL, true, false);
            uint32_t drained = 0;                              // bit mt: wait parity of acc_empty[mt]
            uint32_t used = 0;                                 // bit mt: tile mt has completed at least one chain
            for (int i = 0; i < nsub; i++) {
                const int os = i % kNST, oph = (i / kNST) & 1;
                mbar_wait_parked(&op_full[os], oph, 100);
                tc_fence_after();
                const uint32_t phi = smem_u32(smem + C::OFF_PHI + os * C::PHI_STAGE);
                const uint32_t gam = smem_u32(smem + C::OFF_G + os * C::G_STAGE);
#pragma unroll
                for (int mt = 0; mt < C::MT; mt++) {
                    const bool first = chain_starts(i, mt), first2 = chain2_starts(i, mt);
                    if (first && ((used >> mt) & 1u)) {        // the previous chain of this tile must have been drained
                        mbar_wait_parked(&acc_empty[mt], (drained >> mt) & 1u, 100);
                        drained ^= 1u << mt;
                        tc_fence_after();
                    }
                    const uint32_t dcol = tmem + mt * 128;
#pragma unroll
                    for (int ks = 0; ks < kTE / 16; ks++) {
                        const uint64_t bdesc = make_smem_desc(gam + ks * 256, /*LBO*/ 128, /*SBO*/ 512);     // rows 0-63 gh, 64-127 gl
                        const uint64_t sdesc = make_smem_desc(gam + 2 * C::G_PART + ks * 256, 128, 512);     // gs
                        const uint64_t ah = make_smem_desc(phi + mt * 8192 + ks * 256, /*LBO*/ 128, /*SBO*/ 512);
                        const uint64_t al = make_smem_desc(phi + C::PHI_PART + mt * 8192 + ks * 256, 128, 512);
                        if (first && !first2 && ks == 0) {     // restart the exact group only: the two halves as separate N = 64 steps
                            const uint64_t ldesc = make_smem_desc(gam + C::G_PART + ks * 256, 128, 512);
                            mma_f16_ss(dcol, ah, bdesc, idesc64, false);                //  ph gh
                            mma_f16_ss(dcol + kNCL, ah, ldesc, idesc64, true);          //          += ph gl
                        } else {
                            mma_f16_ss(dcol, ah, bdesc, idesc128, !(first && ks == 0)); // [ph gh | ph gl]
                        }
                        mma_f16_ss(dcol + kNCL, al, sdesc, idesc64, true);             //          += pl gs
                    }
                    if (chain_ends(i, mt, nsub)) { mma_commit(&acc_full[mt]); used |= 1u << mt; }
                }
                mma_commit(&op_empty[os]);                    // operand stage reusable once these MMAs retire
            }
        }
      }
    } else if (warp < 12) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
        // ===================== operand builders =====================
        // two builder warpgroups work on alternate sub-tiles (two sub-tiles in flight), the four warps
        // of a group split the 16-byte feature chunks (c = part mod 4)
        const int bwg = (warp - 4) >> 2;           // sub-tiles i = bwg (mod 2)
        const int part = (warp - 4) & 3;
        const int bt = threadIdx.x - 128 - bwg * 128;   // 0..127 inside the group
        for (int i = bwg; i < nsub; i += 2) {
            const int rs = i % kNRAW, rph = (i / kNRAW) & 1;
            const int os = i % kNST, oph = (i / kNST) & 1;
            mbar_wait_parked(&raw_full[rs], rph, 200);
            // --- features of event `lane` ---
            float z[D];                                // already centred and scaled (tc_set_shift_scale writes the z copy), rotated by part * S
            {
                const float* xr = reinterpret_cast<const float*>(smem + C::OFF_RAWX + rs * C::RAWX) + lane;   // [d][32]: conflict-free
                int dd = part * C::S;
#pragma unroll
                for (int d = 0; d < D; d++) { z[d] = xr[dd * kTE]; dd = dd + 1 == D ? 0 : dd + 1; }
            }
            // --- responsibilities: thread -> (cluster row k, 8-event chunk ce), two items per thread.
            // The raw tile is written by TMA with SWIZZLE_128B (16-byte chunk c of row r sits at chunk
            // c ^ (r & 7)), so 8 lanes reading the same chunk of 8 consecutive rows hit 8 different
            // bank groups; the operand image puts the 4 K-chunks of an 8-row group next to each other
            // (LBO = 128, SBO = 512), so a warp stores 512 contiguous bytes: no bank conflicts either way.
            uint4 gh[2], gl[2], gs[2];
            float gdep = 0.0f;
#pragma unroll
            for (int it2 = 0; it2 < 2; it2++) {
                const int item = bt + it2 * 128;
                const int kg = item >> 5, l = item & 31;
                const int k = kg * 8 + (l & 7), ce = l >> 3;
                const uint8_t* grow = smem + C::OFF_RAWG + rs * C::RAWG + k * (kTE * 4);
                const float4 a = *reinterpret_cast<const float4*>(grow + (((2 * ce) ^ (k & 7)) << 4));
                const float4 b = *reinterpret_cast<const float4*>(grow + (((2 * ce + 1) ^ (k & 7)) << 4));
                const float g[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                gdep += a.x + b.x;
                float hi[8], lo[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {                  // gh = 16 * round(64 g) (0 .. 1024), gl = 1024 g - gh, both from the exact product
                    hi[u] = __fsub_rn(__fmaf_rn(g[u], kGammaScale, kGammaMagic), kGammaMagic);
                    lo[u] = __fmaf_rn(g[u], kGammaScale, -hi[u]);
                }
                gh[it2] = make_uint4(pack_half2(hi[0], hi[1]), pack_half2(hi[2], hi[3]), pack_half2(hi[4], hi[5]), pack_half2(hi[6], hi[7]));
                gl[it2] = make_uint4(pack_half2(lo[0], lo[1]), pack_half2(lo[2], lo[3]), pack_half2(lo[4], lo[5]), pack_half2(lo[6], lo[7]));
                gs[it2] = make_uint4(pack_half2(g[0] * kGammaScale, g[1] * kGammaScale), pack_half2(g[2] * kGammaScale, g[3] * kGammaScale),
                                     pack_half2(g[4] * kGammaScale, g[5] * kGammaScale), pack_half2(g[6] * kGammaScale, g[7] * kGammaScale));
            }
            // The raw tiles must BE in registers before the stage goes back to the TMA producer: an mbarrier arrive does
            // not wait for the warp's outstanding LDS (measured in round 1: with nothing consuming the z loads before the
            // arrive, the refill of the stage overtook the loads of the last dimensions).  The arrive is therefore made
            // data-dependent on every load of this thread: a sum over z and one component of each responsibility vector,
            // folded into the arrive's own operand list below (the asm statement consumes the value, so neither the
            // compiler nor the hardware can retire it before the loads have landed).
            float dep = gdep;
#pragma unroll
            for (int d = 0; d < D; d++) dep += z[d];
            __syncwarp();
            if (lane == 0) mbar_arrive_after(&raw_empty[rs], dep);
            else asm volatile("" ::"f"(dep));
            mbar_wait_parked(&op_empty[os], oph ^ 1, 200);
            uint8_t* phi_hi = smem + C::OFF_PHI + os * C::PHI_STAGE;
            uint8_t* phi_lo = phi_hi + C::PHI_PART;
            build_phi_chunks<D>(z, magic, phi_hi, phi_lo, lane, part);
            {
                // K-major B image: byte(k, e) = (k/8)*512 + (e/8)*128 + (k%8)*16 + (e%8)*2      (LBO = 128, SBO = 512); gl = rows 64..127
                uint8_t* g_hi = smem + C::OFF_G + os * C::G_STAGE;
#pragma unroll
                for (int it2 = 0; it2 < 2; it2++) {
                    const int item = bt + it2 * 128;
                    const int kg = item >> 5, l = item & 31;
                    *reinterpret_cast<uint4*>(g_hi + kg * 512 + l * 16) = gh[it2];
                    *reinterpret_cast<uint4*>(g_hi + C::G_PART + kg * 512 + l * 16) = gl[it2];
                    *reinterpret_cast<uint4*>(g_hi + 2 * C::G_PART + kg * 512 + l * 16) = gs[it2];
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&op_full[os]);
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 240;");
        // ===================== flush: TMEM -> register-resident FP32 partial sums =====================
        const int q = warp - 12;                                   // TMEM lane quadrant (= warp % 4)
        float racc[C::MT * kNCL];
#pragma unroll
        for (int j = 0; j < C::MT * kNCL; j++) racc[j] = 0.0f;
        uint32_t full = 0;                                         // bit mt: wait parity of acc_full[mt]
        for (int i = 0; i < nsub; i++) {
#pragma unroll
            for (int mt = 0; mt < C::MT; mt++) {
                if (!chain_ends(i, mt, nsub)) continue;
                mbar_wait_parked(&acc_full[mt], (full >> mt) & 1u, 300);
                full ^= 1u << mt;
                tc_fence_after();
                const uint32_t tbase = tmem + ((uint32_t)(q * 32) << 16) + mt * 128;
                // group 0: exact leading products; group 1 (only when its longer chain ends here): remainder products.
                // One copy of the code for both (not unrolled: the kernel's SASS has to stay inside the 32 KB L1.5 I-cache).
                const int ngroups = chain2_ends(i, mt, nsub) ? 2 : 1;
#pragma unroll 1
                for (int grp = 0; grp < ngroups; grp++) {
#pragma unroll
                    for (int b = 0; b < kNCL / 32; b++) {
                        uint32_t a[32];
                        tmem_ld_32x32(tbase + grp * kNCL + b * 32, a);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; j++) racc[mt * kNCL + b * 32 + j] += __uint_as_float(a[j]);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[mt]);
            }
        }
        // one plain store of this thread's partial sums: [cta][tile][row][64 clusters]
        float* my = scratch + ((size_t)(blockIdx.y * gridDim.x + blockIdx.x) * C::MT * 128 + q * 32 + lane) * kNCL;
#pragma unroll
        for (int mt = 0; mt < C::MT; mt++)
#pragma unroll
            for (int j = 0; j < kNCL; j += 4)
                *reinterpret_cast<float4*>(my + (size_t)mt * 128 * kNCL + j) =
                    make_float4(racc[mt * kNCL + j], racc[mt * kNCL + j + 1], racc[mt * kNCL + j + 2], racc[mt * kNCL + j + 3]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc<512>(tmem);
}

// z = (x - shift) * inv_scale over the SoA event copy, once per data set: the centred/scaled copy the M-step
// tiles are cut from (the E-step converters apply the same two operations to the AoS rows, so both kernels
// see bit-identical z).
__global__ void standardise_soa_kernel(const float* __restrict__ xs, float* __restrict__ zs, size_t pitch, int n, int D,
                                       const float* __restrict__ shift_f, const float* __restrict__ inv_scale_f) {
    const int d = blockIdx.y;
    const float s = shift_f[d], isc = inv_scale_f[d];
    const float* x = xs + (size_t)d * pitch;
    float* z = zs + (size_t)d * pitch;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        z[e] = __fmul_rn(__fsub_rn(x[e], s), isc);
}

// Reduce the per-CTA FP32 partials in double, undo the operand scaling and write the packed statistics.
// rowmap[row] = (packed statistic index or -1, dimension i, dimension j) of operand row `row` (tc_row_info).
__global__ void __launch_bounds__(256)
mstep_tc_finalize_kernel(const float* __restrict__ scratch, int ncta_x, int MT, int K, int F, const int3* __restrict__ rowmap,
                         const double* __restrict__ scale, double* __restrict__ stats) {
    // one block per operand row; thread -> (cluster column, quarter of the CTAs): 256-byte coalesced reads
    __shared__ double part[4][kNCL];
    const int3 rm = rowmap[blockIdx.x];
    if (rm.x < 0) return;
    const int mt = blockIdx.x / 128, row = blockIdx.x % 128;
    const int col = threadIdx.x & (kNCL - 1), q = threadIdx.x / kNCL;
    double fac = 1.0 / (double)kGammaScale;
    if (rm.y >= 0) fac *= scale[rm.y];
    if (rm.z >= 0) fac *= scale[rm.z];
    for (int ty = 0; ty * kNCL < K; ty++) {
        double s = 0;
        for (int cx = q; cx < ncta_x; cx += 4)
            s += (double)scratch[(((size_t)(ty * ncta_x + cx) * MT + mt) * 128 + row) * kNCL + col];
        part[q][col] = s;
        __syncthreads();
        const int k = ty * kNCL + col;
        if (q == 0 && k < K) stats[(size_t)k * F + rm.x] += (part[0][col] + part[1][col] + part[2][col] + part[3][col]) * fac;
        __syncthreads();
    }
}

// ===========================================================================
// E-step (estep1 + estep2 of the reference, gaussian_kernel.cu:383-512) on
// tensor cores.  With Rinv = W^T W (W upper triangular, from the Cholesky
// factor of Rinv computed on the host) the quadratic form is
//     q_k(x) = || W_k (x - mu_k) ||^2 = || W'_k z + v_k ||^2 ,   z = (x - shift) * inv_scale,
// i.e. ONE GEMM  Y[n][(k,d)] = Z~[n][:] . B[(k,d)][:]  with the constant folded in
// through a ones column, followed by a square-and-sum epilogue, the log-sum-exp
// over the clusters and the log-likelihood reduction.  Operands are FP16 hi/lo
// split (z = zh + zl, W' = Wh + Wl); the K dimension concatenates
//     [ zh_c zl_c ]_c | [ zh | 1 1 0.. ]     x     [ Wh_c Wh_c ]_c | [ Wl | vh vl 0.. ]
// (the lo*lo product is dropped), FP32 accumulation in TMEM.  The duplicated Wh
// chunk is not stored twice: the B descriptor of those MMA steps uses a leading
// byte offset of 0, so both 8-element K chunks alias the same shared-memory chunk
// (verified by csrc/probe/tc_probe.cu, test T5).  That makes the whole B operand
// (all clusters: 172 KB at K=64, D=24) RESIDENT in the shared memory of one CTA;
// only the event tiles stream.
//
// One persistent CTA per SM, 768 threads in six warpgroups (round 2: the epilogue is split in two stages — round 1's
// eight epilogue warps did squares, log-sum-exp and stores back to back, 6370 cycles per 128-event tile of which the MMA
// issuer was stalled 3500 behind full accumulators while they were busy with log-sum-exp and stores; the per-phase
// counters of that kernel are in profiles/):
//   warp 1       MMA issuer: per 128-event tile, per supergroup of 16 clusters and per block c of 8
//                output dimensions, the k-steps that block needs (tcgen05.mma M=128, N=128, K=16)
//   warp 2       TMEM allocation: 3 accumulator buffers x 128 columns + 2 x 64 columns for the hand-over of q
//   warps 4-7    converters: coalesced loads of the event rows, centre/scale, FP16 hi/lo
//                split, K-major SWIZZLE_NONE operand image (2 stages)
//   warps 8-15   squares (two warpgroups, each takes 8 of the 16 clusters of every supergroup): tcgen05.ld of the
//                accumulators (buffer released as soon as the values are in registers) -> packed fma.f32x2 sums of
//                squares carried over the blocks -> q[event][cluster] written back to TMEM (tcgen05.st)
//   warps 16-23  log-sum-exp + stores (two warpgroups, 32 clusters each): tcgen05.ld of q -> base-2 logits ->
//                max / sum-exp2 (+ exchange between the warpgroups) -> responsibilities (coalesced 128-byte row
//                segments) + log-likelihood (double) — for tile t while the MMAs and the squares of tile t+1 run
// ===========================================================================

// Block structure.  W is upper triangular, so the 8 output columns d in [8c, 8c+8) of a cluster
// ("block" c) only need the K chunks z_j with j >= c.  Columns are therefore grouped by block:
// one MMA N tile = block c of 16 clusters (N = 128), and block c issues only the k-steps it needs —
// 5 + 4 + 2 = 11 instead of 15 at D = 24 (-27 % tensor work and TMEM accumulator traffic).
template <int D> struct ECfg {
    static_assert(D % 8 == 0, "tensor E-step: D must be a multiple of 8");
    static constexpr int CP = D / 8;                          // 8-wide chunks of z / blocks of output columns
    static constexpr int NLO = (CP + 1 + 1) / 2 * 2;          // chunks of the [zh | ones (| pad)] x [Wl | v] part
    static constexpr int NCHKA = 2 * CP + 2;                  // A image chunks: (zh_c, zl_c) pairs, then the constant chunks ones, zero
    static constexpr int NCHKB = CP + NLO;                    // B image chunks: Wh_c, then Wl.., v, pad
    static constexpr int GB = 16;                             // clusters per supergroup
    static constexpr int N = GB * 8;                          // MMA N = one block of a supergroup (128 columns)
    static constexpr int MAXSG = 64 / GB;                     // up to 64 clusters resident
    static constexpr int NBUF = 3;                            // TMEM accumulator buffers (3 x 128 columns)
    static constexpr int QCOL = NBUF * N;                     // first column of the q hand-over: 2 tiles x 64 clusters
    static constexpr int NWG = 2;                             // warpgroups per epilogue stage
    static constexpr int CW = GB / NWG;                       // clusters per warpgroup per supergroup
    static constexpr int LPT = MAXSG * CW;                    // logits held per log-sum-exp thread (32)
    static constexpr int A_STAGE = NCHKA * 128 * 16;
    static constexpr int B_BLOCK = NCHKB * N * 16;            // one block of one supergroup
    static constexpr int B_SG = CP * B_BLOCK;
    static constexpr int OFF_B = 0;
    static constexpr int OFF_A = OFF_B + MAXSG * B_SG;
    static constexpr int OFF_CK = OFF_A + 2 * A_STAGE;        // float[64] (constant + ln(pi)) * log2(e), then float[64] -0.5 * log2(e) / scale_k^2
    static constexpr int OFF_EX = OFF_CK + 512;               // exchange: [2 parity][NWG][128] x (max, sum)
    static constexpr int OFF_BAR = OFF_EX + 2 * NWG * 128 * 8;
    static constexpr int SMEM_BYTES = OFF_BAR + 512;
    static constexpr int THREADS = 256 + 2 * 128 * NWG;       // warpgroup 0, converters, 2 square + 2 log-sum-exp warpgroups
    static_assert(QCOL + 2 * 64 <= 512, "TMEM columns");
};

template <int D>
__global__ void __launch_bounds__(768, 1)
estep_tc_kernel(const float* __restrict__ x_aos, const uint8_t* __restrict__ b_img, const float* __restrict__ ck,
                const float* __restrict__ shift_f, const float* __restrict__ inv_scale_f, float* __restrict__ memb,
                size_t pitch, int n, int K, int NSG, double* __restrict__ ll_out, int mode, const float* den_in,
                float* den_out) {
    // K / NSG / b_img / ck / memb describe ONE pass of at most 64 clusters.  More than 64 clusters take 2P - 1 launches
    // for P passes, and every responsibility is written exactly once (round 1 normalised each pass within itself and
    // rescaled all of them in a read-modify-write pass over the memberships):
    //   mode 1 (passes 0 .. P-2)  log-denominator only: den_out[e] = ln(sum_k exp(logit)) (+ den_in[e] in log space), no stores
    //   mode 2 (pass P-1)         its own log-sum-exp joined with den_in[e] (all other passes): final responsibilities of this
    //                             pass, den_out[e] = the event's total log-denominator, log-likelihood
    //   mode 3 (passes 0 .. P-2)  responsibilities against the known total den_in[e]: no log-sum-exp, no exchange
    //   mode 0                    single pass (K <= 64)
    using C = ECfg<D>;
    constexpr int NWG = C::NWG;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);
    uint64_t* a_full = bars;            // [2]  4 converter warps
    uint64_t* a_empty = bars + 2;       // [2]  tcgen05.commit
    uint64_t* b_full = bars + 4;        // [1]
    uint64_t* acc_full = bars + 5;      // [NBUF]  tcgen05.commit
    uint64_t* acc_empty = bars + 8;     // [NBUF]  8 square warps
    uint64_t* q_full = bars + 11;       // [2]  8 square warps: q of a tile is in TMEM
    uint64_t* q_empty = bars + 13;      // [2]  8 log-sum-exp warps: q of a tile is in their registers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 15);
    float* ck_s = reinterpret_cast<float*>(smem + C::OFF_CK);          // [64] additive logit constants, [64] multipliers
    float2* ex = reinterpret_cast<float2*>(smem + C::OFF_EX);
    float* sh_s = reinterpret_cast<float*>(smem + C::OFF_BAR + 128);   // [32] shift, [32] inverse scale
    float* isc_s = sh_s + 32;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntiles = (n + 127) / 128;
    const int my_tiles = (int)blockIdx.x < ntiles ? (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; s++) { mbar_init(&a_full[s], 4); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < C::NBUF; s++) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], 4 * NWG); }
        for (int s = 0; s < 2; s++) { mbar_init(&q_full[s], 4 * NWG); mbar_init(&q_empty[s], 4 * NWG); }
        mbar_init(b_full, 1);
        fence_mbar_init();
    }
    // base-2 logits in the epilogue: l2 = ck * log2(e) + (-0.5 * log2(e) / scale_k^2) * |scale_k * y|^2   (the per-cluster
    // power-of-two scale_k keeps the FP16 whitening factors in range whatever the cluster's width, see bimg_cluster)
    if (threadIdx.x < 64) { ck_s[threadIdx.x] = ck[threadIdx.x] * 1.4426950408889634f; ck_s[64 + threadIdx.x] = ck[64 + threadIdx.x]; }
    if (threadIdx.x < D) { sh_s[threadIdx.x] = shift_f[threadIdx.x]; isc_s[threadIdx.x] = inv_scale_f[threadIdx.x]; }
    if (threadIdx.x >= 128 && threadIdx.x < 256) {             // constant chunks of both A stages: {1, 1, 0 ...} and zeros
        const int row = threadIdx.x - 128;
#pragma unroll
        for (int st = 0; st < 2; st++) {
            uint8_t* a = smem + C::OFF_A + st * C::A_STAGE + row * 16;
            *reinterpret_cast<uint4*>(a + (2 * C::CP) * 2048) = make_uint4(0x3C003C00u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(a + (2 * C::CP + 1) * 2048) = make_uint4(0u, 0u, 0u, 0u);
        }
        fence_proxy_async_smem();
    }
    __syncthreads();
    if (threadIdx.x == 0) {                    // resident B operand: one TMA bulk copy per block
        mbar_arrive_expect_tx(b_full, (uint32_t)NSG * C::B_SG);
        for (int g = 0; g < NSG * C::CP; g++) tma_load_1d(smem + C::OFF_B + g * C::B_BLOCK, b_img + (size_t)g * C::B_BLOCK, C::B_BLOCK, b_full);
    }
    if (warp == 2) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    // register pools (launch: 768 x 80 = 61440): WG0 24, converters 72, squares 2 x 112, log-sum-exp 2 x 80
    if (warp < 4) {
      asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
      if (warp == 1) {
        // ===================== MMA issuer =====================
        if (elect_one()) {
            constexpr uint32_t idesc = make_idesc_f16(128, C::N, false, false);
            uint32_t pe = (1u << C::NBUF) - 1u;                // wait parity of acc_empty[b], one bit per buffer
            mbar_wait(b_full, 0);                              // the resident B image has landed (the converters did not wait for it)
            for (int it = 0; it < my_tiles; it++) {
                const int as = it & 1, aph = (it >> 1) & 1;
                mbar_wait_parked(&a_full[as], aph, 200);
                tc_fence_after();
                const uint32_t abase = smem_u32(smem + C::OFF_A + as * C::A_STAGE);
                uint32_t buf = 0;                              // the buffer sequence restarts with every tile (squares: same rule)
                for (int sg = 0; sg < NSG; sg++) {
#pragma unroll
                    for (int c = 0; c < C::CP; c++) {
                        mbar_wait_parked(&acc_empty[buf], (pe >> buf) & 1u, 100);
                        pe ^= 1u << buf;
                        tc_fence_after();
                        const uint32_t bbase = smem_u32(smem + C::OFF_B + (sg * C::CP + c) * C::B_BLOCK);
                        bool acc = false;
#pragma unroll
                        for (int j = c; j < C::CP; j++) {       // (zh_j, zl_j) x (Wh_j, Wh_j): B chunk aliased through LBO = 0
                            const uint64_t adesc = make_smem_desc(abase + (2 * j) * 2048, /*LBO*/ 2048, /*SBO*/ 128);
                            const uint64_t bdesc = make_smem_desc(bbase + j * (C::N * 16), /*LBO*/ 0, /*SBO*/ 128);
                            mma_f16_ss(tmem + buf * C::N, adesc, bdesc, idesc, acc);
                            acc = true;
                        }
#pragma unroll
                        for (int t = 0; t < C::NLO / 2; t++) {  // (zh.., ones) x (Wl.., v): needed iff it holds a chunk index >= c
                            if (2 * t + 1 >= c) {
                                // A side of this step: elements 2t and 2t+1 of [zh_0 .. zh_{CP-1}, ones, zero] — zh_m is the chunk the
                                // (zh_m, zl_m) steps already use (chunk 2m), so the step's two K chunks are simply further apart
                                constexpr int CP_ = C::CP;
                                const int m0 = 2 * t, m1 = 2 * t + 1;
                                const int ch0 = m0 < CP_ ? 2 * m0 : 2 * CP_ + (m0 - CP_), ch1 = m1 < CP_ ? 2 * m1 : 2 * CP_ + (m1 - CP_);
                                const uint64_t adesc = make_smem_desc(abase + ch0 * 2048, /*LBO*/ (uint32_t)(ch1 - ch0) * 2048, /*SBO*/ 128);
                                const uint64_t bdesc = make_smem_desc(bbase + (C::CP + 2 * t) * (C::N * 16), /*LBO*/ C::N * 16, /*SBO*/ 128);
                                mma_f16_ss(tmem + buf * C::N, adesc, bdesc, idesc, acc);
                                acc = true;
                            }
                        }
                        mma_commit(&acc_full[buf]);
                        buf = (buf + 1) % C::NBUF;
                    }
                }
                mma_commit(&a_empty[as]);
            }
        }
      }
    } else if (warp < 8) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
        // ===================== converters =====================
        const int row = threadIdx.x - 128;
        for (int it = 0; it < my_tiles; it++) {
            const int st = it & 1, ph = (it >> 1) & 1;
            const long long e = (long long)((int)blockIdx.x + it * (int)gridDim.x) * 128 + row;
            float4 xv[D / 4];
            if (e < n) {
                const float4* xr = reinterpret_cast<const float4*>(x_aos + (size_t)e * D);
#pragma unroll
                for (int v = 0; v < D / 4; v++) xv[v] = __ldg(xr + v);
            } else {
#pragma unroll
                for (int v = 0; v < D / 4; v++) xv[v] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            uint32_t hi[D / 2], lo[D / 2];
#pragma unroll
            for (int v = 0; v < D / 4; v++) {
                const float4 t = xv[v];
                const float4 s4 = reinterpret_cast<const float4*>(sh_s)[v], i4 = reinterpret_cast<const float4*>(isc_s)[v];
                const float z0 = (t.x - s4.x) * i4.x, z1 = (t.y - s4.y) * i4.y;
                const float z2 = (t.z - s4.z) * i4.z, z3 = (t.w - s4.w) * i4.w;
                const __half2 h01 = __floats2half2_rn(z0, z1), h23 = __floats2half2_rn(z2, z3);
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                hi[2 * v] = *reinterpret_cast<const uint32_t*>(&h01);
                hi[2 * v + 1] = *reinterpret_cast<const uint32_t*>(&h23);
                lo[2 * v] = pack_half2(z0 - f01.x, z1 - f01.y);
                lo[2 * v + 1] = pack_half2(z2 - f23.x, z3 - f23.y);
            }
            mbar_wait_parked(&a_empty[st], ph ^ 1, 1000);
            uint8_t* a = smem + C::OFF_A + st * C::A_STAGE + row * 16;     // K-major: [chunk][row][16 B]
#pragma unroll
            for (int c = 0; c < C::CP; c++) {                  // the constant chunks (ones, zero) were written once at kernel start
                const uint4 h = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
                const uint4 l = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
                *reinterpret_cast<uint4*>(a + (2 * c) * 2048) = h;
                *reinterpret_cast<uint4*>(a + (2 * c + 1) * 2048) = l;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&a_full[st]);
        }
    } else if (warp < 16) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        // ===================== squares: accumulators -> q[event][cluster] (TMEM) =====================
        const int sq = (warp - 8) >> 2, qd = warp & 3;
        const uint32_t lane_base = (uint32_t)(qd * 32) << 16;
        uint32_t pf = 0u;                                      // wait parity of acc_full[b], one bit per buffer
        for (int it = 0; it < my_tiles; it++) {
            const int tb = it & 1;
            mbar_wait_parked(&q_empty[tb], ((it >> 1) & 1) ^ 1, 200);      // the previous tile in this q buffer has been read
            tc_fence_after();
            uint32_t buf = 0;                                  // the buffer sequence restarts with every tile (MMA issuer: same rule)
#pragma unroll 1
            for (int sg = 0; sg < NSG; sg++) {                 // not unrolled: the kernel's SASS has to stay inside the 32 KB L1.5 I-cache
                {
                    uint64_t qa[C::CW], qb[C::CW];             // packed partial sums of squares of this warpgroup's 8 clusters
#pragma unroll
                    for (int i = 0; i < C::CW; i++) { qa[i] = 0ull; qb[i] = 0ull; }
#pragma unroll
                    for (int c = 0; c < C::CP; c++) {
                        mbar_wait_parked(&acc_full[buf], (pf >> buf) & 1u, 200);
                        pf ^= 1u << buf;
                        tc_fence_after();
                        const uint32_t tcol = tmem + lane_base + buf * C::N + sq * (C::CW * 8);
                        uint32_t v[C::CW * 8];                 // CW clusters x 8 columns
                        tmem_ld_32x32(tcol, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
                        tmem_ld_32x32(tcol + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&acc_empty[buf]);   // the block is in registers: hand the buffer back
                        buf = buf + 1 == C::NBUF ? 0 : buf + 1;
#pragma unroll
                        for (int i = 0; i < C::CW; i++) {
                            sq_acc2(qa[i], v[i * 8 + 0], v[i * 8 + 1]);
                            sq_acc2(qb[i], v[i * 8 + 2], v[i * 8 + 3]);
                            sq_acc2(qa[i], v[i * 8 + 4], v[i * 8 + 5]);
                            sq_acc2(qb[i], v[i * 8 + 6], v[i * 8 + 7]);
                        }
                    }
                    uint32_t qv[C::CW];
#pragma unroll
                    for (int i = 0; i < C::CW; i++) qv[i] = __float_as_uint(hsum2(qa[i], qb[i]));
                    // column of cluster (sg, sq, i) in the hand-over: tile buffer tb, warpgroup sq, then sg * 8 + i
                    tmem_st_32x8(tmem + lane_base + C::QCOL + tb * 64 + sq * (C::MAXSG * C::CW) + sg * C::CW, qv);
                }
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&q_full[tb]);
        }
    } else {
        // ===================== log-sum-exp + stores (80 registers: the launch allocation) =====================
        const int wg = (warp - 16) >> 2, qd = warp & 3;
        const int row = qd * 32 + lane;
        const uint32_t lane_base = (uint32_t)(qd * 32) << 16;
        double ll_acc = 0.0;
        constexpr float kLn2 = 0.6931471805599453f;
        for (int it = 0; it < my_tiles; it++) {
            const int tb = it & 1;
            const long long e = (long long)((int)blockIdx.x + it * (int)gridDim.x) * 128 + row;
            // q, then base-2 logits, then 2^(logit - max), as PACKED pairs of neighbouring clusters (fma / add / mul .f32x2:
            // half the instructions and FMA-pipe cycles of this stage; the pipe is shared with the squares)
            uint64_t lgp[C::LPT / 2];
            mbar_wait_parked(&q_full[tb], (it >> 1) & 1, 200);
            tc_fence_after();
            {
                uint32_t qraw[C::LPT];
                tmem_ld_32x32(tmem + lane_base + C::QCOL + tb * 64 + wg * C::LPT, qraw);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&q_empty[tb]);
#pragma unroll
                for (int sg = 0; sg < C::MAXSG; sg++) {
                    if (sg < NSG) {
                        const float4* cp = reinterpret_cast<const float4*>(ck_s + sg * C::GB + wg * C::CW);
                        const float4* mp = reinterpret_cast<const float4*>(ck_s + 64 + sg * C::GB + wg * C::CW);
                        const float4 c0 = cp[0], c1 = cp[1], m0 = mp[0], m1 = mp[1];
                        const int j = sg * C::CW;
                        lgp[j / 2 + 0] = ffma2(pack2f(m0.x, m0.y), pack2u(qraw[j + 0], qraw[j + 1]), pack2f(c0.x, c0.y));
                        lgp[j / 2 + 1] = ffma2(pack2f(m0.z, m0.w), pack2u(qraw[j + 2], qraw[j + 3]), pack2f(c0.z, c0.w));
                        lgp[j / 2 + 2] = ffma2(pack2f(m1.x, m1.y), pack2u(qraw[j + 4], qraw[j + 5]), pack2f(c1.x, c1.y));
                        lgp[j / 2 + 3] = ffma2(pack2f(m1.z, m1.w), pack2u(qraw[j + 6], qraw[j + 7]), pack2f(c1.z, c1.w));
                    } else {                                   // columns of unused supergroups are not written
#pragma unroll
                        for (int u = 0; u < C::CW / 2; u++) lgp[sg * C::CW / 2 + u] = pack2f(-INFINITY, -INFINITY);
                    }
                }
            }
            float mx = -INFINITY;
#pragma unroll
            for (int u = 0; u < C::LPT / 2; u++) { mx = fmaxf(mx, lo2f(lgp[u])); mx = fmaxf(mx, hi2f(lgp[u])); }
            float scale;
            if (mode == 3) {
                // the event's total log-denominator is known: gamma = 2^(l2 - denom * log2 e)
                const float d2 = e < n ? den_in[e] * 1.4426950408889634f : 0.f;
                const uint64_t nd = pack2f(-d2, -d2);
#pragma unroll
                for (int u = 0; u < C::LPT / 2; u++) {
                    const uint64_t t2 = fadd2(lgp[u], nd);
                    lgp[u] = pack2f(ex2_approx(lo2f(t2)), ex2_approx(hi2f(t2)));
                }
                scale = 1.0f;
            } else {
                // log-sum-exp over the clusters (estep2, gaussian_kernel.cu:481-503): local part, then the two warpgroups combine
                const uint64_t nm = pack2f(-mx, -mx);
                uint64_t s0 = 0ull, s1 = 0ull;                       // two packed running sums (four independent chains)
#pragma unroll
                for (int u = 0; u < C::LPT / 2; u++) {
                    const uint64_t t2 = fadd2(lgp[u], nm);
                    lgp[u] = pack2f(ex2_approx(lo2f(t2)), ex2_approx(hi2f(t2)));
                    if (u & 1) s1 = fadd2(s1, lgp[u]); else s0 = fadd2(s0, lgp[u]);
                }
                const uint64_t s2 = fadd2(s0, s1);
                const float sm = lo2f(s2) + hi2f(s2);
                float2* exb = ex + (it & 1) * (NWG * 128);
                exb[wg * 128 + row] = make_float2(mx, sm);
                // den_in may alias den_out (running log-denominator updated in place by warpgroup 0): both warpgroups read
                // it BEFORE the barrier, the write comes after
                const float dx = (mode != 0 && den_in != nullptr && e < n) ? den_in[e] : 0.f;
                named_bar_sync(1, NWG * 128);
                const float2 o = exb[(wg ^ 1) * 128 + row];
                const float M = fmaxf(mx, o.x);
                const float own = ex2_approx(mx - M);
                const float S = sm * own + o.y * ex2_approx(o.x - M);
                float denom = fmaf(M, kLn2, logf(S));                // :490-494, back in natural units
                scale = own / S;                                     // exp(l - denom) = 2^(l2 - mx) * 2^(mx - M) / S
                if (mode != 0 && e < n) {
                    if (den_in != nullptr) {                         // join with the other passes' log-denominator
                        const float g = fmaxf(denom, dx);
                        const float tot = g + logf(__expf(denom - g) + __expf(dx - g));
                        scale *= __expf(denom - tot);
                        denom = tot;
                    }
                    if (wg == 0) den_out[e] = denom;
                }
                if (wg == 0 && e < n && (mode == 0 || mode == 2)) ll_acc += (double)denom;
            }
            if (e < n && mode != 1) {
                // Rows [K, 8*ceil(K/8)) are written too (zeros of the padding clusters): the buffer is allocated in
                // multiples of 8 rows, which keeps the 8 stores of a group unpredicated.
                float* gp = memb + (size_t)(wg * C::CW) * pitch + e;      // row of this warpgroup's first cluster
                const uint64_t sc2 = pack2f(scale, scale);
#pragma unroll
                for (int sg = 0; sg < C::MAXSG; sg++) {
                    if (sg * C::GB + wg * C::CW < K) {
                        float* gq = gp + (size_t)(sg * C::GB) * pitch;
#pragma unroll
                        for (int u = 0; u < C::CW / 2; u++) {
                            const uint64_t g2 = fmul2(lgp[sg * C::CW / 2 + u], sc2);      // :498-501
                            gq[0] = lo2f(g2);
                            gq[pitch] = hi2f(g2);
                            gq += 2 * pitch;
                        }
                    }
                }
            }
        }
        if (wg == 0 && (mode == 0 || mode == 2)) {
            ll_acc = ll_acc + __shfl_down_sync(0xffffffffu, ll_acc, 16);
            ll_acc = ll_acc + __shfl_down_sync(0xffffffffu, ll_acc, 8);
            ll_acc = ll_acc + __shfl_down_sync(0xffffffffu, ll_acc, 4);
            ll_acc = ll_acc + __shfl_down_sync(0xffffffffu, ll_acc, 2);
            ll_acc = ll_acc + __shfl_down_sync(0xffffffffu, ll_acc, 1);
            if (lane == 0) atomicAdd(ll_out, ll_acc);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc<512>(tmem);
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct TcState {
    const float* d_x = nullptr;
    const float* d_x_soa = nullptr;
    float* d_z_soa = nullptr;        // [D][memb_pitch] centred/scaled SoA copy (M-step TMA source)
    float* d_memb = nullptr;
    size_t memb_pitch = 0;
    int n = 0, D = 0, Kmax = 0, num_sms = 148;
    CUtensorMap tm_x{}, tm_g{};
    bool maps_ok = false;
    float* d_shift_f = nullptr;      // [32]
    float* d_inv_scale_f = nullptr;  // [32]
    double* d_scale = nullptr;       // [32] = 1 / inv_scale_f (double)
    float* d_scratch = nullptr;      // [CTAs][MT][128][64] per-CTA partial sums, written once per launch
    size_t scratch_floats = 0;
    bool have_shift = false;
    bool mstep_ready = false;        // the fixed-point quanta of the feature rows are set and inside the supported range
    float zmax[GMM_MAX_DIMENSIONS] = {0};    // power-of-two bound of |z_d| over the whole data set
    MMagic magic{0.f, 0.f};          // rounding constants of the coordinate / product rows
    int3* d_rowmap = nullptr;        // [MT * 128] operand row -> (packed statistic, dimension i, dimension j)
    // E-step
    CUtensorMap tm_x128{};
    bool emap_ok = false;
    uint8_t* d_bimg = nullptr;       // [MAXNG * B_GROUP] resident B operand image
    uint8_t* h_bimg = nullptr;       // pinned
    size_t bimg_bytes = 0;
    uint8_t* d_opnd = nullptr;       // [ck (e_ck_len floats) | B image]; d_ck / d_bimg point into it
    uint8_t* h_opnd = nullptr;       // pinned mirror
    cudaEvent_t ev_h2d = nullptr;    // the last operand copy has left the pinned buffer
    bool h2d_pending = false;
    float* d_ck = nullptr;           // [passes][ck 64 | mult 64]: additive constant and quadratic-form multiplier per cluster
    float* h_ck = nullptr;           // pinned mirror
    float* d_den = nullptr;          // [memb_pitch] running / total log-denominator per event (Kmax > 64 only)
    int e_ck_len = 0;                // Kmax rounded up to whole passes of 64
    int e_NG = 0;
    // cudaFuncAttributeMaxDynamicSharedMemorySize is per device: the "already set" flags live with the (per-device) state
    bool attr_estep = false, attr_mstep = false;
    double h_shift[GMM_MAX_DIMENSIONS] = {0}, h_scale[GMM_MAX_DIMENSIONS] = {0};
};

static PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }
    return fn;
}

static int make_map_2d(CUtensorMap* m, const void* base, uint64_t dim0, uint64_t dim1, uint64_t stride1_bytes, uint32_t box0, uint32_t box1,
                       bool swizzle128 = false) {
    auto fn = encode_fn();
    if (!fn) return fail(GMM_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[2] = {dim0, dim1};
    cuuint64_t strides[1] = {stride1_bytes};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(GMM_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return GMM_OK;
}

bool tc_mstep_supported(int D, int K) {
    (void)K;
    return D == 4 || D == 8 || D == 12 || D == 16 || D == 20 || D == 24;
}
bool tc_estep_supported(int D, int K) { return (D == 8 || D == 16 || D == 24) && K >= 1 && K <= GMM_MAX_CLUSTERS; }

// bytes of the B image of one pass (64 clusters = MAXSG supergroups)
template <int D> static size_t ecfg_pass_bytes() { return (size_t)ECfg<D>::MAXSG * ECfg<D>::B_SG; }
static size_t pass_bytes_for(int D) {
    switch (D) { case 8: return ecfg_pass_bytes<8>(); case 16: return ecfg_pass_bytes<16>(); case 24: return ecfg_pass_bytes<24>(); default: return 0; }
}

int tc_create(TcState** out, const float* d_x_aos, const float* d_x_soa, int n, int D, int Kmax, float* d_memb, size_t memb_pitch, int num_sms,
              cudaStream_t stream) {
    (void)stream;
    TcState* t = new TcState();
    t->d_x = d_x_aos; t->d_x_soa = d_x_soa; t->d_memb = d_memb; t->memb_pitch = memb_pitch; t->n = n; t->D = D; t->Kmax = Kmax; t->num_sms = num_sms;
    *out = t;
    if (n <= 0 || !tc_mstep_supported(D, Kmax)) return GMM_OK;
    TC_CUDA_TRY(cudaMalloc(&t->d_shift_f, sizeof(float) * GMM_MAX_DIMENSIONS));
    TC_CUDA_TRY(cudaMalloc(&t->d_inv_scale_f, sizeof(float) * GMM_MAX_DIMENSIONS));
    TC_CUDA_TRY(cudaMalloc(&t->d_scale, sizeof(double) * GMM_MAX_DIMENSIONS));
    // tensor maps: SoA events [D][pitch] viewed as (events, dims) -> smem tile [D][32 events];
    // responsibilities [Kmax][pitch] viewed as (events, clusters)
    TC_CUDA_TRY(cudaMalloc(&t->d_z_soa, sizeof(float) * memb_pitch * D));
    if (int rc = make_map_2d(&t->tm_x, t->d_z_soa, (uint64_t)n, (uint64_t)D, (uint64_t)memb_pitch * 4, kTE, (uint32_t)D)) return rc;
    if (int rc = make_map_2d(&t->tm_g, d_memb, (uint64_t)n, (uint64_t)Kmax, (uint64_t)memb_pitch * 4, kTE, kNCL, /*swizzle128=*/true)) return rc;
    t->maps_ok = true;
    if (D == 8 || D == 16 || D == 24) {
        const int passes = (Kmax + 63) / 64;
        t->e_ck_len = passes * 64;
        t->bimg_bytes = (size_t)passes * pass_bytes_for(D);
        // one staging / device buffer [ck | B image]: the operand of an iteration travels in ONE H2D copy
        const size_t ck_bytes = sizeof(float) * 2 * t->e_ck_len;     // 512 B per pass: keeps the image 16-byte aligned
        TC_CUDA_TRY(cudaMalloc(&t->d_opnd, ck_bytes + t->bimg_bytes));
        TC_CUDA_TRY(cudaMallocHost(&t->h_opnd, ck_bytes + t->bimg_bytes));
        t->d_ck = reinterpret_cast<float*>(t->d_opnd);
        t->h_ck = reinterpret_cast<float*>(t->h_opnd);
        t->d_bimg = t->d_opnd + ck_bytes;
        t->h_bimg = t->h_opnd + ck_bytes;
        TC_CUDA_TRY(cudaEventCreateWithFlags(&t->ev_h2d, cudaEventDisableTiming));
        if (passes > 1) TC_CUDA_TRY(cudaMalloc(&t->d_den, sizeof(float) * memb_pitch));
        t->emap_ok = true;
    }
    const int rpp = 1 + 2 * (D / 4) + (D / 4) * (D / 2), nrows = 4 * ((rpp + 7) / 8) * 8;
    const int mt = (nrows + 127) / 128;
    {
        std::vector<int3> rm((size_t)mt * 128);
        std::vector<char> seen((size_t)num_features(D), 0);
        for (int row = 0; row < mt * 128; row++) {
            const RowInfo ri = tc_row_info(D, row);
            rm[row] = make_int3(ri.f, ri.i, ri.j);
            if (ri.f >= 0) {
                if (seen[ri.f]) return fail(GMM_ERR_STATE, "tensor M-step row map: a statistic is produced twice");
                seen[ri.f] = 1;
            }
        }
        for (char c : seen) if (!c) return fail(GMM_ERR_STATE, "tensor M-step row map: a statistic is not produced");
        TC_CUDA_TRY(cudaMalloc(&t->d_rowmap, sizeof(int3) * rm.size()));
        TC_CUDA_TRY(cudaMemcpy(t->d_rowmap, rm.data(), sizeof(int3) * rm.size(), cudaMemcpyHostToDevice));
    }
    const int ytiles = (Kmax + kNCL - 1) / kNCL;
    t->scratch_floats = (size_t)num_sms * ytiles * mt * 128 * kNCL;
    TC_CUDA_TRY(cudaMalloc(&t->d_scratch, sizeof(float) * t->scratch_floats));
    return GMM_OK;
}

bool tc_mstep_ready(const TcState* t) { return t && t->maps_ok && t->have_shift && t->mstep_ready; }
bool tc_estep_range_ok(const TcState* t) {
    if (!t || !t->have_shift) return false;
    for (int d = 0; d < t->D; d++)
        if (!(t->zmax[d] <= 16384.0f)) return false;
    return true;
}

void tc_destroy(TcState* t) {
    if (!t) return;
    cudaFree(t->d_shift_f); cudaFree(t->d_inv_scale_f); cudaFree(t->d_scale); cudaFree(t->d_scratch);
    cudaFree(t->d_opnd); cudaFree(t->d_den); cudaFree(t->d_z_soa); cudaFree(t->d_rowmap);
    if (t->h_opnd) cudaFreeHost(t->h_opnd);
    if (t->ev_h2d) cudaEventDestroy(t->ev_h2d);
    delete t;
}

int tc_set_shift_scale(TcState* t, double* shift, const double* scale, const double* xmin, const double* xmax, cudaStream_t stream) {
    if (!t || !t->maps_ok) return GMM_OK;
    float sf[GMM_MAX_DIMENSIONS] = {0}, isf[GMM_MAX_DIMENSIONS] = {0};
    double sc[GMM_MAX_DIMENSIONS] = {0};
    for (int d = 0; d < t->D; d++) {
        sf[d] = (float)shift[d];
        shift[d] = (double)sf[d];                       // the host finalisation must use the value the kernel used
        const double s = (scale && scale[d] > 0) ? scale[d] : 1.0;
        isf[d] = (float)(1.0 / s);
        sc[d] = 1.0 / (double)isf[d];
        t->h_shift[d] = shift[d];
        t->h_scale[d] = sc[d];
        // power-of-two bound of |z_d| = |(x - shift) * inv_scale| over the data (float arithmetic of the kernels + slack)
        const double za = std::fmax(std::fabs(xmax[d] - (double)sf[d]), std::fabs(xmin[d] - (double)sf[d])) * (double)isf[d] * (1.0 + 1e-6);
        int e2 = 0;
        if (za > 0 && std::isfinite(za)) { e2 = std::ilogb(za) + 1; }      // za < 2^e2
        t->zmax[d] = std::isfinite(za) ? (float)std::ldexp(1.0, e2) : INFINITY;
    }
    // Fixed-point quanta of the M-step feature rows: q = bound * 2^-11, magic = 1.5 * 2^23 * q, bound = the power-of-two
    // bound of |z| over all dimensions (squared for the product rows).  Data with outliers beyond 64 standard deviations
    // would leave too few bits below the quantum for the bulk of the events: such a data set is served by the FP64
    // SIMT M-step instead (tc_mstep_ready() false; GMM_PATH_TENSOR reports it).
    {
        float zb = 0.f;
        for (int d = 0; d < t->D; d++) zb = std::fmax(zb, t->zmax[d]);
        t->mstep_ready = zb <= 64.0f;                              // false for inf / nan too
        const double q = (double)zb / (double)(1 << kPhiBits);
        t->magic.lin = (float)(1.5 * 8388608.0 * q);
        t->magic.prod = (float)(1.5 * 8388608.0 * q * (double)zb);
    }
    TC_CUDA_TRY(cudaMemcpyAsync(t->d_shift_f, sf, sizeof(sf), cudaMemcpyHostToDevice, stream));
    TC_CUDA_TRY(cudaMemcpyAsync(t->d_inv_scale_f, isf, sizeof(isf), cudaMemcpyHostToDevice, stream));
    TC_CUDA_TRY(cudaMemcpyAsync(t->d_scale, sc, sizeof(sc), cudaMemcpyHostToDevice, stream));
    {
        dim3 grid((unsigned)std::min<long long>(4LL * t->num_sms, ((long long)t->n + 255) / 256), (unsigned)t->D);
        standardise_soa_kernel<<<grid, 256, 0, stream>>>(t->d_x_soa, t->d_z_soa, t->memb_pitch, t->n, t->D, t->d_shift_f, t->d_inv_scale_f);
        TC_CUDA_TRY(cudaGetLastError());
    }
    TC_CUDA_TRY(cudaStreamSynchronize(stream));         // the staging arrays live on this stack frame
    t->have_shift = true;
    return GMM_OK;
}

// Host side of the tensor E-step operand: per cluster the upper-triangular factor W of
// Rinv = W^T W (Cholesky of the symmetrised inverse covariance, double), expressed in the
// centred/scaled coordinates of the kernel, FP16 hi/lo split, laid out as the resident
// K-major B image ([supergroup][block][chunk][128 rows][16 B]).  Fails (GMM_ERR_STATE) when Rinv
// is not positive definite or the factor overflows FP16; the caller then uses the SIMT kernel
// for this state.

// float -> IEEE half bits, round to nearest even (normal, subnormal and zero; callers check the range)
static inline uint16_t f2h_bits(float f) {
    uint32_t x;
    std::memcpy(&x, &f, 4);
    const uint32_t sign = (x >> 16) & 0x8000u;
    x &= 0x7fffffffu;
    if (x >= 0x47800000u) return (uint16_t)(sign | 0x7c00u);
    if (x < 0x38800000u) {                      // below the smallest normal half: value * 2^24, rounded
        float a;
        std::memcpy(&a, &x, 4);
        return (uint16_t)(sign | (uint32_t)lrintf(a * 16777216.0f));
    }
    x += ((x >> 13) & 1u) + 0xfffu;
    return (uint16_t)(sign | ((x - 0x38000000u) >> 13));
}
static inline float h2f_bits(uint16_t h) {
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    const uint32_t em = h & 0x7fffu;
    float r;
    if (em >= 0x0400u) {                         // normal (inf/nan never produced here)
        const uint32_t x = sign | ((em << 13) + 0x38000000u);
        std::memcpy(&r, &x, 4);
    } else {
        r = (float)em * (1.0f / 16777216.0f);
        if (sign) r = -r;
    }
    return r;
}

// Operand rows of cluster k (k >= K: padding cluster of the last supergroup).  Returns 0, 1 (Rinv not positive
// definite) or 2 (factor outside the FP16 range).  Clusters are independent: callers may run this in parallel.
// Wext (optional): the upper-triangular factor W with Rinv = W^T W already computed by the caller in double (row-major
// [D][D]); otherwise it is derived here from host->Rinv.
template <int D>
static int bimg_cluster(TcState* t, const clusters_t* host, int k, int K, const double* Wext = nullptr) {
    using C = ECfg<D>;
    int bad = 0;
    {
        const int sg = k / C::GB, i = k % C::GB;
        // 16-byte K-chunk `chunk` of output column d of this cluster: K-major SWIZZLE_NONE image
        // [supergroup][block c = d/8][chunk][N = 16 clusters x 8 columns][16 B]
        auto rowp = [&](int d, int chunk) -> uint16_t* {
            const int c = d / 8, ncol = i * 8 + (d % 8);
            return reinterpret_cast<uint16_t*>(t->h_bimg + ((size_t)sg * C::CP + c) * C::B_BLOCK + (size_t)chunk * C::N * 16 + (size_t)ncol * 16);
        };
        if (k >= K) {                                    // padding cluster of the last supergroup: all-zero rows
            for (int d = 0; d < D; d++)
                for (int c = 0; c < C::NCHKB; c++) std::memset(rowp(d, c), 0, 16);
            return 0;
        }
        double A[D][D], Gc[D][D];
        const float* Ri = host->Rinv + (size_t)k * D * D;
        bool ok = true;
        if (Wext) {                                      // W = Gc^T
            for (int r = 0; r < D; r++)
                for (int j = 0; j < D; j++) Gc[r][j] = Wext[j * D + r];
        } else {
            for (int r = 0; r < D; r++)
                for (int j = 0; j < D; j++) { A[r][j] = 0.5 * ((double)Ri[r * D + j] + (double)Ri[j * D + r]); Gc[r][j] = 0.0; }
        }
        for (int j = 0; j < D && !Wext; j++) {                    // right-looking Cholesky A = Gc Gc^T (axpy updates vectorise)
            const double d = A[j][j];
            if (!(d > 0.0) || !std::isfinite(d)) { ok = false; break; }
            const double piv = std::sqrt(d), rp = 1.0 / piv;
            Gc[j][j] = piv;
            for (int r = j + 1; r < D; r++) Gc[r][j] = A[r][j] * rp;
            for (int r = j + 1; r < D; r++) {
                const double l = Gc[r][j];
                for (int cc = j + 1; cc <= r; cc++) A[r][cc] -= l * Gc[cc][j];
            }
        }
        if (!ok) return 1;
        // rows of W = Gc^T in the kernel's coordinates:  y_d = sum_j W'[d][j] z_j + v_d,  W'[d][j] = Gc[j][d] * scale_j (j >= d)
        alignas(32) float wrow[D][D];
        double vd[D];
        float amax = 0.f;
        for (int d = 0; d < D; d++) {
            double v = 0.0;
            for (int j = 0; j < D; j++) {
                const double w = (j >= d) ? Gc[j][d] : 0.0;
                v -= w * ((double)host->means[(size_t)k * D + j] - t->h_shift[j]);
                wrow[d][j] = (float)(w * t->h_scale[j]);
                amax = std::fmax(amax, std::fabs(wrow[d][j]));
            }
            vd[d] = v;
            amax = std::fmax(amax, (float)std::fabs(v));
        }
        if (!std::isfinite(amax)) return 2;
        // Per-cluster power-of-two scale: the largest operand entry lands in [2^12, 2^13) whatever the width of the
        // cluster (a cluster of relative width 1e-4 has factors ~1e4 - 1e5 and used to leave the FP16 range; a very wide
        // one pushed its lo parts into the FP16 subnormals).  The epilogue divides the squared norm by scale^2 (exact).
        int e2 = amax > 0.f ? 12 - std::ilogb(amax) : 0;
        e2 = e2 > 40 ? 40 : (e2 < -40 ? -40 : e2);
        for (int d = 0; d < D; d++) {
            for (int j = 0; j < D; j++) wrow[d][j] = std::ldexp(wrow[d][j], e2);
            vd[d] = std::ldexp(vd[d], e2);
            for (int c = 0; c < C::CP; c++) {
                uint16_t *ph = rowp(d, c), *pl = rowp(d, C::CP + c);      // x (zh_c, zl_c) [aliased], x zh_c
#if defined(__F16C__) && defined(__AVX__)
                const __m256 w8 = _mm256_load_ps(&wrow[d][8 * c]);
                const __m128i h8 = _mm256_cvtps_ph(w8, _MM_FROUND_TO_NEAREST_INT | _MM_FROUND_NO_EXC);
                const __m256 l8 = _mm256_sub_ps(w8, _mm256_cvtph_ps(h8));  // exact: hi is w rounded to 11 bits
                _mm_storeu_si128(reinterpret_cast<__m128i*>(ph), h8);
                _mm_storeu_si128(reinterpret_cast<__m128i*>(pl), _mm256_cvtps_ph(l8, _MM_FROUND_TO_NEAREST_INT | _MM_FROUND_NO_EXC));
#else
                for (int e = 0; e < 8; e++) {
                    const uint16_t wh = f2h_bits(wrow[d][8 * c + e]);
                    ph[e] = wh;
                    pl[e] = f2h_bits(wrow[d][8 * c + e] - h2f_bits(wh));
                }
#endif
            }
            const float vf = (float)vd[d];
            if (!(std::fabs(vf) < 6.0e4f)) bad = 2;
            uint16_t* pv = rowp(d, 2 * C::CP);
            const uint16_t vh = f2h_bits(vf);
            std::memset(pv, 0, 16);
            pv[0] = vh;
            pv[1] = f2h_bits((float)(vd[d] - (double)h2f_bits(vh)));
            if (C::NCHKB > 2 * C::CP + 1) std::memset(rowp(d, 2 * C::CP + 1), 0, 16);
        }
        float* ckp = t->h_ck + (size_t)(k / 64) * 128 + (k % 64);
        ckp[0] = host->constant[k] + logf(host->pi[k]);      // additive term of estep1 (gaussian_kernel.cu:442)
        ckp[64] = (float)std::ldexp(-0.5 * 1.4426950408889634, -2 * e2);
    }
    return bad;
}

static int bimg_cluster_any(TcState* t, const clusters_t* host, int k, int K, const double* Wext = nullptr) {
    switch (t->D) {
        case 8: return bimg_cluster<8>(t, host, k, K, Wext);
        case 16: return bimg_cluster<16>(t, host, k, K, Wext);
        case 24: return bimg_cluster<24>(t, host, k, K, Wext);
        default: return 3;
    }
}

int tc_params_begin(TcState* t, int K, cudaStream_t stream) {
    if (!t || !t->emap_ok) return fail(GMM_ERR_STATE, "tensor E-step not initialised for this shape");
    if (!t->have_shift) return fail(GMM_ERR_STATE, "tensor E-step needs the global moments (shift/scale) first");
    (void)stream;
    if (t->h2d_pending) {                                // the previous copy out of the pinned buffer must have finished
        TC_CUDA_TRY(cudaEventSynchronize(t->ev_h2d));
        t->h2d_pending = false;
    }
    for (int k = K; k < t->e_ck_len; k++) {               // padding clusters: never win the log-sum-exp
        float* ckp = t->h_ck + (size_t)(k / 64) * 128 + (k % 64);
        ckp[0] = -1e30f;
        ckp[64] = 0.f;
    }
    return GMM_OK;
}
int tc_params_padded(const TcState*, int K) { return (K + 15) / 16 * 16; }
int tc_params_cluster(TcState* t, const clusters_t* host, int k, int K) { return bimg_cluster_any(t, host, k, K); }
int tc_params_cluster_w(TcState* t, const clusters_t* host, int k, int K, const double* W) { return bimg_cluster_any(t, host, k, K, W); }
int tc_params_commit(TcState* t, int K, int bad, cudaStream_t stream) {
    if (bad == 1) return fail(GMM_ERR_STATE, "tensor E-step: inverse covariance of a cluster is not positive definite");
    if (bad == 2) return fail(GMM_ERR_STATE, "tensor E-step: whitening factor exceeds the FP16 range");
    if (bad) return fail(GMM_ERR_ARG, "tensor E-step: unsupported D");
    t->e_NG = (K + 15) / 16;
    // only the supergroups in use travel (the image is contiguous per supergroup; 4 supergroups = 64 clusters)
    const size_t used = (size_t)t->e_NG * (pass_bytes_for(t->D) / 4);
    TC_CUDA_TRY(cudaMemcpyAsync(t->d_opnd, t->h_opnd, sizeof(float) * 2 * t->e_ck_len + used, cudaMemcpyHostToDevice, stream));
    TC_CUDA_TRY(cudaEventRecord(t->ev_h2d, stream));
    t->h2d_pending = true;
    return GMM_OK;
}

// ===========================================================================
// Device-side M-step finalisation (one CTA per cluster): everything the host does between the reduced statistics
// and the next E-step — N, means, R (gaussian.cu:611-622, 663-679 with the rules of mstep_covariance1,
// gaussian_kernel.cu:658-675), inverse + constant + pi (constants_kernel, :172-259) and the E-step's resident
// operand (bimg_cluster above) — so that an EM iteration needs no device -> host -> device round trip
// (D2H of the statistics, thread-team wake-up, H2D of the operand: 60 us of an iteration that is 3.1 ms on one GPU
// and 0.6 ms on eight).  Same arithmetic as host_math.cpp (double, results stored as float): reverse Cholesky
// R = U U^T, W = U^-1, Rinv = W^T W, ln det R = 2 sum ln U_ii, here with a right-looking factorisation (rank-1
// updates of the trailing block, all threads) — the summation order differs from the host's dot products in the
// last bit of a double.  A cluster the host would NOT serve this way (R not positive definite, factor outside FP16)
// is not handled here: the kernel records the iteration in bad[0] (first failure wins), every later launch returns
// immediately, and the host replays from the last good parameter set through its own path (gmm_api.cu).
// Parameter set layout (floats, stride Kmax): N | pi | constant | means [Kmax][D] | R [Kmax][D][D] | Rinv [Kmax][D][D].
// ===========================================================================
__host__ __device__ inline size_t pset_off_means(int Kmax) { return 3 * (size_t)Kmax; }
__host__ __device__ inline size_t pset_off_R(int Kmax, int D) { return pset_off_means(Kmax) + (size_t)Kmax * D; }
__host__ __device__ inline size_t pset_off_Rinv(int Kmax, int D) { return pset_off_R(Kmax, D) + (size_t)Kmax * D * D; }

#ifdef GMM_FIN_PROF   // build-time phase stamps of finalize_params_kernel (CTA 0, thread 0 prints cycle deltas); off by default
#define FIN_STAMP(i) do { if (k == 0 && tid == 0) fin_t[i] = clock64(); } while (0)
#else
#define FIN_STAMP(i) do { } while (0)
#endif

template <int D> struct FinCfg { static constexpr int T = (D * D > 256 ? (D * D + 31) / 32 * 32 : 256), NW = T / 32; };   // a thread per matrix element

template <int D>
__global__ void __launch_bounds__(FinCfg<D>::T)
finalize_params_kernel(const double* __restrict__ stats, const float* __restrict__ avgvar, const float* __restrict__ shift_f,
                       const double* __restrict__ scale, float* __restrict__ set, int Kmax, int K, int kp,
                       uint8_t* __restrict__ bimg, float* __restrict__ ck, double* __restrict__ ll_out, int* __restrict__ bad, int iter,
                       int fault_iter) {
    // Latency-bound by construction (one CTA works through a 24 x 24 factorisation, 64 CTAs on 148 SMs; dependent FP64 operations
    // cost ~45 cycles each here — build-time phase stamps, GMM_FIN_PROF): one global round trip (the cluster's statistics row is staged
    // in shared memory), a THREAD PER MATRIX ELEMENT so that the rank-1 update of a column / row step is one pass (three serial passes of
    // 256 threads cost 880 cycles per column), one barrier per column of the factorisation and per row of the triangular inverse, and a
    // reciprocal square root of the pivot from the FP32 approximation + one Newton step (relative error ~1e-13: the results are stored as floats).
#ifdef GMM_FIN_PROF
    long long fin_t[10];
#endif
    using C = ECfg<D>;
    constexpr int T = FinCfg<D>::T, NW = FinCfg<D>::NW;
    constexpr int F = 1 + D + D * (D + 1) / 2;
    constexpr int LD = D + 1;
    const int k = blockIdx.x, tid = threadIdx.x;
    if (bad[0] >= 0) return;                                   // an earlier iteration failed: leave the last good state alone
    float* ckp = ck + (size_t)(k / 64) * 128 + (k % 64);
    const int sg = k / C::GB, ci = k % C::GB;
    auto rowp = [&](int d, int chunk) -> uint8_t* {            // 16-byte K chunk `chunk` of output column d (see bimg_cluster)
        return bimg + ((size_t)sg * C::CP + d / 8) * C::B_BLOCK + (size_t)chunk * C::N * 16 + (size_t)(ci * 8 + d % 8) * 16;
    };
    if (k >= K) {                                              // padding: never wins the log-sum-exp, all-zero operand rows
        if (tid == 0) { ckp[0] = -1e30f; ckp[64] = 0.f; }
        if (k < kp)
            for (int idx = tid; idx < D * C::NCHKB; idx += T) *reinterpret_cast<uint4*>(rowp(idx / C::NCHKB, idx % C::NCHKB)) = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    FIN_STAMP(0);
    __shared__ double sS[F + 3], sA[D][LD], sU[D][LD], sW[D][LD], srd[D], spiv[D], sdm[D], sscale[D], svd[D], sredd[NW];
    __shared__ float swr[D][LD], sredf[NW];
    __shared__ int sbad;
    // ---- stage: the statistics row, the S0 of every cluster (pi), shift / scale ----
    const double* s = stats + (size_t)k * F;
    for (int f = tid; f < F; f += T) sS[f] = s[f];
    double part = 0.0;
    for (int kk = tid; kk < K; kk += T) part += (double)(float)stats[(size_t)kk * F];
    double shift_d = 0.0;
    if (tid < D) { shift_d = (double)shift_f[tid]; sscale[tid] = scale[tid]; }
    const float av = avgvar[k];
    double ll_slot = 0.0;
    if (k == 0 && tid == 0) ll_slot = stats[(size_t)K * F];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((tid & 31) == 0) sredd[tid >> 5] = part;
    if (tid == 0) sbad = 0;
    __syncthreads();
    FIN_STAMP(1);
    const double S0 = sS[0];
    const float Nf = (float)S0;
    if (k == 0 && tid == 0) {
        *ll_out = ll_slot;                                     // log-likelihood of the E-step these statistics came from
        if (isnan(S0)) atomicMax(&sbad, 4);                    // the all-reduce kernel marks a failed exchange with NaN
        if (iter == fault_iter) atomicMax(&sbad, 1);           // test hook (option "finalize_fault_iter"): exercise the host replay
    }
    // ---- pi (compute_pi, gaussian_kernel.cu:172-193), means (gaussian.cu:611-622), R (:663-679, gaussian_kernel.cu:658-675) ----
    double sumN = 0.0;
#pragma unroll
    for (int w = 0; w < NW; w++) sumN += sredd[w];
    const float pik = Nf < 0.5f ? 1e-10f : (float)((double)Nf / sumN);
    if (tid < D) {
        const double m = (S0 != 0.0) ? sS[1 + tid] / S0 : 0.0;
        const float mu = (Nf > 0.5f) ? (float)(m + shift_d) : 0.0f;
        sdm[tid] = (double)mu - shift_d;                       // mu - shift as the operand rows need it
        set[pset_off_means(Kmax) + (size_t)k * D + tid] = mu;
    }
    {
        float* R = set + pset_off_R(Kmax, D) + (size_t)k * D * D;
        const double inv = 1.0 / (double)Nf;
        for (int idx = tid; idx < D * D; idx += T) {
            const int i = idx / D, j = idx % D;
            if (j > i) continue;
            float v;
            if (Nf > 0.5f) {
                const double mi = (S0 != 0.0) ? sS[1 + i] / S0 : 0.0;
                double cov = (Nf >= 1.0f) ? sS[1 + D + i * (i + 1) / 2 + j] - mi * sS[1 + j] : 0.0;
                if (i == j) cov += av;
                v = (float)(cov * inv);
            } else {
                v = (i == j) ? 1.0f : 0.0f;
            }
            R[i * D + j] = v; R[j * D + i] = v;
            sA[j][i] = (double)v;                              // upper triangle (row <= column) is what the factorisation reads
            if (i == j) sW[i][i] = 0.0; else { sW[j][i] = 0.0; sW[i][j] = 0.0; }
        }
    }
    __syncthreads();
    FIN_STAMP(2);
    // ---- R = U U^T from the last column: ONE barrier per column.  sA keeps the unscaled trailing block (upper triangle),
    //      the scaled column goes to sU, its reciprocal pivot to srd, the pivot's square to spiv (ln det) ----
    bool ok = true;
    for (int j = D - 1; j >= 0; j--) {
        const double d = sA[j][j];
        if (!(d > 0.0) || !isfinite(d)) { ok = false; break; }    // the same value in every thread
        const double y0 = (d > 1e-30 && d < 1e30) ? (double)rsqrtf((float)d) : rsqrt(d);   // 22 bits (float range), else the full routine
        const double rp = y0 * fma(-0.5 * d, y0 * y0, 1.5), invd = rp * rp;
        if (tid < j) sU[tid][j] = sA[tid][j] * rp;
        else if (tid == j) { srd[j] = rp; spiv[j] = d; }
        for (int idx = tid; idx < D * D; idx += T) {            // (i, m) with i <= m < j:  A[i][m] -= A[i][j] A[m][j] / d
            const int i = idx / D, m = idx % D;
            if (i <= m && m < j) sA[i][m] -= sA[i][j] * sA[m][j] * invd;
        }
        __syncthreads();
    }
    if (!ok) {
        if (tid == 0) { atomicCAS(&bad[0], -1, iter); atomicMax(&bad[1], 1); }
        return;
    }
    FIN_STAMP(3);
    // ---- W = U^-1 (upper triangular), row by row from the bottom, ONE barrier per row: when row m is final, every row i < m
    //      takes its term U[i][m] W[m][j]; the thread that completes row m - 1 scales it (W[i][j] = -(sum) / U[i][i]) ----
    if (tid < D) sW[tid][tid] = srd[tid];
    __syncthreads();
    for (int m = D - 1; m >= 1; m--) {
        for (int idx = tid; idx < D * D; idx += T) {
            const int i = idx / D, j = idx % D;
            if (i < m && j >= m) {
                double acc = sW[i][j] + sU[i][m] * sW[m][j];
                if (i == m - 1) acc = -acc * srd[i];
                sW[i][j] = acc;
            }
        }
        __syncthreads();
    }
    FIN_STAMP(4);
    // ---- Rinv = W^T W, ln det, constant (gaussian_kernel.cu:241), N, pi; operand rows: W'[d][j] = W[d][j] * scale_j, v = -W (mu - shift) ----
    {
        float* Ri = set + pset_off_Rinv(Kmax, D) + (size_t)k * D * D;
        for (int idx = tid; idx < D * D; idx += T) {
            const int i = idx / D, j = idx % D;
            if (j < i) continue;
            double v = 0.0;
#pragma unroll 4
            for (int m = 0; m <= i; m++) v += sW[m][i] * sW[m][j];
            Ri[i * D + j] = (float)v; Ri[j * D + i] = (float)v;
        }
    }
    FIN_STAMP(5);
    float amax = 0.f;
    for (int idx = tid; idx < D * D; idx += T) {
        const int d = idx / D, j = idx % D;
        const float w = (j >= d) ? (float)(sW[d][j] * sscale[j]) : 0.f;
        swr[d][j] = w;
        amax = fmaxf(amax, fabsf(w));
    }
    if (tid >= 64 && tid < 64 + D) {                              // (a warp of its own: the row sums are serial)
        const int d = tid - 64;
        double v = 0.0;
#pragma unroll 4
        for (int j = d; j < D; j++) v -= sW[d][j] * sdm[j];
        svd[d] = v;
        amax = fmaxf(amax, (float)fabs(v));
    }
    double ld2 = (tid >= 32 && tid < 32 + D) ? log(spiv[tid - 32]) : 0.0;   // ln det R = sum ln (pivot^2)
    if (tid >= 32 && tid < 64) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ld2 += __shfl_xor_sync(0xffffffffu, ld2, o);
        if (tid == 32) sredd[0] = ld2;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    if ((tid & 31) == 0) sredf[tid >> 5] = amax;
    __syncthreads();
    FIN_STAMP(6);
    const double ld = 0.5 * sredd[0];                          // sum ln U_jj
    const float cst = (float)(-D * 0.5 * log(2.0 * 3.1415926535897931) - 0.5 * (2.0 * ld));
    if (tid == 0) { set[k] = Nf; set[Kmax + k] = pik; set[2 * (size_t)Kmax + k] = cst; }
    amax = 0.f;
#pragma unroll
    for (int w = 0; w < NW; w++) amax = fmaxf(amax, sredf[w]);
    if (!isfinite(amax)) {
        if (tid == 0) { atomicCAS(&bad[0], -1, iter); atomicMax(&bad[1], 2); }
        return;
    }
    // per-cluster power-of-two scale: the largest operand entry lands in [2^12, 2^13) (see bimg_cluster)
    int e2 = amax > 0.f ? 12 - ilogbf(amax) : 0;
    e2 = e2 > 40 ? 40 : (e2 < -40 ? -40 : e2);
    for (int idx = tid; idx < D * C::CP; idx += T) {
        const int d = idx / C::CP, c = idx % C::CP;
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const float w0 = ldexpf(swr[d][8 * c + 2 * e], e2), w1 = ldexpf(swr[d][8 * c + 2 * e + 1], e2);
            const __half2 h = __floats2half2_rn(w0, w1);
            const float2 hf = __half22float2(h);
            hi[e] = *reinterpret_cast<const uint32_t*>(&h);
            lo[e] = pack_half2(w0 - hf.x, w1 - hf.y);          // exact difference: hi is w rounded to 11 bits
        }
        *reinterpret_cast<uint4*>(rowp(d, c)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);             // x (zh_c, zl_c) [aliased]
        *reinterpret_cast<uint4*>(rowp(d, C::CP + c)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);     // x zh_c
    }
    if (tid >= 128 && tid < 128 + D) {
        const int d = tid - 128;
        const double vs = ldexp(svd[d], e2);
        const float vf = (float)vs;
        if (!(fabsf(vf) < 6.0e4f)) atomicMax(&sbad, 2);
        const __half vh = __float2half_rn(vf);
        const __half vl = __float2half_rn((float)(vs - (double)__half2float(vh)));
        const uint32_t p = (uint32_t)__half_as_ushort(vh) | ((uint32_t)__half_as_ushort(vl) << 16);
        *reinterpret_cast<uint4*>(rowp(d, 2 * C::CP)) = make_uint4(p, 0u, 0u, 0u);
        if (C::NCHKB > 2 * C::CP + 1) *reinterpret_cast<uint4*>(rowp(d, 2 * C::CP + 1)) = make_uint4(0u, 0u, 0u, 0u);
    }
    if (tid == 0) {
        ckp[0] = cst + logf(pik);                              // additive term of estep1 (gaussian_kernel.cu:442)
        ckp[64] = (float)ldexp(-0.5 * 1.4426950408889634, -2 * e2);
    }
    __syncthreads();
    FIN_STAMP(7);
#ifdef GMM_FIN_PROF
    if (k == 0 && tid == 0)
        printf("fin phases (cycles): stage %lld  means+R %lld  cholesky %lld  inverse %lld  Rinv %lld  rows+v+log %lld  operand %lld\n",
               fin_t[1] - fin_t[0], fin_t[2] - fin_t[1], fin_t[3] - fin_t[2], fin_t[4] - fin_t[3], fin_t[5] - fin_t[4], fin_t[6] - fin_t[5], fin_t[7] - fin_t[6]);
#endif
    if (tid == 0 && sbad) { atomicCAS(&bad[0], -1, iter); atomicMax(&bad[1], sbad); }
}

size_t tc_param_set_floats(int Kmax, int D) { return (size_t)Kmax * (3 + (size_t)D + 2 * (size_t)D * D); }
size_t tc_param_set_off(int Kmax, int D, int which) {
    switch (which) {
        case 0: return 0;                                   // N
        case 1: return (size_t)Kmax;                        // pi
        case 2: return 2 * (size_t)Kmax;                    // constant
        case 3: return pset_off_means(Kmax);
        case 4: return pset_off_R(Kmax, D);
        default: return pset_off_Rinv(Kmax, D);
    }
}
bool tc_finalize_supported(const TcState* t, int K) {
    return t && t->emap_ok && t->have_shift && tc_estep_supported(t->D, K) && tc_estep_range_ok(t);
}
int tc_launch_finalize(TcState* t, int K, const double* d_stats, const float* d_avgvar, float* d_set, double* d_ll, int* d_bad, int iter,
                       int fault_iter, cudaStream_t stream) {
    if (!tc_finalize_supported(t, K)) return fail(GMM_ERR_STATE, "device-side finalisation not available for this state");
    const int kp = tc_params_padded(t, K);
    const int grid = ((K + 63) / 64) * 64;                     // whole passes: the padding clusters of the last pass get their constants
#define GMM_FIN(d) finalize_params_kernel<d><<<grid, FinCfg<d>::T, 0, stream>>>(d_stats, d_avgvar, t->d_shift_f, t->d_scale, d_set, t->Kmax, K, kp, \
                                                                     t->d_bimg, t->d_ck, d_ll, d_bad, iter, fault_iter)
    switch (t->D) {
        case 8: GMM_FIN(8); break;
        case 16: GMM_FIN(16); break;
        case 24: GMM_FIN(24); break;
        default: return fail(GMM_ERR_ARG, "device-side finalisation: unsupported D");
    }
#undef GMM_FIN
    TC_CUDA_TRY(cudaGetLastError());
    t->e_NG = (K + 15) / 16;
    return GMM_OK;
}

template <int D>
static int launch_estep_d(TcState* t, int K, double* d_ll, cudaStream_t stream) {
    using C = ECfg<D>;
    static_assert(C::SMEM_BYTES <= 232448, "shared memory budget");
    if (!t->attr_estep) {
        TC_CUDA_TRY(cudaFuncSetAttribute(estep_tc_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
        t->attr_estep = true;
    }
    const int ntiles = (t->n + 127) / 128;
    int grid = t->num_sms;
    if (grid > ntiles) grid = ntiles;
    if (grid < 1) grid = 1;
    const int NP = (K + 63) / 64;
    if (NP > 1 && !t->d_den) return fail(GMM_ERR_STATE, "tensor E-step: context was created for at most 64 clusters");
    // P passes of 64 clusters: log-denominators of passes 0 .. P-2 (mode 1), then the last pass writes its final
    // responsibilities and the events' total log-denominators (mode 2, or mode 0 when P = 1), then passes 0 .. P-2 write
    // theirs against those totals (mode 3): 2P - 1 launches, every responsibility stored once
    auto launch = [&](int p, int mode, const float* den_in, float* den_out) {
        const int Kp = K - 64 * p < 64 ? K - 64 * p : 64;
        estep_tc_kernel<D><<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(
            t->d_x, t->d_bimg + (size_t)p * C::MAXSG * C::B_SG, t->d_ck + 128 * p, t->d_shift_f, t->d_inv_scale_f,
            t->d_memb + (size_t)(64 * p) * t->memb_pitch, t->memb_pitch, t->n, Kp, (Kp + C::GB - 1) / C::GB, d_ll, mode, den_in, den_out);
        return cudaGetLastError();
    };
    if (NP == 1) TC_CUDA_TRY(launch(0, 0, nullptr, nullptr));
    else {
        for (int p = 0; p + 1 < NP; p++) TC_CUDA_TRY(launch(p, 1, p ? t->d_den : nullptr, t->d_den));
        TC_CUDA_TRY(launch(NP - 1, 2, t->d_den, t->d_den));
        for (int p = 0; p + 1 < NP; p++) TC_CUDA_TRY(launch(p, 3, t->d_den, nullptr));
    }
    return GMM_OK;
}

int tc_launch_estep(TcState* t, int K, double* d_ll, cudaStream_t stream) {
    if (!t || !t->emap_ok) return fail(GMM_ERR_STATE, "tensor E-step not initialised for this shape");
    switch (t->D) {
        case 8: return launch_estep_d<8>(t, K, d_ll, stream);
        case 16: return launch_estep_d<16>(t, K, d_ll, stream);
        case 24: return launch_estep_d<24>(t, K, d_ll, stream);
        default: return fail(GMM_ERR_ARG, "tensor E-step: unsupported D");
    }
}

template <int D>
static int launch_mstep_d(TcState* t, int K, double* d_stats, cudaStream_t stream) {
    using C = MCfg<D>;
    static_assert(C::SMEM_BYTES <= 232448, "shared memory budget");
    static_assert(C::TMEM_COLS <= 512, "TMEM budget");
    if (!t->attr_mstep) {
        TC_CUDA_TRY(cudaFuncSetAttribute(mstep_tc_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
        t->attr_mstep = true;
    }
    int gx = t->num_sms;
    int per = (t->n + gx - 1) / gx;
    per = (per + kTE - 1) / kTE * kTE;
    gx = (t->n + per - 1) / per;
    const int gy = (K + kNCL - 1) / kNCL;
    if ((size_t)gx * gy * C::MT * 128 * kNCL > t->scratch_floats) return fail(GMM_ERR_STATE, "tensor M-step scratch too small");
    dim3 grid(gx, gy);
    mstep_tc_kernel<D><<<grid, kMThreads, C::SMEM_BYTES, stream>>>(t->tm_x, t->tm_g, t->n, t->d_scratch, per, t->magic);
    TC_CUDA_TRY(cudaGetLastError());
    mstep_tc_finalize_kernel<<<C::NCHUNK * 8, 256, 0, stream>>>(t->d_scratch, gx, C::MT, K, C::F, t->d_rowmap, t->d_scale, d_stats);
    TC_CUDA_TRY(cudaGetLastError());
    return GMM_OK;
}

int tc_launch_mstep(TcState* t, int K, double* d_stats, cudaStream_t stream) {
    if (!t || !t->maps_ok) return fail(GMM_ERR_STATE, "tensor-core M-step not initialised for this shape");
    if (!t->have_shift) return fail(GMM_ERR_STATE, "tensor-core M-step needs gmm_seed (shift/scale) first");
    if (!t->mstep_ready) return fail(GMM_ERR_STATE, "tensor-core M-step: the data range exceeds the fixed-point operand budget");
    switch (t->D) {
        case 4: return launch_mstep_d<4>(t, K, d_stats, stream);
        case 8: return launch_mstep_d<8>(t, K, d_stats, stream);
        case 12: return launch_mstep_d<12>(t, K, d_stats, stream);
        case 16: return launch_mstep_d<16>(t, K, d_stats, stream);
        case 20: return launch_mstep_d<20>(t, K, d_stats, stream);
        case 24: return launch_mstep_d<24>(t, K, d_stats, stream);
        default: return fail(GMM_ERR_ARG, "tensor-core M-step: unsupported D");
    }
}

}  // namespace gmm
