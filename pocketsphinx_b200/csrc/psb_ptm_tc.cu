// psb_ptm_tc.cu -- PTM top-N selection without the recurrence over time: a tensor-core filter,
// exact rescoring of the few survivors, and a sequential fix-up for exact ties.
//
// What the reference computes per frame and (codebook, stream) pair is a list of four codewords:
// eval_topn re-scores last frame's four, eval_cb scans all codewords in order and inserts every one
// whose distance beats the current worst (ptm_mgau.c:88-226).  ptm_topnq_kernel (psb_ptm.cu)
// follows that literally: time is sequential, every frame evaluates all 256 distances.  Two facts
// make most of that work unnecessary, with the SAME bits in the result:
//
//  (1) The list does not depend on the previous frame unless scores tie.  Let s(1) >= s(2) >= ...
//      be the truncated integer scores of ALL codewords of the pair in this frame.  The worst
//      listed score only rises during a scan and every codeword that is rejected or evicted has a
//      score <= the final worst, so the final worst is >= s(4).  If s(1) > s(2) > s(3) > s(4) > s(5),
//      each of the four best is accepted when the scan (or eval_topn) meets it -- at most three
//      listed scores exceed its own and none equals it, so the worst listed score is smaller and
//      `d >= (float)worst` holds -- and can never be evicted.  The list is then exactly those four
//      in descending order, whatever the seeds were.  Only when two of the five best integer scores
//      coincide do the order-dependent rules (`>=` shifting, strict `>` in eval_topn,
//      skip-if-listed) matter; those frames are flagged and redone by ptm_fixup_warp_kernel, which
//      replays the reference's loop literally with the previous frame's list as seeds.
//  (2) The five best can be found without computing 256 exact distances.  With y = x - m (m = the
//      codebook's mean centre) the exponent d = det - sum_j v_j (y_j - mu'_j)^2 is the inner product
//      of X = (y_j^2, y_j, 1) with W_c = (-v_cj, 2 v_cj mu'_cj, det_c - sum_j v_cj mu'_cj^2): one
//      [frames x 32] x [32 x n_density] TF32 GEMM per pair on the tensor cores (tcgen05.mma, three
//      products of high and low TF32 halves; W is split on the host).  Its result a_c differs from the
//      reference's float d_c by at most eps = ERR * (sum_j Amax_j y_j^2 + Bmax_j |y_j| + Cmax), a
//      bound every row computes for itself (Amax/Bmax/Cmax: per-pair maxima of |W| entries).  Five
//      distinct codewords with a_c >= L0 (the four per-lane row maxima of the accumulator fragment
//      and the best of the four runner-up half maxima) give the integer L' = floor(L0 - eps) - 1
//      <= s(5) - 1, and every codeword with s_c >= s(5) has d_c > L', hence a_c >= L' - eps: the
//      candidate set C (about a dozen of 256 on the BASELINE shape).  Among them, with a(4) the
//      fourth largest a_c, only E = {c : a_c >= a(4) - 2 eps - 1} can reach the four best or tie with
//      them (anything else has d_c < d(4) - 1, i.e. a strictly smaller integer score): E (five to
//      seven codewords) is what gets the reference's exact float arithmetic.
//
// The exact stage: a row the filter values leave in doubt goes on a work list that ptm_tc_exact_kernel
// rescores, one thread per row, with the reference's float arithmetic over its candidates (over all
// codewords when the row's candidate list overflowed its shared-memory slots).
//
// Nothing here is approximate in its output: tests/test_gpu_parity.py compares every record with the
// oracle's lists, PSB_TC_CHECK=1 makes the filter kernel measure max |a_c - d_c| / eps on the device.
#include "psb_gau.cuh"
#include "psb_internal.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace {

constexpr int TC_ROWS = 128;          // frames per CTA (4 warps x 2 m-tiles x 16 rows)
constexpr int TC_K = 32;              // GEMM depth: 2 * FL + 1 <= 32
constexpr int TC_CAP = 18;            // candidate slots per row: the row's X storage, 144 B / 8 B
constexpr float TC_ERR = 1.0f / 262144.f;  // 2^-18 of the magnitude sum S: 3 x TF32 leaves 3 * 2^-22 per product, the rest is
                                           // room for the tensor core's fp32 accumulation (<= 2^-23 per step assumed, 12 steps per
                                           // chain) and the reference's own 52 roundings; PSB_TC_CHECK=1 measures what is used of it

__device__ __forceinline__ float to_tf32(float x)
{
    unsigned r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

struct Top5 {
    int s[5];
    unsigned c;           // codewords of entries 0..3, byte j = entry j
    int c4;               // codeword of entry 4 (unused by the record)
    int n;
};

__device__ __forceinline__ void top5_insert(Top5 &t, int s, int c)
{
    // sorted descending; equal scores keep arrival order (irrelevant: ties are redone by the fix-up)
    int p = 0;
#pragma unroll
    for (int j = 0; j < 5; ++j) p += (j < t.n && t.s[j] >= s) ? 1 : 0;
    if (p >= 5) return;
#pragma unroll
    for (int j = 4; j >= 1; --j)
        if (j > p) t.s[j] = t.s[j - 1];
#pragma unroll
    for (int j = 0; j < 5; ++j)
        if (j == p) t.s[j] = s;
    // codeword bytes: entries p..3 move up one byte, entry 3 falls into c4
    if (p < 4) {
        const unsigned lowmask = p == 0 ? 0u : (0xffffffffu >> (32 - 8 * p));
        t.c4 = (int)(t.c >> 24);
        t.c = (t.c & lowmask) | ((unsigned)c << (8 * p)) | ((t.c << 8) & ~(lowmask | (0xffu << (8 * p))));
    }
    else
        t.c4 = c;
    if (t.n < 5) ++t.n;
}

// ---------------------------------------------------------------------------------------
// The filter on the 5th-generation tensor cores (tcgen05): mma.sync tops out
// near 290 TFLOP/s of TF32 (8 cycles per m16n8k8 and sub-core), which makes the 3 x TF32 GEMM -- 6.2 TFLOP
// per 10^6-frame batch -- the longest stage.  Here one elected thread issues twelve
// tcgen05.mma.cta_group::1.kind::tf32 (M 128 frames x N n_density x K 8; lo*hi, hi*lo, hi*hi over four
// K steps) per 128-frame tile, A (the X tile, split into TF32 halves) and B (W, both halves) in shared memory
// in the canonical K-major no-swizzle layout (8-row x 16-byte core matrices; descriptors built below), the
// fp32 accumulator in TENSOR MEMORY: 128 lanes x n_density columns.  tcgen05.commit arrives on an mbarrier;
// after the wait every thread reads ITS OWN frame's row (TMEM lane = frame = thread) with tcgen05.ld.32x32b in
// slabs of 32 columns, twice: group maxima -> threshold, then the columns above it.  No accumulator registers
// across the sweep, no shuffles, no shared-memory atomics -- the whole selection is thread-private.  A CTA keeps
// W resident and walks `tiles_per_cta` consecutive tiles of its pair.
__device__ __forceinline__ uint64_t umma_smem_desc(const void *p, unsigned lbo_bytes, unsigned sbo_bytes)
{
    // cute::UMMA::SmemDescriptor (mma_sm100_desc.hpp): start address, leading / stride byte offsets in 16-byte units,
    // version 1 (Blackwell) at bit 46, base offset 0, layout type 0 = no swizzle
    const uint64_t a = (uint64_t)((unsigned)__cvta_generic_to_shared(p) >> 4) & 0x3fffu;
    return a | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}

__device__ __forceinline__ void umma_tf32(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc, unsigned accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}

__device__ __forceinline__ void tmem_ld32_issue(unsigned taddr, float (&v)[32])
{
    // destination = the caller's registers themselves (bit-size operands take .f32 registers): no move may sit between the
    // load and the wait that makes them valid
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]), "=f"(v[9]),
          "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]), "=f"(v[16]), "=f"(v[17]), "=f"(v[18]),
          "=f"(v[19]), "=f"(v[20]), "=f"(v[21]), "=f"(v[22]), "=f"(v[23]), "=f"(v[24]), "=f"(v[25]), "=f"(v[26]), "=f"(v[27]),
          "=f"(v[28]), "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// the same wait, but the compiler is told that the slab's registers pass through it: nothing that reads them can be
// scheduled above the wait when the load was issued earlier (software pipelining of the sweeps)
__device__ __forceinline__ void tmem_wait_ld_dep(float (&v)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]), "+f"(v[8]), "+f"(v[9]),
                   "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15]), "+f"(v[16]), "+f"(v[17]), "+f"(v[18]),
                   "+f"(v[19]), "+f"(v[20]), "+f"(v[21]), "+f"(v[22]), "+f"(v[23]), "+f"(v[24]), "+f"(v[25]), "+f"(v[26]), "+f"(v[27]),
                   "+f"(v[28]), "+f"(v[29]), "+f"(v[30]), "+f"(v[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(unsigned taddr, float (&v)[32])
{
    tmem_ld32_issue(taddr, v);
    tmem_wait_ld();
}

__device__ __forceinline__ void mbar_init1(uint64_t *bar)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)));
}
__device__ __forceinline__ void mbar_wait_parity(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TCW_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra TCD_%=;\n"
        "bra TCW_%=;\n"
        "TCD_%=:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)),
        "r"(parity)
        : "memory");
}

// Filter + resolution for a pair's tiles of 128 frames.
//   wumma   [K][2][8][ND][4] float   W halves (high, low) in the canonical K-major layout: chunk kc holds k = 4 kc .. 4 kc + 3
//   cen     [K][16]                    centre m
//   bnd     [K][32]                    Amax[FL], Bmax[FL], Cmax at [2 FL]
//   rec     scalar records {det, mu0, v0, ...} of the model (exact distances of ambiguous rows, read through L1/L2)
//   flags   [K][flag_words]            bit (row & 31) of word row >> 5: frame must be redone by the fix-up
//   check   (debug) float[2]: max over everything of |a_c - d_c| / eps, and of the candidate count
//   stats   (debug) unsigned long long[4]: rows, rows resolved from the filter alone, exact distances, tie flags
template <int FL, int ND, bool CHECK>
__global__ void __launch_bounds__(TC_ROWS, 2)
ptm_tc5_kernel(const float *__restrict__ feats, long long total, int D, const int32_t *__restrict__ featoff,
               const int32_t *__restrict__ klist, const float *__restrict__ wumma, const float *__restrict__ cen,
               const float *__restrict__ bnd, const float *__restrict__ rec, const size_t *__restrict__ rec_off,
               int4 *__restrict__ out, unsigned *__restrict__ flags, long long flag_words, int K, int n_feat,
               int tiles_per_cta, uint4 *__restrict__ items, unsigned *__restrict__ n_items, unsigned item_cap,
               float *__restrict__ check, unsigned long long *__restrict__ stats)
{
    constexpr int RF = (1 + 2 * FL + 3) / 4 * 4;
    constexpr int GW = ND / 8;                           // columns per maximum group: 8 groups per row
    static_assert(2 * FL + 1 <= TC_K && ND % 32 == 0 && ND <= 256 && ND % 64 == 0, "shape");
    extern __shared__ __align__(128) unsigned char t5_smem[];
    float *sW = reinterpret_cast<float *>(t5_smem);                                   // [2][8][ND][4]
    float *sX = sW + 2 * 8 * ND * 4;                                                  // [2][8][128][4]; after the MMA: lists + staging
    // thread-private and transposed ([slot][thread]: conflict-free): candidate values, candidate columns, one 32-column slab
    float *Lv = sX;                                                                   // [TC_CAP][TC_ROWS]
    unsigned char *Lc = reinterpret_cast<unsigned char *>(Lv + TC_CAP * TC_ROWS);     // [TC_CAP][TC_ROWS]
    float *stage = reinterpret_cast<float *>(Lc + ((TC_CAP * TC_ROWS + 15) & ~15));   // [32][TC_ROWS]
    static_assert(TC_CAP * TC_ROWS * 5 + 16 + 32 * TC_ROWS * 4 <= 2 * 8 * TC_ROWS * 16, "lists + staging must fit the X tile");
    __shared__ __align__(8) uint64_t mma_done;
    __shared__ unsigned tmem_base_s;

    // grid: x = pair (fastest), y = group of tiles: CTAs that run together read the SAME frames for different pairs, so
    // the feature rows come out of L2 (with tiles fastest every pair re-read the whole feature matrix from HBM: 23 GB
    // per 998 k frames in the first ncu capture) while the 126 W blocks (8 MB) stay L2-resident
    const int k = klist[blockIdx.x];
    const int f = k % n_feat;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int r = tid;                                   // this thread's frame of the tile

    if (warp == 0) {                                     // 256 (or fewer) TMEM columns for the accumulator
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(&tmem_base_s)),
                     "n"(ND < 32 ? 32 : ND));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        mbar_init1(&mma_done);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {
        const float4 *src = reinterpret_cast<const float4 *>(wumma + (size_t)k * 2 * 8 * ND * 4);
        float4 *dst = reinterpret_cast<float4 *>(sW);
        for (int i = tid; i < 2 * 8 * ND; i += TC_ROWS) dst[i] = src[i];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem_d = tmem_base_s;
    // instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A / B tf32, both K-major, N >> 3, M >> 4
    constexpr unsigned IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(ND >> 3) << 17) | ((unsigned)(TC_ROWS >> 4) << 24);
    const float *m = cen + (size_t)k * 16, *bb = bnd + (size_t)k * 32;
    const float *rc = rec + rec_off[k];

    // the next tile's feature row is fetched while this tile's GEMM runs
    float xn[FL];
    {
        const long long r0 = (long long)blockIdx.y * tiles_per_cta * TC_ROWS + r;
        const float *p = feats + (r0 < total ? r0 : 0) * D + featoff[f];
#pragma unroll
        for (int j = 0; j < FL; ++j) xn[j] = r0 < total ? p[j] : 0.f;
    }
    for (int tile = 0; tile < tiles_per_cta; ++tile) {
        const long long row = ((long long)blockIdx.y * tiles_per_cta + tile) * TC_ROWS + r;
        if (row - r >= total) break;                     // uniform: the whole tile lies past the end
        const bool valid = row < total;
        // ---- this thread's frame: X row (TF32 halves, canonical layout) and its error bound ----
        float x[FL], ee;
        {
            float v[TC_K];
            float S = bb[2 * FL];
#pragma unroll
            for (int j = 0; j < FL; ++j) {
                x[j] = xn[j];
                const float y = __fsub_rn(x[j], m[j]);
                const float y2 = __fmul_rn(y, y);
                v[j] = y2;
                v[FL + j] = y;
                S = __fadd_ru(S, __fmul_ru(bb[j], y2));               // no FMA anywhere in these kernels: tests/test_abi.py greps for it
                S = __fadd_ru(S, __fmul_ru(bb[FL + j], fabsf(y)));
            }
            v[2 * FL] = 1.0f;
#pragma unroll
            for (int j = 2 * FL + 1; j < TC_K; ++j) v[j] = 0.f;
            ee = __fadd_ru(__fmul_ru(S, TC_ERR), 2.0f);
#pragma unroll
            for (int kc = 0; kc < 8; ++kc) {
                float4 h, l;
                h.x = to_tf32(v[4 * kc]); h.y = to_tf32(v[4 * kc + 1]); h.z = to_tf32(v[4 * kc + 2]); h.w = to_tf32(v[4 * kc + 3]);
                l.x = to_tf32(__fsub_rn(v[4 * kc], h.x)); l.y = to_tf32(__fsub_rn(v[4 * kc + 1], h.y));
                l.z = to_tf32(__fsub_rn(v[4 * kc + 2], h.z)); l.w = to_tf32(__fsub_rn(v[4 * kc + 3], h.w));
                reinterpret_cast<float4 *>(sX)[kc * TC_ROWS + r] = h;
                reinterpret_cast<float4 *>(sX)[(8 + kc) * TC_ROWS + r] = l;
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy writes -> visible to the tensor core
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            // chunk kc of A at sX + kc * 2048 B (128 rows x 16 B), of B at sW + kc * ND * 16 B; core matrices 128 B apart
            for (int pass = 0; pass < 3; ++pass) {        // lo*hi, hi*lo, hi*hi
                const int ha = pass == 0 ? 1 : 0, hb = pass == 1 ? 1 : 0;
                for (int ks = 0; ks < 4; ++ks) {
                    const uint64_t ad = umma_smem_desc(sX + ((size_t)(ha * 8 + 2 * ks) * TC_ROWS) * 4, TC_ROWS * 16, 128);
                    const uint64_t bd = umma_smem_desc(sW + ((size_t)(hb * 8 + 2 * ks) * ND) * 4, ND * 16, 128);
                    umma_tf32(tmem_d, ad, bd, IDESC, (pass | ks) ? 1u : 0u);
                }
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                             (unsigned)__cvta_generic_to_shared(&mma_done))
                         : "memory");
        }
        if (tile + 1 < tiles_per_cta) {
            const long long rn = row + TC_ROWS;
            const float *p = feats + (rn < total ? rn : 0) * D + featoff[f];
#pragma unroll
            for (int j = 0; j < FL; ++j) xn[j] = rn < total ? p[j] : 0.f;
        }
        mbar_wait_parity(&mma_done, (unsigned)tile & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

        // ---- this thread's row of the accumulator: group maxima, threshold, the columns above it ----
        const unsigned trow = tmem_d + ((unsigned)((warp & 3) * 32) << 16);
        float gm[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) gm[i] = -INFINITY;
        auto maxima = [&](int c0, const float (&v)[32]) {
            if (GW >= 32) {
                // a tree, not a chain: with two warps per scheduler the dependent-issue latency is what counts
                float m8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) m8[i] = fmaxf(fmaxf(v[i], v[i + 8]), fmaxf(v[i + 16], v[i + 24]));
                const float mx = fmaxf(fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])), fmaxf(fmaxf(m8[4], m8[5]), fmaxf(m8[6], m8[7])));
                const int gi = c0 / GW;
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if (q == gi) gm[q] = fmaxf(gm[q], mx);
            }
            else {
                constexpr int PER = 32 / (GW < 32 ? GW : 32);       // groups inside one 32-column slab
#pragma unroll
                for (int s2 = 0; s2 < PER; ++s2) {
                    float mx = v[s2 * GW];
#pragma unroll
                    for (int i = 1; i < GW; ++i) mx = fmaxf(mx, v[s2 * GW + i]);
                    const int gi = c0 / GW + s2;
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        if (q == gi) gm[q] = fmaxf(gm[q], mx);
                }
            }
        };
        {   // two slabs in flight: the load of the next one runs while this one is reduced
            float va[32], vb[32];
            tmem_ld32_issue(trow, va);
#pragma unroll 1
            for (int c0 = 0; c0 < ND; c0 += 64) {
                tmem_wait_ld_dep(va);
                tmem_ld32_issue(trow + c0 + 32, vb);
                maxima(c0, va);
                tmem_wait_ld_dep(vb);
                if (c0 + 64 < ND) tmem_ld32_issue(trow + c0 + 64, va);
                maxima(c0 + 32, vb);
            }
        }
        // five distinct columns >= L0: the fifth largest of the eight group maxima
        float L0;
        {
            float a5[5] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                float v = gm[q];
#pragma unroll
                for (int j = 0; j < 5; ++j) { const float hi = fmaxf(a5[j], v); v = fminf(a5[j], v); a5[j] = hi; }
            }
            L0 = a5[4];
        }
        // L' = floor(L0 - eps) - 1, candidates: a_c >= L' - eps; every step rounded towards -inf
        const float thr = __fsub_rd(__fsub_rd(floorf(__fsub_rd(L0, ee)), 1.0f), ee);
        // no block barrier here: any thread that saw the mbarrier flip knows the GEMM is complete, so the X tile is dead for
        // everybody; lists and staging slab are thread-private
        int n = 0;
        float worst = 0.f;
        auto collect = [&](int c0, const float (&v)[32]) {
            unsigned h4[4] = {0u, 0u, 0u, 0u};            // branch-free: one compare and one predicated OR per column, four chains
#pragma unroll
            for (int i = 0; i < 32; ++i) h4[i & 3] |= v[i] >= thr ? (1u << i) : 0u;
            const unsigned hit_all = (h4[0] | h4[1]) | (h4[2] | h4[3]);
            if (__any_sync(0xffffffffu, hit_all != 0u)) {    // registers cannot be indexed by a run-time column: through shared memory
#pragma unroll
                for (int i = 0; i < 32; ++i) stage[i * TC_ROWS + tid] = v[i];
                unsigned hit = hit_all;
                while (hit) {
                    const int i = __ffs(hit) - 1;
                    hit &= hit - 1;
                    if (n < TC_CAP) {
                        Lv[n * TC_ROWS + tid] = stage[i * TC_ROWS + tid];
                        Lc[n * TC_ROWS + tid] = (unsigned char)(c0 + i);
                    }
                    ++n;
                }
            }
            if (CHECK && valid) {
                for (int i = 0; i < 32; ++i) {
                    const float *rp = rc + (size_t)(c0 + i) * RF;
                    float d = rp[0];
                    for (int j = 0; j < FL; ++j) {
                        const float df = __fsub_rn(x[j], rp[1 + 2 * j]);
                        d = __fsub_rn(d, __fmul_rn(__fmul_rn(df, df), rp[2 + 2 * j]));
                    }
                    worst = fmaxf(worst, __fdividef(fabsf(v[i] - d), ee));
                }
            }
        };
        {
            float va[32], vb[32];
            tmem_ld32_issue(trow, va);
#pragma unroll 1
            for (int c0 = 0; c0 < ND; c0 += 64) {
                tmem_wait_ld_dep(va);
                tmem_ld32_issue(trow + c0 + 32, vb);
                collect(c0, va);
                tmem_wait_ld_dep(vb);
                if (c0 + 64 < ND) tmem_ld32_issue(trow + c0 + 64, va);
                collect(c0 + 32, vb);
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        const bool listed = n >= 5 && n <= TC_CAP;
        auto cand_v = [&](int i) { return Lv[i * TC_ROWS + r]; };
        auto cand_c = [&](int i) { return (int)Lc[i * TC_ROWS + r]; };
        if (CHECK) {
            atomicMax(reinterpret_cast<int *>(check), __float_as_int(worst));
            if (valid) atomicMax(reinterpret_cast<int *>(check) + 1, n);
        }

        // ---- the record straight from the filter values when they leave no doubt ----
        if (valid) {
            bool certain = listed;
            if (certain) {
                float a[5] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY, -INFINITY};
                int c[5] = {0, 0, 0, 0, 0};
                for (int i = 0; i < n; ++i) {
                    float v = cand_v(i);
                    int cv = cand_c(i);
#pragma unroll
                    for (int j = 0; j < 5; ++j)
                        if (v > a[j]) { const float tv = a[j]; const int tc = c[j]; a[j] = v; c[j] = cv; v = tv; cv = tc; }
                }
                const float gap = __fadd_ru(__fadd_ru(ee, ee), 1.0f);
                int qv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    certain &= __fsub_rd(a[j], a[j + 1]) > gap;
                    const int lo = __float2int_ru(__fsub_rd(a[j], ee)), hi = __float2int_ru(__fadd_ru(a[j], ee));
                    certain &= (lo >> PSB_SENSCR_SHIFT) == (hi >> PSB_SENSCR_SHIFT);
                    qv[j] = lo >> PSB_SENSCR_SHIFT;
                }
                certain &= __fadd_ru(a[0], ee) < -2.0f && a[4] > -2.0e9f;
                if (certain) {
                    unsigned cb = 0, eb = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        int ev = qv[0] - qv[j];
                        ev = ev > 255 ? 255 : ev;
                        cb |= (unsigned)c[j] << (8 * j);
                        eb |= (unsigned)ev << (8 * j);
                    }
                    out[row * K + k] = make_int4(qv[0], (int)cb, (int)eb, 0);
                    if (CHECK) { atomicAdd(stats, 1ull); atomicAdd(stats + 1, 1ull); }
                }
            }
            // doubt: the row goes to ptm_tc_exact_kernel's work list (one atomic per warp); only when that list is full
            // is the exact arithmetic done here
            if (!certain && items) {
                const unsigned who = __activemask();
                const unsigned need = __ballot_sync(who, true);
                const int leader = __ffs(need) - 1;
                unsigned base = 0;
                if ((tid & 31) == leader) base = atomicAdd(n_items, (unsigned)__popc(need));
                base = __shfl_sync(need, base, leader);
                const unsigned slot = base + (unsigned)__popc(need & ((1u << (tid & 31)) - 1u));
                if (slot < item_cap) {
                    unsigned wv[5] = {0u, 0u, 0u, 0u, 0u};
                    if (listed)
                        for (int i = 0; i < n; ++i) wv[i >> 2] |= (unsigned)cand_c(i) << (8 * (i & 3));
                    items[2 * (size_t)slot] = make_uint4((unsigned)row, (unsigned)k | ((listed ? (unsigned)n : 255u) << 16), wv[0], wv[1]);
                    items[2 * (size_t)slot + 1] = make_uint4(wv[2], wv[3], wv[4], (unsigned)(row >> 32));
                    certain = true;                       // handled
                    if (CHECK) atomicAdd(stats, 1ull);
                }
            }
            if (!certain) {
                // the reference's exact arithmetic for this row's candidates (all codewords if the list overflowed)
                Top5 top;
                top.n = 0; top.c = 0u; top.c4 = 0;
#pragma unroll
                for (int j = 0; j < 5; ++j) top.s[j] = INT_MIN;
                int n_exact = 0;
                const int cnt_l = listed ? n : ND;
                for (int i = 0; i < cnt_l; ++i) {
                    const int cw = listed ? cand_c(i) : i;
                    const float d = gau_dist<FL>(reinterpret_cast<const float4 *>(rc + (size_t)cw * RF), x);
                    top5_insert(top, f2i_clamped(d), cw);
                    ++n_exact;
                }
                const bool distinct = top.n >= 5 && top.s[0] > top.s[1] && top.s[1] > top.s[2] && top.s[2] > top.s[3] && top.s[3] > top.s[4];
                const int tp = top.s[0] >> PSB_SENSCR_SHIFT;
                unsigned eb = 0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    int ev = tp - (top.s[j] >> PSB_SENSCR_SHIFT);
                    ev = ev > 255 ? 255 : ev;
                    eb |= (unsigned)ev << (8 * j);
                }
                out[row * K + k] = make_int4(tp, (int)top.c, (int)eb, 0);
                if (!distinct) atomicOr(&flags[(size_t)k * flag_words + (row >> 5)], 1u << (row & 31));
                if (CHECK) { atomicAdd(stats, 1ull); atomicAdd(stats + 2, (unsigned long long)n_exact); if (!distinct) atomicAdd(stats + 3, 1ull); }
            }
        }
        __syncthreads();                                  // lists consumed, accumulator read: the next tile may overwrite both
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(ND < 32 ? 32 : ND));
}

// Rows the filter values left in doubt (work list of ptm_tc5_kernel): one thread per row, the reference's exact
// arithmetic for its candidate codewords (all codewords when its list had overflowed), the five best, the record;
// exact ties go on to the fix-up.  Item: {row low, pair | n << 16, 18 codeword bytes, row high}.
template <int FL>
__global__ void __launch_bounds__(128)
ptm_tc_exact_kernel(const float *__restrict__ feats, int D, const int32_t *__restrict__ featoff, const uint4 *__restrict__ items,
                    const unsigned *__restrict__ n_items, unsigned item_cap, const float *__restrict__ rec,
                    const size_t *__restrict__ rec_off, int4 *__restrict__ out, unsigned *__restrict__ flags, long long flag_words,
                    int K, int n_feat, int nd, unsigned long long *__restrict__ stats)
{
    constexpr int RF = (1 + 2 * FL + 3) / 4 * 4;
    const unsigned count = min(*n_items, item_cap);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const uint4 a = items[2 * (size_t)i], b = items[2 * (size_t)i + 1];
        const long long row = (long long)a.x | ((long long)b.w << 32);
        const int k = (int)(a.y & 0xffffu), n = (int)(a.y >> 16);
        const unsigned wv[5] = {a.z, a.w, b.x, b.y, b.z};
        const float *px = feats + row * D + featoff[k % n_feat];
        const float *rc = rec + rec_off[k];
        float x[FL];
#pragma unroll
        for (int j = 0; j < FL; ++j) x[j] = px[j];
        Top5 top;
        top.n = 0; top.c = 0u; top.c4 = 0;
#pragma unroll
        for (int j = 0; j < 5; ++j) top.s[j] = INT_MIN;
        const int cnt = n == 255 ? nd : n;
        for (int q = 0; q < cnt; ++q) {
            const int cw = n == 255 ? q : (int)((wv[q >> 2] >> (8 * (q & 3))) & 0xffu);
            const float d = gau_dist<FL>(reinterpret_cast<const float4 *>(rc + (size_t)cw * RF), x);
            top5_insert(top, f2i_clamped(d), cw);
        }
        const bool distinct = top.n >= 5 && top.s[0] > top.s[1] && top.s[1] > top.s[2] && top.s[2] > top.s[3] && top.s[3] > top.s[4];
        const int tp = top.s[0] >> PSB_SENSCR_SHIFT;
        unsigned eb = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int ev = tp - (top.s[j] >> PSB_SENSCR_SHIFT);
            ev = ev > 255 ? 255 : ev;
            eb |= (unsigned)ev << (8 * j);
        }
        out[row * K + k] = make_int4(tp, (int)top.c, (int)eb, 0);
        if (!distinct) atomicOr(&flags[(size_t)k * flag_words + (row >> 5)], 1u << (row & 31));
        if (stats) { atomicAdd(stats + 2, (unsigned long long)cnt); if (!distinct) atomicAdd(stats + 3, 1ull); }
    }
}

// Frames whose five best scores tie: the reference's loop, literally (eval_topn ptm_mgau.c:88-136,
// eval_cb :152-226), seeded with the previous frame's list -- the record the filter kernel (or this
// warp, one frame earlier) wrote -- or with codewords 0..3 at the start of an utterance (:791-792).
// One WARP per (utterance, pair) chain: lanes = codewords (ND / 32 each), the flagged frames of the
// chain in order.  All distances of a frame in parallel, the four seeds fetched by shuffle, then the scan only visits --
// in ascending codeword order -- the codewords whose distance reaches the seeds' worst score (ballots), each re-tested
// against the list as it stands: eval_topn + eval_cb literally, like semi_scan_kernel does for semi-continuous models.
// A thread per chain serialises 260 distances per flagged frame inside one lane (15 ms per 10^6 frames at a 0.04 % tie
// rate); a warp costs a few hundred warp instructions per flagged frame.
template <int FL, int NDW>
__global__ void __launch_bounds__(128)
ptm_fixup_warp_kernel(const float *__restrict__ feats, int D, const int32_t *__restrict__ featoff, const int32_t *__restrict__ utt_off,
                      int n_utt, const float *__restrict__ rec, const size_t *__restrict__ rec_off, int4 *__restrict__ out,
                      const unsigned *__restrict__ flags, long long flag_words, int K, int n_feat)
{
    constexpr int RF = (1 + 2 * FL + 3) / 4 * 4;
    constexpr unsigned FULL = 0xffffffffu;
    const long long id = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (id >= (long long)n_utt * K) return;
    const int u = (int)(id / K), k = (int)(id % K);
    const int f = k % n_feat;
    const long long f0 = utt_off[u], f1 = utt_off[u + 1];
    if (f1 <= f0) return;
    const unsigned *fl = flags + (size_t)k * flag_words;
    const float *rc = rec + rec_off[k];
    for (long long w0 = f0 >> 5; w0 <= (f1 - 1) >> 5; w0 += 32) {
        const long long wd_l = w0 + lane;
        unsigned mine = wd_l <= ((f1 - 1) >> 5) ? fl[wd_l] : 0u;
        unsigned any = __ballot_sync(FULL, mine != 0u);
        while (any) {
            const int wl = __ffs(any) - 1;
            any &= any - 1;
            unsigned bits = __shfl_sync(FULL, mine, wl);
            while (bits) {
                const int b = __ffs(bits) - 1;
                bits &= bits - 1;
                const long long row = (w0 + wl) * 32 + b;
                if (row < f0 || row >= f1) continue;
                const float *px = feats + row * D + featoff[f];
                float x[FL];
#pragma unroll
                for (int j = 0; j < FL; ++j) x[j] = px[j];
                float d[NDW];
#pragma unroll
                for (int q = 0; q < NDW; ++q) d[q] = gau_dist<FL>(reinterpret_cast<const float4 *>(rc + (size_t)(lane + 32 * q) * RF), x);
                auto dist_of = [&](int c) {                            // uniform c: the owner lane's value
                    float v = d[0];
#pragma unroll
                    for (int q = 1; q < NDW; ++q) v = (c >> 5) == q ? d[q] : v;
                    return __shfl_sync(FULL, v, c & 31);
                };
                const unsigned seeds = row == f0 ? 0x03020100u : (unsigned)out[(row - 1) * K + k].y;
                int cw[4], sc[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {                          // eval_topn: stable, strict >
                    const int c = (seeds >> (8 * i)) & 0xff;
                    const int s = f2i_clamped(dist_of(c));
                    int p = 0;
#pragma unroll
                    for (int j = 0; j < i; ++j) p += (s > sc[j]) ? 0 : 1;
#pragma unroll
                    for (int j = 2; j >= 0; --j)
                        if (j < i && j >= p) { sc[j + 1] = sc[j]; cw[j + 1] = cw[j]; }
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (j == p) { sc[j] = s; cw[j] = c; }
                }
                const float th0 = (float)sc[3];                        // the scan's threshold only rises from here
#pragma unroll
                for (int q = 0; q < NDW; ++q) {
                    unsigned cand = __ballot_sync(FULL, d[q] >= th0);
                    while (cand) {
                        const int l = __ffs(cand) - 1;
                        cand &= cand - 1;
                        const int c = l + 32 * q;
                        const float dv = __shfl_sync(FULL, d[q], l);
                        if (!(dv >= (float)sc[3])) continue;            // eval_cb :207
                        if (cw[0] == c || cw[1] == c || cw[2] == c || cw[3] == c) continue;   // :209-215
                        const int s = f2i_clamped(dv);
                        int p = 0;
#pragma unroll
                        for (int j = 0; j < 3; ++j) p += (s >= sc[j]) ? 0 : 1;     // insertion_sort_cb :140-149
#pragma unroll
                        for (int j = 2; j >= 0; --j)
                            if (j >= p) { sc[j + 1] = sc[j]; cw[j + 1] = cw[j]; }
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (j == p) { sc[j] = s; cw[j] = c; }
                    }
                }
                if (lane == 0) {
                    const int tp = sc[0] >> PSB_SENSCR_SHIFT;
                    unsigned cb = 0, eb = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        int ev = tp - (sc[j] >> PSB_SENSCR_SHIFT);
                        ev = ev > 255 ? 255 : ev;
                        cb |= (unsigned)cw[j] << (8 * j);
                        eb |= (unsigned)ev << (8 * j);
                    }
                    out[row * K + k] = make_int4(tp, (int)cb, (int)eb, 0);
                }
                __syncwarp();
            }
        }
    }
}

float round_tf32_host(float x)
{
    // cvt.rna.tf32.f32: round to nearest, ties away from zero, 10 explicit mantissa bits
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7f800000u) == 0x7f800000u) return x;
    u = (u + 0x1000u) & ~0x1fffu;
    float r;
    memcpy(&r, &u, 4);
    return r;
}

template <int FL, int ND>
int launch_tc5(psb_batch_t *b, const float *d_feats, long long total, const int32_t *d_klist, int n_k, const int32_t *d_featoff,
               bool check)
{
    psb_model_t *m = b->m;
    const size_t smem = (size_t)2 * 8 * ND * 16 + (size_t)2 * 8 * TC_ROWS * 16;
    const long long tiles = (total + TC_ROWS - 1) / TC_ROWS;
    // W (64 KB at 256 densities) is staged once per CTA: a few tiles per CTA, but still >= 4 waves of 2 CTAs per SM
    int tpc = 1;
    while (tpc < 8 && (tiles / (tpc * 2)) * n_k >= 148LL * 2 * 4) tpc *= 2;
    PSB_REQUIRE((tiles + tpc - 1) / tpc <= 65535, "too many frames for one launch of the tensor-core filter");
    const dim3 grid((unsigned)n_k, (unsigned)((tiles + tpc - 1) / tpc));
    float *chk = b->d_tc_check;
    unsigned long long *stats = reinterpret_cast<unsigned long long *>(b->d_tc_check + 4);
    if (check) {
        auto kern = ptm_tc5_kernel<FL, ND, true>;
        PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, TC_ROWS, smem, b->stream>>>(d_feats, total, m->sumlen, d_featoff, d_klist, m->d_tc_wumma, m->d_tc_cen, m->d_tc_bnd,
                                                m->d_rec, m->d_rec_off, b->d_topn, b->d_tc_flags, (long long)b->tc_flag_words, m->K,
                                                m->n_feat, tpc, b->d_tc_items, b->d_tc_nitems, b->tc_item_cap, chk, stats);
    }
    else {
        auto kern = ptm_tc5_kernel<FL, ND, false>;
        PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, TC_ROWS, smem, b->stream>>>(d_feats, total, m->sumlen, d_featoff, d_klist, m->d_tc_wumma, m->d_tc_cen, m->d_tc_bnd,
                                                m->d_rec, m->d_rec_off, b->d_topn, b->d_tc_flags, (long long)b->tc_flag_words, m->K,
                                                m->n_feat, tpc, b->d_tc_items, b->d_tc_nitems, b->tc_item_cap, nullptr, nullptr);
    }
    PSB_LAUNCH_CHECK();
    if (b->d_tc_items) {
        // the rows in doubt: the count lives on the device, so the grid covers the list's capacity (grid-stride loop, idle
        // blocks leave at once)
        const unsigned blocks = (unsigned)std::min<size_t>(((size_t)b->tc_item_cap + 127) / 128, 148 * 64);
        ptm_tc_exact_kernel<FL><<<blocks, 128, 0, b->stream>>>(d_feats, m->sumlen, d_featoff, b->d_tc_items, b->d_tc_nitems, b->tc_item_cap,
                                                              m->d_rec, m->d_rec_off, b->d_topn, b->d_tc_flags, (long long)b->tc_flag_words,
                                                              m->K, m->n_feat, ND, check ? stats : nullptr);
        PSB_LAUNCH_CHECK();
    }
    return PSB_OK;
}

}  // namespace

// Host side: the GEMM operand W, the centre and the error-bound coefficients of every pair.
// hm / hv / hd: the model's means, variance terms and determinants on the host (build_records).
int psb_tc_prepare(psb_model_t *m, const float *hm, const float *hv, const float *hd)
{
    m->tc_ok = false;
    if (m->kind != PSB_KIND_PTM || m->fixed_point || m->topn != 4) return PSB_OK;
    if (m->n_density != 64 && m->n_density != 128 && m->n_density != 256) return PSB_OK;
    for (int f = 0; f < m->n_feat; ++f)
        if (m->featlen[f] != 13) return PSB_OK;              // the kernels are instantiated for 13-dimensional streams
    const int nd = m->n_density, FL = 13, K = m->K;
    std::vector<float> cen((size_t)K * 16, 0.f), bnd((size_t)K * 32, 0.f);
    std::vector<float> wu((size_t)K * 2 * 8 * nd * 4, 0.f);     // canonical K-major layout of the tcgen05 operand: [half][chunk][n][4]
    std::vector<double> W((size_t)TC_K * nd);
    for (int cb = 0; cb < m->n_mgau; ++cb)
        for (int f = 0; f < m->n_feat; ++f) {
            const int k = cb * m->n_feat + f;
            const size_t src = ((size_t)cb * m->sumlen + m->featoff[f]) * nd;
            const float *mu = hm + src, *vv = hv + src, *dt = hd + (size_t)k * nd;
            float *c = cen.data() + (size_t)k * 16, *bb = bnd.data() + (size_t)k * 32;
            for (int j = 0; j < FL; ++j) {
                double s = 0;
                for (int q = 0; q < nd; ++q) s += mu[(size_t)q * FL + j];
                c[j] = (float)(s / nd);
            }
            std::fill(W.begin(), W.end(), 0.0);
            double cmax = 0;
            for (int q = 0; q < nd; ++q) {
                double c0 = dt[q], quad = 0;
                for (int j = 0; j < FL; ++j) {
                    const double v = vv[(size_t)q * FL + j], mp = (double)mu[(size_t)q * FL + j] - (double)c[j];
                    W[(size_t)j * nd + q] = -v;
                    W[(size_t)(FL + j) * nd + q] = 2.0 * v * mp;
                    quad += std::fabs(v) * mp * mp;
                    c0 -= v * mp * mp;
                    bb[j] = std::max(bb[j], (float)std::fabs(v));
                    bb[FL + j] = std::max(bb[FL + j], (float)std::fabs(2.0 * v * mp));
                }
                W[(size_t)(2 * FL) * nd + q] = c0;
                cmax = std::max(cmax, std::fabs((double)dt[q]) + quad);
            }
            bb[2 * FL] = (float)(cmax * 1.0001);
            for (int j = 0; j < 2 * FL; ++j) bb[j] = std::nextafter(bb[j] * 1.0001f, INFINITY);
            // high and low TF32 halves of the fp32 value of every W entry: w = hi + lo + O(2^-22 w)
            float *u = wu.data() + (size_t)k * 2 * 8 * nd * 4;
            for (int kk = 0; kk < TC_K; ++kk)
                for (int q = 0; q < nd; ++q) {
                    const float v = (float)W[(size_t)kk * nd + q], h = round_tf32_host(v);
                    u[((size_t)(kk >> 2) * nd + q) * 4 + (kk & 3)] = h;
                    u[((size_t)(8 + (kk >> 2)) * nd + q) * 4 + (kk & 3)] = round_tf32_host(v - h);
                }
            for (int i = 0; i < 32; ++i)
                if (!std::isfinite(bb[i])) return PSB_OK;    // degenerate model: keep the scan kernels
        }
    if (!m->d_tc_wumma) {
        PSB_CUDA(cudaMalloc(&m->d_tc_wumma, wu.size() * sizeof(float)));
        PSB_CUDA(cudaMalloc(&m->d_tc_cen, cen.size() * sizeof(float)));
        PSB_CUDA(cudaMalloc(&m->d_tc_bnd, bnd.size() * sizeof(float)));
    }
    PSB_CUDA(cudaMemcpy(m->d_tc_wumma, wu.data(), wu.size() * sizeof(float), cudaMemcpyHostToDevice));
    PSB_CUDA(cudaMemcpy(m->d_tc_cen, cen.data(), cen.size() * sizeof(float), cudaMemcpyHostToDevice));
    PSB_CUDA(cudaMemcpy(m->d_tc_bnd, bnd.data(), bnd.size() * sizeof(float), cudaMemcpyHostToDevice));
    m->tc_ok = true;
    return PSB_OK;
}

bool psb_tc_usable(const psb_batch_t *b)
{
    const psb_model_t *m = b->m;
    return m->tc_ok && m->ds_ratio == 1 && !b->force_scan;
}

// Top-N records of a whole batch into b->d_topn (same format as the scan kernels write).
int psb_launch_ptm_tc(psb_batch_t *b, const float *d_feats, const int32_t *utt_off, int32_t n_utt, const int32_t *d_klist,
                      const int32_t *d_featoff)
{
    psb_model_t *m = b->m;
    const long long total = utt_off[n_utt];
    const size_t fw = (size_t)((total + 31) / 32) + 1;
    if (fw * m->K > b->tc_flag_cap) {
        cudaFree(b->d_tc_flags);
        b->d_tc_flags = nullptr;
        b->tc_flag_cap = fw * m->K + fw * m->K / 8;
        PSB_CUDA(cudaMalloc(&b->d_tc_flags, b->tc_flag_cap * 4));
    }
    if ((size_t)n_utt + 1 > b->uttoff_cap) {
        if (b->d_uttoff) cudaFree(b->d_uttoff);
        b->d_uttoff = nullptr;
        b->uttoff_cap = (size_t)n_utt + 1 + 64;
        PSB_CUDA(cudaMalloc(&b->d_uttoff, b->uttoff_cap * sizeof(int32_t)));
    }
    if (!b->d_tc_check) {                                     // float[2] check values, then (16-byte offset) four 64-bit counters
        PSB_CUDA(cudaMalloc(&b->d_tc_check, 64));
        PSB_CUDA(cudaMemsetAsync(b->d_tc_check, 0, 64, b->stream));
    }
    {
        // work list of the rows the filter leaves in doubt: room for a quarter of all (frame, pair) rows, 32 bytes each
        const size_t want = std::max<size_t>(4096, (size_t)total * m->K / 4);
        if (want > b->tc_item_cap || !b->d_tc_items) {
            cudaFree(b->d_tc_items);
            b->d_tc_items = nullptr;
            if (!b->d_tc_nitems) PSB_CUDA(cudaMalloc(&b->d_tc_nitems, 4));
            b->tc_item_cap = (unsigned)std::min<size_t>(want + want / 8, 0x7fffffffu);
            PSB_CUDA(cudaMalloc(&b->d_tc_items, (size_t)b->tc_item_cap * 32));
        }
        PSB_CUDA(cudaMemsetAsync(b->d_tc_nitems, 0, 4, b->stream));
    }
    b->tc_flag_words = fw;
    PSB_CUDA(cudaMemsetAsync(b->d_tc_flags, 0, fw * m->K * 4, b->stream));
    PSB_CUDA(cudaMemcpyAsync(b->d_uttoff, utt_off, ((size_t)n_utt + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream));
    static const bool check = [] { const char *v = getenv("PSB_TC_CHECK"); return v && atoi(v) != 0; }();
    int rc;
    switch (m->n_density) {
    case 256: rc = launch_tc5<13, 256>(b, d_feats, total, d_klist, m->K, d_featoff, check); break;
    case 128: rc = launch_tc5<13, 128>(b, d_feats, total, d_klist, m->K, d_featoff, check); break;
    default: rc = launch_tc5<13, 64>(b, d_feats, total, d_klist, m->K, d_featoff, check); break;
    }
    if (rc) return rc;
    const long long chains = (long long)n_utt * m->K;
    const unsigned blocks = (unsigned)((chains * 32 + 127) / 128);
#define PSB_FIXW(NDW) ptm_fixup_warp_kernel<13, NDW><<<blocks, 128, 0, b->stream>>>(d_feats, m->sumlen, d_featoff, b->d_uttoff, n_utt, \
        m->d_rec, m->d_rec_off, b->d_topn, b->d_tc_flags, (long long)fw, m->K, m->n_feat)
    if (m->n_density == 256) PSB_FIXW(8);
    else if (m->n_density == 128) PSB_FIXW(4);
    else PSB_FIXW(2);
#undef PSB_FIXW
    PSB_LAUNCH_CHECK();
    return PSB_OK;
}

// debug (PSB_TC_CHECK=1): max |a - d| / eps and max candidate count seen by the filter kernels of this batch;
// stats4 = rows, rows resolved from the filter values alone, exact distances computed, rows handed to the tie fix-up
extern "C" int psb_batch_tc_check(psb_batch_t *b, float *ratio, int32_t *max_candidates, int64_t *stats4)
{
    PSB_REQUIRE(b && ratio && max_candidates, "psb_batch_tc_check: null argument");
    *ratio = 0.f; *max_candidates = 0;
    if (stats4) stats4[0] = stats4[1] = stats4[2] = stats4[3] = 0;
    if (!b->d_tc_check) return PSB_OK;
    PSB_CUDA(cudaSetDevice(b->m->device));
    PSB_CUDA(cudaStreamSynchronize(b->stream));
    unsigned char h[64];
    PSB_CUDA(cudaMemcpy(h, b->d_tc_check, sizeof(h), cudaMemcpyDeviceToHost));
    memcpy(ratio, h, 4);
    memcpy(max_candidates, h + 4, 4);
    if (stats4) memcpy(stats4, h + 16, 32);
    return PSB_OK;
}
