// psb_ptm.cu -- batched PTM senone evaluation for sm_100a.
//
// Replaces, for whole batches of utterances with all senones computed (compallsen):
//   eval_topn / eval_cb / ptm_mgau_codebook_eval  (ptm_mgau.c:88-254)   -> ptm_topn_kernel
//   ptm_mgau_codebook_norm / ptm_mgau_senone_eval (ptm_mgau.c:266-403)  -> ptm_senone_kernel
//
// Work decomposition (DESIGN.md "Kernels"):
//  * The top-N list of a (codebook, stream) pair is a recurrence over time (frame t is seeded
//    by frame t-1's codewords), so time is the sequential axis and the parallel axes are
//    utterance x codebook x stream.  One *lane* owns one utterance; one CTA owns one
//    (codebook, stream) pair whose Gaussians sit in shared memory as warp-uniform records, so
//    every lane of a warp evaluates the same codeword against its own feature vector: the
//    model is read by LDS.128 broadcasts (one wavefront per 16 bytes for 32 lanes) and the
//    features come from a lane-major ("transposed") copy, one coalesced 128-byte load per
//    dimension per warp.
//  * The float accumulation is the reference's, rounding for rounding: x-mu, square,
//    times precomputed variance term, subtract -- four separately rounded operations per
//    dimension (__fsub_rn/__fmul_rn are never contracted into FMA), dimensions ascending.
//    The reference's early exit is result-neutral (d only decreases and the same float test
//    is repeated after the last dimension, SURVEY A.1.3), so distances are computed in full
//    and the insertion scan is replayed per lane in codeword order.
//  * Senone evaluation is embarrassingly parallel over (utterance, frame): one CTA per
//    frame, one thread per senone, mixture weights gathered from the L2-resident table.
#include "psb_gau.cuh"
#include "psb_internal.cuh"

#include <algorithm>
#include <numeric>

namespace {

constexpr int TOPN = 4;               // kernels below are specialised for -topn 4 (the default)
constexpr int TOPN_WARPS = 4;         // warps per CTA of the scan kernels
constexpr int MAX_NDW = 8;            // up to 256 codewords per codebook

// FIXED_POINT build of the reference (mfcc_t = int32 Q12, SURVEY A.1.11): the same records and the
// same feature rows carry int32 bit patterns.  FIXMUL (fe/fixpoint.h:98-100) is the 64-bit product
// shifted right by 12 and truncated to 32 bits; GMMSUB (tied_mgau_common.h:62-66) as gcc compiles it
// is (b < 0) ? INT_MIN : wrap32(a - b).  The scan's early exits are observable here (a wrapped
// subtraction can climb back over the threshold), so next to the final value the minimum of d at
// the reference's test points is returned: PTM tests before each of the leading FL % 4 dimensions,
// then before every group of four (ptm_mgau.c:182-206); the semi-continuous scan before every
// dimension (s2_semi_mgau.c:137-143); both once more after the last one.  A codeword survives the
// scan iff that minimum is >= the worst listed score.
__device__ __forceinline__ int fx_mul(int a, int b)
{
    return (int)(unsigned)(((long long)a * (long long)b) >> 12);
}
__device__ __forceinline__ int fx_gmmsub(int a, int b)
{
    return b < 0 ? INT_MIN : (int)((unsigned)a - (unsigned)b);
}
template <int FL, bool SEMI>
__device__ __forceinline__ int gau_dist_fx(const float4 *__restrict__ r, const float (&x)[FL], int *dmin)
{
    constexpr int RECF = (1 + 2 * FL + 3) / 4 * 4;
    int rr[RECF];
#pragma unroll
    for (int q = 0; q < RECF / 4; ++q) {
        float4 v = r[q];
        rr[4 * q + 0] = __float_as_int(v.x); rr[4 * q + 1] = __float_as_int(v.y);
        rr[4 * q + 2] = __float_as_int(v.z); rr[4 * q + 3] = __float_as_int(v.w);
    }
    int d = rr[0], mn = rr[0];
#pragma unroll
    for (int j = 0; j < FL; ++j) {
        if (SEMI || j < FL % 4 || (j - FL % 4) % 4 == 0) mn = min(mn, d);
        const int diff = (int)((unsigned)__float_as_int(x[j]) - (unsigned)rr[1 + 2 * j]);
        d = fx_gmmsub(d, fx_mul(fx_mul(diff, diff), rr[2 + 2 * j]));
    }
    *dmin = min(mn, d);
    return d;
}

// Lane/group tables built on the host per call (see psb_launch_ptm_batch):
//   lane_len[g*32+l]  frames of the utterance owned by lane l of group g (0 = padding lane)
//   lane_off[g*32+l]  flat frame offset of that utterance in feats / outputs
//   grp_base[g]       float offset of the group's block in featT; block is [maxT_g][D][32]
//   grp_maxT[g]
struct GroupTabs {
    const int32_t *lane_len, *lane_off, *grp_maxT;
    const long long *grp_base;
};

// feats [total][D] -> per group [t][D][32] (lane-major).  One warp per (group, t).
__global__ void __launch_bounds__(256)
transpose_feats_kernel(const float *__restrict__ feats, float *__restrict__ featT, GroupTabs tabs,
                       const long long *__restrict__ warp_base, int n_groups, int D)
{
    // warp_base[g] = first (group, t) work item of group g in a flat enumeration
    extern __shared__ float tile[];           // [warps][32][D+1]
    const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    long long item = (long long)blockIdx.x * warps + warp;
    // binary search the group of this item
    int lo = 0, hi = n_groups;                // warp_base has n_groups+1 entries
    if (item >= warp_base[n_groups]) return;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (warp_base[mid] <= item) lo = mid; else hi = mid;
    }
    const int g = lo;
    const int t = (int)(item - warp_base[g]);
    float *tl = tile + (size_t)warp * 32 * (D + 1);
    for (int l = 0; l < 32; ++l) {
        int len = tabs.lane_len[g * 32 + l];
        const float *row = feats + ((long long)tabs.lane_off[g * 32 + l] + t) * D;
        for (int d = lane; d < D; d += 32)
            tl[l * (D + 1) + d] = t < len ? row[d] : 0.f;
    }
    __syncwarp();
    float *dst = featT + tabs.grp_base[g] + (long long)t * D * 32;
    for (int d = 0; d < D; ++d)
        dst[d * 32 + lane] = tl[lane * (D + 1) + d];
}

// Top-N record written per (frame, codebook-stream pair), consumed by ptm_senone_kernel:
//   .x = best score >> 10           (ptm_mgau.c:277)
//   .y = codewords, byte j = cw_j
//   .z = byte j = min(255, (best >> 10) - (score_j >> 10))
//   .w = 0
// From these, ptm_mgau_codebook_norm's value min(96, norm - (score_j >> 10)) is
// min(96, (norm - .x) + .z byte j) exactly (norm >= .x, so saturating byte j at 255 is safe).

// SEMI = false: PTM (ptm_mgau.c); SEMI = true: semi-continuous (s2_semi_mgau.c:70-203), whose
// scan accepts a codeword iff the partial sum before the last dimension is >= (float)worst AND
// the truncated final score is >= worst (int), and whose record is already normalised per stream
// (mgau_norm :186-203): .x = number of entries inside topn_beam, .y = codeword bytes,
// .z = bytes min(96, -((score_j >> 10) - (score_0 >> 10))).
template <int FL, bool SEMI, bool FX = false>
__global__ void __launch_bounds__(TOPN_WARPS * 32, 7)
ptm_topn_kernel(const float *__restrict__ rec, const size_t *__restrict__ rec_off,
                const int32_t *__restrict__ klist, const float *__restrict__ featT, GroupTabs tabs,
                int4 *__restrict__ out, int n_groups, int nd, int n_feat, int D,
                const int32_t *__restrict__ featoff, int K, int ds_ratio, const int32_t *__restrict__ topn_beam)
{
    constexpr int RECF = (1 + 2 * FL + 3) / 4 * 4;
    constexpr int RECQ = RECF / 4;
    extern __shared__ float4 srec[];          // [nd][RECQ] records
    const int k = klist[blockIdx.x];
    const int f = k % n_feat;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    {   // stage this pair's Gaussian records (L2 -> SMEM), 16 bytes per thread per step
        const float4 *src = reinterpret_cast<const float4 *>(rec + rec_off[k]);
        for (int i = threadIdx.x; i < nd * RECQ; i += blockDim.x)
            srec[i] = src[i];
    }
    __syncthreads();

    const int g = blockIdx.y * (blockDim.x >> 5) + warp;
    if (g >= n_groups) return;
    const int len = tabs.lane_len[g * 32 + lane];
    const long long off = tabs.lane_off[g * 32 + lane];
    const int maxT = tabs.grp_maxT[g];
    const float *xT = featT + tabs.grp_base[g] + (long long)featoff[f] * 32 + lane;

    int cw[TOPN], sc[TOPN];
#pragma unroll
    for (int i = 0; i < TOPN; ++i) { cw[i] = i; sc[i] = INT_MIN; }   // ptm_mgau.c:791-792

    float xn[FL];
#pragma unroll
    for (int j = 0; j < FL; ++j) xn[j] = maxT > 0 ? xT[j * 32] : 0.f;

    for (int t = 0; t < maxT; ++t) {
        float x[FL];
#pragma unroll
        for (int j = 0; j < FL; ++j) x[j] = xn[j];
        if (t + 1 < maxT) {
            const float *nx = xT + (long long)(t + 1) * D * 32;
#pragma unroll
            for (int j = 0; j < FL; ++j) xn[j] = nx[j * 32];
        }
        if (t >= len) continue;

        // ---- eval_topn (ptm_mgau.c:88-136): re-score last frame's codewords, stable sort ----
        // The scan must skip the codewords already listed (ptm_mgau.c:212-218).  Only *seeds* can
        // be met by the scan (inserted codewords lie behind it), so two registers suffice:
        // seedpack = the four seed codewords (one byte each), seedbit = byte i is 1 << (cw_i & 7)
        // while seed i is still listed, 0 once it has been evicted.
        unsigned seedpack = 0u, seedbit = 0u;
        {
            int ncw[TOPN], nsc[TOPN];
#pragma unroll
            for (int i = 0; i < TOPN; ++i) {
                const int c = cw[i];
                int s, smin;
                if (FX) s = gau_dist_fx<FL, SEMI>(srec + c * RECQ, x, &smin);       // no early exit in eval_topn
                else s = f2i_clamped(gau_dist<FL>(srec + c * RECQ, x));
                seedpack |= (unsigned)c << (8 * i);
                seedbit |= (1u << (c & 7)) << (8 * i);
                // insert (c, s) into the sorted prefix nsc[0..i-1]: entries with score < s move down
                int p = 0;
#pragma unroll
                for (int j = 0; j < i; ++j) p += (s > nsc[j]) ? 0 : 1;
#pragma unroll
                for (int j = TOPN - 2; j >= 0; --j)
                    if (j < i && j >= p) { nsc[j + 1] = nsc[j]; ncw[j + 1] = ncw[j]; }
#pragma unroll
                for (int j = 0; j < TOPN; ++j)
                    if (j == p) { nsc[j] = s; ncw[j] = c; }
            }
#pragma unroll
            for (int i = 0; i < TOPN; ++i) { cw[i] = ncw[i]; sc[i] = nsc[i]; }
        }

        // ---- eval_cb (ptm_mgau.c:152-226) unless this frame is skipped by -ds (:242) ----
        if (t % ds_ratio == 0) {
            float thresh = (float)sc[TOPN - 1];
            const unsigned seedchunk = (seedpack >> 3) & 0x1f1f1f1fu;   // chunk (8 codewords) of each seed
            for (int ch = 0; ch < nd / 8; ++ch) {
                const float4 *rq = srec + (size_t)ch * 8 * RECQ;
                // m8 = bits of this chunk's codewords that are listed seeds
                unsigned m8;
                {
                    const unsigned t = seedchunk ^ ((unsigned)ch * 0x01010101u);      // zero byte = match
                    const unsigned nz = (((t & 0x7f7f7f7fu) + 0x7f7f7f7fu) | t) & 0x80808080u;
                    const unsigned hit = ((nz ^ 0x80808080u) >> 7) * 0xffu;           // 0xff per matching byte
                    const unsigned b = seedbit & hit;
                    m8 = (b | (b >> 8) | (b >> 16) | (b >> 24)) & 0xffu;
                }
#pragma unroll
                for (int cc = 0; cc < 8; ++cc) {
                    float dpen, d;
                    int di, dmin;
                    bool hit;
                    if (FX) {
                        di = gau_dist_fx<FL, SEMI>(rq + cc * RECQ, x, &dmin);
                        hit = dmin >= sc[TOPN - 1];
                    }
                    else {
                        d = gau_dist<FL, SEMI>(rq + cc * RECQ, x, &dpen);
                        di = f2i_clamped(d);
                        if (SEMI) hit = dpen >= thresh && di >= sc[TOPN - 1];
                        else hit = d >= thresh;
                    }
                    if (hit && !(m8 & (1u << cc))) {
                        const int c = ch * 8 + cc;
                        const int s = di;
                        const int ev = cw[TOPN - 1];
                        // insertion_sort_cb (:140-149): entries with score <= s shift down
                        int p = 0;
#pragma unroll
                        for (int j = 0; j < TOPN - 1; ++j) p += (s >= sc[j]) ? 0 : 1;
#pragma unroll
                        for (int j = TOPN - 2; j >= 0; --j)
                            if (j >= p) { sc[j + 1] = sc[j]; cw[j + 1] = cw[j]; }
#pragma unroll
                        for (int j = 0; j < TOPN; ++j)
                            if (j == p) { sc[j] = s; cw[j] = c; }
                        // An evicted seed becomes scannable again (it may lie ahead of the scan).
                        {
                            const unsigned t2 = seedpack ^ ((unsigned)ev * 0x01010101u);
                            const unsigned nz2 = (((t2 & 0x7f7f7f7fu) + 0x7f7f7f7fu) | t2) & 0x80808080u;
                            const unsigned keep = (nz2 >> 7) * 0xffu;                   // 0 for the byte == ev
                            seedbit &= keep;
                            if ((ev >> 3) == ch) m8 &= ~(1u << (ev & 7));
                        }
                        thresh = (float)sc[TOPN - 1];
                    }
                }
            }
        }

        // ---- emit the record ----
        const int top = sc[0] >> PSB_SENSCR_SHIFT;
        unsigned cwb = 0, eb = 0;
        int n_in_beam = TOPN;
#pragma unroll
        for (int j = 0; j < TOPN; ++j) {
            int e = top - (sc[j] >> PSB_SENSCR_SHIFT);
            if (SEMI) {
                e = e > PSB_MAX_NEG_ASCR ? PSB_MAX_NEG_ASCR : e;          // mgau_norm :196-198
                const int beam = topn_beam[f];
                if (beam && e > beam && n_in_beam == TOPN) n_in_beam = j;   // :199-200
            }
            else
                e = e > 255 ? 255 : e;
            cwb |= (unsigned)cw[j] << (8 * j);
            eb |= (unsigned)e << (8 * j);
        }
        out[(off + t) * K + k] = make_int4(SEMI ? n_in_beam : top, (int)cwb, (int)eb, 0);
    }
}

// The scan of ptm_topn_kernel<FL, true> with two codewords per packed distance (pair records, FADD2 / FMUL2): the
// semi-continuous models the split path below does not take.
template <int FL>
__global__ void __launch_bounds__(TOPN_WARPS * 32, 7)
ptm_topn2_kernel(const float *__restrict__ rec2, const size_t *__restrict__ rec2_off,
                 const int32_t *__restrict__ klist, const float *__restrict__ featT, GroupTabs tabs,
                 int4 *__restrict__ out, int n_groups, int nd, int n_feat, int D,
                 const int32_t *__restrict__ featoff, int K, int ds_ratio, const int32_t *__restrict__ topn_beam)
{
    constexpr int RECF2 = (2 + 4 * FL + 3) / 4 * 4;
    constexpr int RECQ2 = RECF2 / 4;
    extern __shared__ float4 srec[];          // [nd/2][RECQ2] pair records
    const int k = klist[blockIdx.x];
    const int f = k % n_feat;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {
        const float4 *src = reinterpret_cast<const float4 *>(rec2 + rec2_off[k]);
        for (int i = threadIdx.x; i < (nd >> 1) * RECQ2; i += blockDim.x)
            srec[i] = src[i];
    }
    __syncthreads();
    const int g = blockIdx.y * TOPN_WARPS + warp;
    if (g >= n_groups) return;
    const int len = tabs.lane_len[g * 32 + lane];
    const long long off = tabs.lane_off[g * 32 + lane];
    const int maxT = tabs.grp_maxT[g];
    const float *xT = featT + tabs.grp_base[g] + (long long)featoff[f] * 32 + lane;

    int cw[TOPN], sc[TOPN];
#pragma unroll
    for (int i = 0; i < TOPN; ++i) { cw[i] = i; sc[i] = INT_MIN; }
    float xn[FL];
#pragma unroll
    for (int j = 0; j < FL; ++j) xn[j] = maxT > 0 ? xT[j * 32] : 0.f;

    for (int t = 0; t < maxT; ++t) {
        float2 xx[FL];
#pragma unroll
        for (int j = 0; j < FL; ++j) xx[j] = make_float2(xn[j], xn[j]);
        if (t + 1 < maxT) {
            const float *nx = xT + (long long)(t + 1) * D * 32;
#pragma unroll
            for (int j = 0; j < FL; ++j) xn[j] = nx[j * 32];
        }
        if (t >= len) continue;

        // ---- eval_topn: re-score the listed codewords (each through its pair record) ----
        unsigned seedpack = 0u, seedbit = 0u;
        {
            int ncw[TOPN], nsc[TOPN];
#pragma unroll
            for (int i = 0; i < TOPN; ++i) {
                const int c = cw[i];
                const float2 d2 = gau_dist2<FL>(srec + (c >> 1) * RECQ2, xx);
                const int s = f2i_clamped((c & 1) ? d2.y : d2.x);
                seedpack |= (unsigned)c << (8 * i);
                seedbit |= (1u << (c & 7)) << (8 * i);
                int p = 0;
#pragma unroll
                for (int j = 0; j < i; ++j) p += (s > nsc[j]) ? 0 : 1;
#pragma unroll
                for (int j = TOPN - 2; j >= 0; --j)
                    if (j < i && j >= p) { nsc[j + 1] = nsc[j]; ncw[j + 1] = ncw[j]; }
#pragma unroll
                for (int j = 0; j < TOPN; ++j)
                    if (j == p) { nsc[j] = s; ncw[j] = c; }
            }
#pragma unroll
            for (int i = 0; i < TOPN; ++i) { cw[i] = ncw[i]; sc[i] = nsc[i]; }
        }

        // ---- eval_cb: scan in codeword order, two codewords per packed distance ----
        if (t % ds_ratio == 0) {
            float thresh = (float)sc[TOPN - 1];
            const unsigned seedchunk = (seedpack >> 3) & 0x1f1f1f1fu;
            for (int ch = 0; ch < nd / 8; ++ch) {
                const float4 *rq = srec + (size_t)ch * 4 * RECQ2;
                unsigned m8;
                {
                    const unsigned tt = seedchunk ^ ((unsigned)ch * 0x01010101u);
                    const unsigned nz = (((tt & 0x7f7f7f7fu) + 0x7f7f7f7fu) | tt) & 0x80808080u;
                    const unsigned hitb = ((nz ^ 0x80808080u) >> 7) * 0xffu;
                    const unsigned b = seedbit & hitb;
                    m8 = (b | (b >> 8) | (b >> 16) | (b >> 24)) & 0xffu;
                }
#pragma unroll
                for (int pp = 0; pp < 4; ++pp) {
                    float2 dpen2;
                    const float2 d2 = gau_dist2<FL, true>(rq + pp * RECQ2, xx, &dpen2);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int cc = 2 * pp + h;
                        const float d = h ? d2.y : d2.x;
                        const bool hit = (h ? dpen2.y : dpen2.x) >= thresh && f2i_clamped(d) >= sc[TOPN - 1];
                        if (hit && !(m8 & (1u << cc))) {
                            const int c = ch * 8 + cc;
                            const int s = f2i_clamped(d);
                            const int ev = cw[TOPN - 1];
                            int p = 0;
#pragma unroll
                            for (int j = 0; j < TOPN - 1; ++j) p += (s >= sc[j]) ? 0 : 1;
#pragma unroll
                            for (int j = TOPN - 2; j >= 0; --j)
                                if (j >= p) { sc[j + 1] = sc[j]; cw[j + 1] = cw[j]; }
#pragma unroll
                            for (int j = 0; j < TOPN; ++j)
                                if (j == p) { sc[j] = s; cw[j] = c; }
                            {
                                const unsigned t2 = seedpack ^ ((unsigned)ev * 0x01010101u);
                                const unsigned nz2 = (((t2 & 0x7f7f7f7fu) + 0x7f7f7f7fu) | t2) & 0x80808080u;
                                seedbit &= (nz2 >> 7) * 0xffu;
                                if ((ev >> 3) == ch) m8 &= ~(1u << (ev & 7));
                            }
                            thresh = (float)sc[TOPN - 1];
                        }
                    }
                }
            }
        }

        // ---- emit the record (same format as ptm_topn_kernel<FL, true>) ----
        const int top = sc[0] >> PSB_SENSCR_SHIFT;
        unsigned cwb = 0, eb = 0;
        int n_in_beam = TOPN;
#pragma unroll
        for (int j = 0; j < TOPN; ++j) {
            int e = top - (sc[j] >> PSB_SENSCR_SHIFT);
            e = e > PSB_MAX_NEG_ASCR ? PSB_MAX_NEG_ASCR : e;
            const int beam = topn_beam[f];
            if (beam && e > beam && n_in_beam == TOPN) n_in_beam = j;
            cwb |= (unsigned)cw[j] << (8 * j);
            eb |= (unsigned)e << (8 * j);
        }
        out[(off + t) * K + k] = make_int4(n_in_beam, (int)cwb, (int)eb, 0);
    }
}

// ---------------------------------------------------------------------------------------
// Deferred-insertion kernel ("Q").  ncu on ptm_topn2_kernel: 39 % of the executed instructions
// are NOT distance arithmetic -- the insertion path runs for a warp whenever ANY of its 32
// utterances accepts the current codeword (~80 of 256 codewords per frame), each time with one
// or two lanes live -- and the warp-uniform LDS.128 record stream sits at 64 % of the
// shared-memory data pipe (a broadcast delivers 8 bytes per wavefront).  The pair record {A,B}
// is used as is with duplicated feature registers (x,x), so there is no repacking, and:
//  * The scan only FILTERS: a codeword whose distance passes `d >= thresh` against a stale
//    (= lower or equal, the worst score only rises during a scan) threshold is pushed on a small
//    per-utterance queue in shared memory (distance) and a register (codeword byte).  All lanes
//    drain their queues together -- when any queue is nearly full and at the end of the frame --
//    replaying eval_cb's tests literally and in codeword order against the then-current list:
//    `d < thresh -> continue`, `already listed -> continue`, insertion_sort_cb
//    (ptm_mgau.c:207-222).  The queued set is a superset of the codewords the reference inserts
//    and every skipped codeword fails the reference's own test at its own scan position, so the
//    list after the drain equals the reference's.
constexpr int QCAP = 4;               // queue slots per utterance (codeword bytes fit one register)

struct QState {
    unsigned cwp;           // listed codewords, byte j = cw_j
    int sc[TOPN];
    float thresh;           // (float)sc[TOPN-1] as of the last drain; +inf for a finished utterance
    unsigned qc;            // queued codewords, newest in byte 0
    unsigned qw;            // shared-window byte address of the next free queue slot (this lane's
                            // column; slots are NT floats apart)
};

__device__ __forceinline__ void sts_f32(unsigned addr, float v)
{
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float lds_f32(unsigned addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}

__device__ __forceinline__ void q_insert(QState &st, int c, int s)
{
    int p = 0;
#pragma unroll
    for (int j = 0; j < TOPN - 1; ++j) p += (s >= st.sc[j]) ? 0 : 1;       // insertion_sort_cb (ptm_mgau.c:140-149)
#pragma unroll
    for (int j = TOPN - 2; j >= 0; --j)
        if (j >= p) st.sc[j + 1] = st.sc[j];
#pragma unroll
    for (int j = 0; j < TOPN; ++j)
        if (j == p) st.sc[j] = s;
    const unsigned lowmask = (1u << (8 * p)) - 1u;                          // p <= 3
    st.cwp = (st.cwp & lowmask) | ((unsigned)c << (8 * p)) | ((st.cwp << 8) & ~((lowmask << 8) | 0xffu));
}

// q: this lane's slot 0 of the utterance's queue, slots are `stride` floats apart
template <int stride>
__device__ __forceinline__ void q_drain(QState &st, unsigned q, bool active)
{
    const int qn = (int)(st.qw - q) / (stride * 4);
#pragma unroll
    for (int i = 0; i < QCAP; ++i) {
        if (i < qn) {
            const float d = lds_f32(q + i * stride * 4);
            if (d >= (float)st.sc[TOPN - 1]) {                              // ptm_mgau.c:207
                const unsigned c = (st.qc >> (8 * (qn - 1 - i))) & 0xffu;
                const unsigned x = st.cwp ^ (c * 0x01010101u);              // zero byte <=> already listed (:209-215)
                if (!((x - 0x01010101u) & ~x & 0x80808080u))
                    q_insert(st, (int)c, f2i_clamped(d));
            }
        }
    }
    st.qw = q;
    if (active) st.thresh = (float)st.sc[TOPN - 1];
}

template <int FL>
__global__ void __launch_bounds__(TOPN_WARPS * 32, 7)
ptm_topnq_kernel(const float *__restrict__ rec2, const size_t *__restrict__ rec2_off,
                 const int32_t *__restrict__ klist, const float *__restrict__ featT, GroupTabs tabs,
                 int4 *__restrict__ out, int n_groups, int nd, int n_feat, int D,
                 const int32_t *__restrict__ featoff, int K, int ds_ratio)
{
    constexpr int RECF2 = (2 + 4 * FL + 3) / 4 * 4;
    constexpr int RECQ2 = RECF2 / 4;
    constexpr int NT = TOPN_WARPS * 32;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ float4 srec[];          // [nd/2][RECQ2] pair records, then float q[QCAP][NT]
    const unsigned qbase = (unsigned)__cvta_generic_to_shared(
        reinterpret_cast<float *>(srec + (size_t)(nd >> 1) * RECQ2) + threadIdx.x);
    const int k = klist[blockIdx.x];
    const int f = k % n_feat;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {
        const float4 *src = reinterpret_cast<const float4 *>(rec2 + rec2_off[k]);
        for (int i = threadIdx.x; i < (nd >> 1) * RECQ2; i += blockDim.x)
            srec[i] = src[i];
    }
    __syncthreads();
    const int g = blockIdx.y * TOPN_WARPS + warp;
    if (g >= n_groups) return;
    const int len = tabs.lane_len[g * 32 + lane];
    const long long off = tabs.lane_off[g * 32 + lane];
    const int maxT = max(0, tabs.grp_maxT[g]);
    const float *xT = featT + tabs.grp_base[g] + (long long)featoff[f] * 32 + lane;

    QState st;
    st.cwp = 0x03020100u;                                          // codewords 0..3 (ptm_mgau.c:791-792)
#pragma unroll
    for (int i = 0; i < TOPN; ++i) st.sc[i] = INT_MIN;
    st.thresh = 0.f;
    st.qc = 0u;
    st.qw = qbase;

    for (int t = 0; t < maxT; ++t) {
        float2 xx[FL];
        {
            const float *p = xT + (long long)t * D * 32;
#pragma unroll
            for (int j = 0; j < FL; ++j) {
                const float v = p[j * 32];
                xx[j] = make_float2(v, v);
            }
        }
        const bool act = t < len;
        if (!__any_sync(FULL, act)) continue;                       // warp-uniform: the votes below need all lanes

        // ---- eval_topn: re-score the listed codewords (ptm_mgau.c:88-135) ----
        {
            int ncw[TOPN], nsc[TOPN];
#pragma unroll
            for (int i = 0; i < TOPN; ++i) {
                const int c = (st.cwp >> (8 * i)) & 0xff;
                const float2 d2 = gau_dist2<FL>(srec + (c >> 1) * RECQ2, xx);
                const int s = f2i_clamped((c & 1) ? d2.y : d2.x);
                int p = 0;
#pragma unroll
                for (int j = 0; j < i; ++j) p += (s > nsc[j]) ? 0 : 1;
#pragma unroll
                for (int j = TOPN - 2; j >= 0; --j)
                    if (j < i && j >= p) { nsc[j + 1] = nsc[j]; ncw[j + 1] = ncw[j]; }
#pragma unroll
                for (int j = 0; j < TOPN; ++j)
                    if (j == p) { nsc[j] = s; ncw[j] = c; }
            }
            unsigned cp = 0u;
#pragma unroll
            for (int i = 0; i < TOPN; ++i) { st.sc[i] = nsc[i]; cp |= (unsigned)ncw[i] << (8 * i); }
            st.cwp = cp;
            st.thresh = act ? (float)nsc[TOPN - 1] : __int_as_float(0x7f800000);
        }

        // ---- eval_cb: filter in codeword order ----
        if (t % ds_ratio == 0) {
#pragma unroll 2
            for (int pp = 0; pp < (nd >> 1); ++pp) {
                const float4 *r = srec + (size_t)pp * RECQ2;
                float2 rr[RECF2 / 2];
#pragma unroll
                for (int q = 0; q < RECQ2; ++q) {
                    const float4 v = r[q];
                    rr[2 * q] = make_float2(v.x, v.y);
                    rr[2 * q + 1] = make_float2(v.z, v.w);
                }
                float2 d = rr[0];
#pragma unroll
                for (int j = 0; j < FL; ++j) {
                    float2 tt = __fadd2_rn(xx[j], rr[1 + 2 * j]);
                    tt = __fmul2_rn(tt, tt);
                    tt = __fmul2_rn(tt, rr[2 + 2 * j]);
                    d.x = __fadd_rn(d.x, tt.x);                        // scalar on purpose: see gau_dist2
                    d.y = __fadd_rn(d.y, tt.y);
                }
                if (d.x >= st.thresh) {
                    sts_f32(st.qw, d.x);
                    st.qc = __byte_perm(st.qc, (unsigned)(2 * pp), 0x2104);
                    st.qw += NT * 4;
                }
                if (d.y >= st.thresh) {
                    sts_f32(st.qw, d.y);
                    st.qc = __byte_perm(st.qc, (unsigned)(2 * pp + 1), 0x2104);
                    st.qw += NT * 4;
                }
                if (__any_sync(FULL, st.qw > qbase + (QCAP - 2) * NT * 4))
                    q_drain<NT>(st, qbase, act);
            }
            if (__any_sync(FULL, st.qw != qbase))
                q_drain<NT>(st, qbase, act);
        }

        // ---- emit the record (same format as ptm_topn_kernel) ----
        if (!act) continue;
        const int top = st.sc[0] >> PSB_SENSCR_SHIFT;
        unsigned eb = 0;
#pragma unroll
        for (int j = 0; j < TOPN; ++j) {
            int e = top - (st.sc[j] >> PSB_SENSCR_SHIFT);
            e = e > 255 ? 255 : e;
            eb |= (unsigned)e << (8 * j);
        }
        out[(off + t) * K + k] = make_int4(top, (int)st.cwp, (int)eb, 0);
    }
}

// ---------------------------------------------------------------------------------------
// Semi-continuous models have ONE codebook per stream (K = n_feat pairs, 4 for s2_4x), so the
// lane-per-utterance kernels above leave most of the machine idle (512 utterances = 16 CTAs).
// Their distance work is small (4 x 256 Gaussians per frame), so it is taken out of the
// time recurrence: semi_dist_kernel computes every (frame, codeword) distance in parallel and
// parks {d, partial-before-last-dim} in HBM (8 B x n_density x K per frame), and
// semi_scan_kernel -- one WARP per (utterance, stream), lanes = codewords -- replays
// eval_topn / the scan of mgau_dist (s2_semi_mgau.c:70-183) per frame with the list held
// redundantly (uniformly) in every lane: ballots pick the codewords that pass the current
// threshold, they are handled in ascending order with the exact accept / skip-if-listed /
// insert rules, re-tested against the list as it stands.  No staleness, no queues, no
// divergence; 4 x n_utt warps instead of 4 x n_utt / 32.
template <int FL>
__global__ void __launch_bounds__(256)
semi_dist_kernel(const float *__restrict__ rec, const size_t *__restrict__ rec_off, const int32_t *__restrict__ klist,
                 const float *__restrict__ feats, float2 *__restrict__ dist, long long total, int nd, int n_feat, int D,
                 const int32_t *__restrict__ featoff)
{
    constexpr int RECF = (1 + 2 * FL + 3) / 4 * 4;
    const int k = klist[blockIdx.y];
    const long long fr = blockIdx.x;
    const int c = threadIdx.x;
    if (c >= nd) return;
    float x[FL];
    const float *xp = feats + fr * D + featoff[k % n_feat];
#pragma unroll
    for (int j = 0; j < FL; ++j) x[j] = xp[j];
    float dpen;
    const float d = gau_dist<FL, true>(reinterpret_cast<const float4 *>(rec + rec_off[k] + (size_t)c * RECF), x, &dpen);
    dist[((size_t)k * total + fr) * nd + c] = make_float2(d, dpen);
}

struct ScanList {
    unsigned cwp;
    int sc[TOPN];
};

__device__ __forceinline__ void scan_insert(ScanList &L, int c, int s)
{
    int p = 0;
#pragma unroll
    for (int j = 0; j < TOPN - 1; ++j) p += (s >= L.sc[j]) ? 0 : 1;        // insertion sort, s2_semi_mgau.c:157-167
#pragma unroll
    for (int j = TOPN - 2; j >= 0; --j)
        if (j >= p) L.sc[j + 1] = L.sc[j];
#pragma unroll
    for (int j = 0; j < TOPN; ++j)
        if (j == p) L.sc[j] = s;
    const unsigned lowmask = (1u << (8 * p)) - 1u;
    L.cwp = (L.cwp & lowmask) | ((unsigned)c << (8 * p)) | ((L.cwp << 8) & ~((lowmask << 8) | 0xffu));
}

// NDW = n_density / 32 codewords per lane
template <int NDW>
__global__ void __launch_bounds__(128)
semi_scan_kernel(const float2 *__restrict__ dist, const int32_t *__restrict__ utt_off, int n_utt, int K, long long total,
                 int nd, int ds_ratio, const int32_t *__restrict__ topn_beam, int4 *__restrict__ out)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= n_utt * K) return;
    const int u = w / K, k = w % K;
    const long long f0 = utt_off[u];
    const int T = utt_off[u + 1] - utt_off[u];
    const float2 *row = dist + ((size_t)k * total + f0) * nd;
    ScanList L;
    L.cwp = 0x03020100u;                                           // s2_semi_mgau.c:1319-1327
#pragma unroll
    for (int i = 0; i < TOPN; ++i) L.sc[i] = INT_MIN;
    for (int t = 0; t < T; ++t, row += nd) {
        float2 v[NDW];
#pragma unroll
        for (int i = 0; i < NDW; ++i) v[i] = row[i * 32 + lane];
        // eval_topn (:70-109): re-score the listed codewords, stable descending sort (strict >)
        {
            int ncw[TOPN], nsc[TOPN];
#pragma unroll
            for (int i = 0; i < TOPN; ++i) {
                const int c = (L.cwp >> (8 * i)) & 0xff;
                float dv = 0.f;
#pragma unroll
                for (int q = 0; q < NDW; ++q) {
                    const float cand = __shfl_sync(0xffffffffu, v[q].x, c & 31);
                    if ((c >> 5) == q) dv = cand;
                }
                const int s = f2i_clamped(dv);
                int p = 0;
#pragma unroll
                for (int j = 0; j < i; ++j) p += (s > nsc[j]) ? 0 : 1;
#pragma unroll
                for (int j = TOPN - 2; j >= 0; --j)
                    if (j < i && j >= p) { nsc[j + 1] = nsc[j]; ncw[j + 1] = ncw[j]; }
#pragma unroll
                for (int j = 0; j < TOPN; ++j)
                    if (j == p) { nsc[j] = s; ncw[j] = c; }
            }
            unsigned cp = 0u;
#pragma unroll
            for (int i = 0; i < TOPN; ++i) { L.sc[i] = nsc[i]; cp |= (unsigned)ncw[i] << (8 * i); }
            L.cwp = cp;
        }
        if (t % ds_ratio == 0) {
#pragma unroll
            for (int q = 0; q < NDW; ++q) {
                // accept iff the partial sum before the last dimension is >= (float)worst AND the
                // truncated final score is >= worst (:137-155)
                unsigned m = __ballot_sync(0xffffffffu, v[q].y >= (float)L.sc[TOPN - 1] && f2i_clamped(v[q].x) >= L.sc[TOPN - 1]);
                while (m) {
                    const int b = __ffs(m) - 1;
                    m &= m - 1;
                    const float dv = __shfl_sync(0xffffffffu, v[q].x, b), pv = __shfl_sync(0xffffffffu, v[q].y, b);
                    const int c = q * 32 + b, s = f2i_clamped(dv);
                    if (!(pv >= (float)L.sc[TOPN - 1] && s >= L.sc[TOPN - 1])) continue;   // the list moved on
                    const unsigned xx = L.cwp ^ ((unsigned)c * 0x01010101u);
                    if ((xx - 0x01010101u) & ~xx & 0x80808080u) continue;                  // already listed (:145-150)
                    scan_insert(L, c, s);
                }
            }
        }
        if (lane == 0) {
            // mgau_norm (:186-203): record as ptm_topn_kernel<SEMI> writes it
            const int f = k;                                       // one codebook: pair index = stream
            const int top = L.sc[0] >> PSB_SENSCR_SHIFT;
            unsigned eb = 0;
            int n_in_beam = TOPN;
#pragma unroll
            for (int j = 0; j < TOPN; ++j) {
                int e = top - (L.sc[j] >> PSB_SENSCR_SHIFT);
                e = e > PSB_MAX_NEG_ASCR ? PSB_MAX_NEG_ASCR : e;
                const int beam = topn_beam[f];
                if (beam && e > beam && n_in_beam == TOPN) n_in_beam = j;
                eb |= (unsigned)e << (8 * j);
            }
            out[(f0 + t) * K + k] = make_int4(n_in_beam, (int)L.cwp, (int)eb, 0);
        }
    }
}

constexpr int SEN_BIAS = 64;          // > 3 * tab[0] for any 8-bit add table the 16x2 senone kernel accepts

// fast_logmath_add (tied_mgau_common.h:111-127) on negated logs.  mixw + normalised score can
// reach 255 + 96, so |x - y| can exceed the reference's 256-entry table (logmath.c:116-120):
// the reference then reads past its allocation (undefined); the add table is identically 0 from
// entry ~30 on, so the kernels continue it with zeros up to PSB_LOGADD8_N entries.
__device__ __forceinline__ int logadd8(const uint8_t *tab, int x, int y)
{
    return min(x, y) - tab[abs(x - y)];
}

template <bool FOURBIT>
__global__ void __launch_bounds__(512)
ptm_senone_kernel(const int4 *__restrict__ topn, const uint8_t *__restrict__ mixw,
                  const uint8_t *__restrict__ mixw_cb, const uint16_t *__restrict__ sen2cb,
                  const uint8_t *__restrict__ logadd_tab, int16_t *__restrict__ senscr,
                  int n_sen, int n_feat, int nd, int K, int mixw_stride)
{
    extern __shared__ int smem_i[];
    // per (codebook, stream) pair i: rowoff[i] = byte offsets of the four listed codewords'
    // mixture-weight rows, nsc[i] = their normalised scores (0..96)
    uint4 *rowoff = reinterpret_cast<uint4 *>(smem_i);             // [K]
    uint4 *nsc = rowoff + K;                                        // [K]
    int *norm = reinterpret_cast<int *>(nsc + K);                   // [8]
    int *red = norm + 8;                                            // [32]
    uint8_t *tab = reinterpret_cast<uint8_t *>(red + 32);           // [PSB_LOGADD8_N]
    uint8_t *cb16 = tab + PSB_LOGADD8_N;                            // [16]
    int16_t *asc = reinterpret_cast<int16_t *>(cb16 + 16);          // [n_sen]
    const long long frame = blockIdx.x;
    const int tid = threadIdx.x;

    for (int i = tid; i < PSB_LOGADD8_N; i += blockDim.x) tab[i] = logadd_tab[i];
    if (FOURBIT && tid < 16) cb16[tid] = mixw_cb[tid];
    if (tid < n_feat) norm[tid] = PSB_WORST_SCORE;                 // ptm_mgau.c:273
    __syncthreads();
    // ptm_mgau_codebook_norm (ptm_mgau.c:266-295), all codebooks active
    int4 r = make_int4(0, 0, 0, 0);
    if (tid < K) {
        r = topn[frame * K + tid];
        atomicMax(&norm[tid % n_feat], r.x);
    }
    __syncthreads();
    if (tid < K) {
        const int f = tid % n_feat;
        const int base = norm[f] - r.x;
        const unsigned eb = (unsigned)r.z, cwb = (unsigned)r.y;
        unsigned ro[TOPN], nv[TOPN];
#pragma unroll
        for (int j = 0; j < TOPN; ++j) {
            int v = base + (int)((eb >> (8 * j)) & 0xff);
            nv[j] = (unsigned)(v > PSB_MAX_NEG_ASCR ? PSB_MAX_NEG_ASCR : v);
            ro[j] = ((unsigned)f * nd + ((cwb >> (8 * j)) & 0xff)) * (unsigned)mixw_stride;
        }
        rowoff[tid] = make_uint4(ro[0], ro[1], ro[2], ro[3]);
        nsc[tid] = make_uint4(nv[0], nv[1], nv[2], nv[3]);
    }
    __syncthreads();

    // ptm_mgau_senone_eval (ptm_mgau.c:327-403), compallsen
    int best = 0x7fffffff;
    for (int s = tid; s < n_sen; s += blockDim.x) {
        const int i0 = (int)sen2cb[s] * n_feat;
        const uint8_t *__restrict__ mw = mixw + (FOURBIT ? (s >> 1) : s);     // column of this senone
        int ascore = 0;
        for (int f = 0; f < n_feat; ++f) {
            const uint4 ro = rowoff[i0 + f], nv = nsc[i0 + f];
            int w0 = mw[ro.x], w1 = mw[ro.y], w2 = mw[ro.z], w3 = mw[ro.w];
            if (FOURBIT) {                                     // sic: low bit of the byte (ptm_mgau.c:376-377)
                w0 = cb16[(w0 & 1) ? w0 >> 4 : w0 & 0x0f];
                w1 = cb16[(w1 & 1) ? w1 >> 4 : w1 & 0x0f];
                w2 = cb16[(w2 & 1) ? w2 >> 4 : w2 & 0x0f];
                w3 = cb16[(w3 & 1) ? w3 >> 4 : w3 & 0x0f];
            }
            int fden = w0 + (int)nv.x;
            fden = logadd8(tab, fden, w1 + (int)nv.y);
            fden = logadd8(tab, fden, w2 + (int)nv.z);
            fden = logadd8(tab, fden, w3 + (int)nv.w);
            ascore += fden;
        }
        best = min(best, ascore);
        asc[s] = (int16_t)ascore;
    }
    // block-wide min
    best = __reduce_min_sync(0xffffffffu, best);
    if ((tid & 31) == 0) red[tid >> 5] = best;
    __syncthreads();
    if (tid < 32) {
        int v = tid < (int)(blockDim.x >> 5) ? red[tid] : 0x7fffffff;
        v = __reduce_min_sync(0xffffffffu, v);
        if (tid == 0) red[0] = v;
    }
    __syncthreads();
    best = red[0];
    int16_t *dst = senscr + frame * n_sen;
    for (int s = tid; s < n_sen; s += blockDim.x)
        dst[s] = (int16_t)(asc[s] - best);                       // ptm_mgau.c:398-400
}

// s2_semi_mgau_frame_eval's senone part, compallsen (get_scores_{8b,4b}_feat_all,
// s2_semi_mgau.c:425-444, 797-831): per stream, log-add mixw + score over the entries inside
// the beam, accumulate into the int16 score.  The 4-bit variant walks senone pairs and stops at
// n_sen & ~1 (:809); nibbles: even senone = low, odd = high (:813-814).
template <bool FOURBIT>
__global__ void __launch_bounds__(256)
semi_senone_kernel(const int4 *__restrict__ topn, const uint8_t *__restrict__ mixw,
                   const uint8_t *__restrict__ mixw_cb, const uint8_t *__restrict__ logadd_tab,
                   int16_t *__restrict__ senscr, int n_sen, int n_feat, int nd, int mixw_stride)
{
    extern __shared__ int smem_i[];
    uint4 *rowoff = reinterpret_cast<uint4 *>(smem_i);             // [n_feat]
    uint4 *nsc = rowoff + n_feat;                                   // [n_feat]
    uint8_t *tab = reinterpret_cast<uint8_t *>(nsc + n_feat);       // [PSB_LOGADD8_N]
    uint8_t *cb16 = tab + PSB_LOGADD8_N;                            // [16]
    __shared__ int cnt[PSB_MAX_FEAT];
    const long long frame = blockIdx.x;
    const int tid = threadIdx.x;
    for (int i = tid; i < PSB_LOGADD8_N; i += blockDim.x) tab[i] = logadd_tab[i];
    if (FOURBIT && tid < 16) cb16[tid] = mixw_cb[tid];
    if (tid < n_feat) {
        const int4 r = topn[frame * n_feat + tid];
        const unsigned cwb = (unsigned)r.y, eb = (unsigned)r.z;
        unsigned ro[TOPN], nv[TOPN];
#pragma unroll
        for (int j = 0; j < TOPN; ++j) {
            ro[j] = ((unsigned)tid * nd + ((cwb >> (8 * j)) & 0xff)) * (unsigned)mixw_stride;
            nv[j] = (eb >> (8 * j)) & 0xff;
        }
        rowoff[tid] = make_uint4(ro[0], ro[1], ro[2], ro[3]);
        nsc[tid] = make_uint4(nv[0], nv[1], nv[2], nv[3]);
        cnt[tid] = r.x;
    }
    __syncthreads();
    const int s = blockIdx.y * blockDim.x + tid;
    if (s >= n_sen) return;
    int16_t acc = 0;
    if (!FOURBIT || s < (n_sen & ~1)) {
        for (int f = 0; f < n_feat; ++f) {
            const uint4 ro = rowoff[f], nv = nsc[f];
            const unsigned rr[TOPN] = {ro.x, ro.y, ro.z, ro.w}, vv[TOPN] = {nv.x, nv.y, nv.z, nv.w};
            const int n = cnt[f];
            int tmp = 0;
#pragma unroll
            for (int k = 0; k < TOPN; ++k) {
                if (k == 0 || k < n) {
                    int w;
                    if (FOURBIT) {
                        const int b = mixw[rr[k] + (unsigned)(s >> 1)];
                        w = cb16[(s & 1) ? b >> 4 : b & 0x0f];
                    }
                    else
                        w = mixw[rr[k] + (unsigned)s];
                    const int v = w + (int)vv[k];
                    tmp = k == 0 ? v : logadd8(tab, tmp, v);
                }
            }
            acc = (int16_t)(acc + tmp);                      // int16 += (s2_semi_mgau.c:441)
        }
    }
    senscr[frame * n_sen + s] = acc;
}

// Four consecutive senones per thread (8-bit mixture weights).  ncu on ptm_senone_kernel shows
// the L1/LSU data pipe at ~90 %: one byte gather per (senone, codeword) and one broadcast LDS of
// row offsets per (senone, stream).  Senones of one codebook are contiguous, so a thread that
// owns senones 4q..4q+3 fetches each weight row with ONE aligned 32-bit load (four senones'
// bytes) and reads the codebook's offsets/scores once; quads that straddle a codebook boundary
// (a few per cent) take the per-senone path.
__global__ void __launch_bounds__(512)
ptm_senone4_kernel(const int4 *__restrict__ topn, const uint8_t *__restrict__ mixw,
                   const uint16_t *__restrict__ sen2cb, const int16_t *__restrict__ quadcb,
                   const int32_t *__restrict__ bsen, int n_bsen, const uint8_t *__restrict__ logadd_tab,
                   int16_t *__restrict__ senscr, int n_sen, int n_feat, int nd, int K, int mixw_stride)
{
    // quadcb[q] = codebook of senones 4q..4q+3 when all four exist and share it, else -1;
    // bsen[] = the senones of the other quads (codebook boundaries, tail), handled one by one.
    extern __shared__ int smem_i[];
    uint4 *rowoff = reinterpret_cast<uint4 *>(smem_i);             // [K]
    uint4 *nsc = rowoff + K;                                        // [K]
    uint4 *nvp = nsc + K;                                           // [K] (score + SEN_BIAS) in both halfwords
    int *norm = reinterpret_cast<int *>(nvp + K);                   // [8]
    int *red = norm + 8;                                            // [32]
    uint8_t *tab = reinterpret_cast<uint8_t *>(red + 32);           // [PSB_LOGADD8_N]
    int16_t *asc = reinterpret_cast<int16_t *>(tab + PSB_LOGADD8_N + 16);     // [n_sen rounded up to 4]
    const long long frame = blockIdx.x;
    const int tid = threadIdx.x;

    for (int i = tid; i < PSB_LOGADD8_N; i += blockDim.x) tab[i] = logadd_tab[i];
    if (tid < n_feat) norm[tid] = PSB_WORST_SCORE;
    __syncthreads();
    int4 r = make_int4(0, 0, 0, 0);
    if (tid < K) {
        r = topn[frame * K + tid];
        atomicMax(&norm[tid % n_feat], r.x);
    }
    __syncthreads();
    if (tid < K) {
        const int f = tid % n_feat;
        const int base = norm[f] - r.x;
        const unsigned eb = (unsigned)r.z, cwb = (unsigned)r.y;
        unsigned ro[TOPN], nv[TOPN];
#pragma unroll
        for (int j = 0; j < TOPN; ++j) {
            int v = base + (int)((eb >> (8 * j)) & 0xff);
            nv[j] = (unsigned)(v > PSB_MAX_NEG_ASCR ? PSB_MAX_NEG_ASCR : v);
            ro[j] = ((unsigned)f * nd + ((cwb >> (8 * j)) & 0xff)) * (unsigned)mixw_stride;
        }
        rowoff[tid] = make_uint4(ro[0], ro[1], ro[2], ro[3]);
        nsc[tid] = make_uint4(nv[0], nv[1], nv[2], nv[3]);
        nvp[tid] = make_uint4((nv[0] + SEN_BIAS) * 0x10001u, (nv[1] + SEN_BIAS) * 0x10001u,
                              (nv[2] + SEN_BIAS) * 0x10001u, (nv[3] + SEN_BIAS) * 0x10001u);
    }
    __syncthreads();

    int best = 0x7fffffff;
    const int n_quads = (n_sen + 3) >> 2;
    for (int q = tid; q < n_quads; q += blockDim.x) {
        const int c = quadcb[q];
        if (c < 0) continue;
        const int s0 = q << 2, i0 = c * n_feat;
        const uint8_t *mw = mixw + s0;
        // Two senones per 32-bit word (unsigned 16x2), all values biased by SEN_BIAS so that the
        // slightly negative intermediate results of fast_logmath_add (>= -3 * tab[0]) stay
        // non-negative halfwords: min, max and |x - y| are bias-free, r - tab[d] carries it.
        unsigned acc01 = 0u, acc23 = 0u;
        for (int f = 0; f < n_feat; ++f) {
            const uint4 ro = rowoff[i0 + f], nv = nvp[i0 + f];
            const unsigned w0 = *reinterpret_cast<const unsigned *>(mw + ro.x);
            const unsigned w1 = *reinterpret_cast<const unsigned *>(mw + ro.y);
            const unsigned w2 = *reinterpret_cast<const unsigned *>(mw + ro.z);
            const unsigned w3 = *reinterpret_cast<const unsigned *>(mw + ro.w);
            unsigned x01 = __byte_perm(w0, 0u, 0x4140) + nv.x;       // (mixw + score + bias) of senones 0,1
            unsigned x23 = __byte_perm(w0, 0u, 0x4342) + nv.x;       // ... of senones 2,3
#define PSB_LADD2(x, w, sel, nvj)                                                               \
            {                                                                                   \
                const unsigned y = __byte_perm(w, 0u, sel);                                     \
                const unsigned mn = __viaddmin_u16x2(y, nvj, x);                                \
                const unsigned mx = __viaddmax_u16x2(y, nvj, x);                                \
                const unsigned d = mx - mn;                                                     \
                const unsigned t = (unsigned)tab[d & 0xffffu] | ((unsigned)tab[d >> 16] << 16); \
                x = mn - t;                                                                     \
            }
            PSB_LADD2(x01, w1, 0x4140, nv.y) PSB_LADD2(x23, w1, 0x4342, nv.y)
            PSB_LADD2(x01, w2, 0x4140, nv.z) PSB_LADD2(x23, w2, 0x4342, nv.z)
            PSB_LADD2(x01, w3, 0x4140, nv.w) PSB_LADD2(x23, w3, 0x4342, nv.w)
#undef PSB_LADD2
            acc01 += x01;
            acc23 += x23;
        }
        const int unbias = n_feat * SEN_BIAS;
        const int a0 = (int)(acc01 & 0xffffu) - unbias, a1 = (int)(acc01 >> 16) - unbias;
        const int a2 = (int)(acc23 & 0xffffu) - unbias, a3 = (int)(acc23 >> 16) - unbias;
        best = min(min(best, a0), min(min(a1, a2), a3));
        *reinterpret_cast<short4 *>(asc + s0) = make_short4((short)a0, (short)a1, (short)a2, (short)a3);
    }
    for (int i = tid; i < n_bsen; i += blockDim.x) {
        const int s = bsen[i];
        const int i0 = (int)sen2cb[s] * n_feat;
        const uint8_t *mw = mixw + s;
        int ascore = 0;
        for (int f = 0; f < n_feat; ++f) {
            const uint4 ro = rowoff[i0 + f], nv = nsc[i0 + f];
            int fden = mw[ro.x] + (int)nv.x;
            fden = logadd8(tab, fden, mw[ro.y] + (int)nv.y);
            fden = logadd8(tab, fden, mw[ro.z] + (int)nv.z);
            fden = logadd8(tab, fden, mw[ro.w] + (int)nv.w);
            ascore += fden;
        }
        best = min(best, ascore);
        asc[s] = (int16_t)ascore;
    }
    best = __reduce_min_sync(0xffffffffu, best);
    if ((tid & 31) == 0) red[tid >> 5] = best;
    __syncthreads();
    if (tid < 32) {
        int v = tid < (int)(blockDim.x >> 5) ? red[tid] : 0x7fffffff;
        v = __reduce_min_sync(0xffffffffu, v);
        if (tid == 0) red[0] = v;
    }
    __syncthreads();
    best = red[0];
    int16_t *dst = senscr + frame * n_sen;
    for (int s = tid; s < n_sen; s += blockDim.x)
        dst[s] = (int16_t)(asc[s] - best);                       // ptm_mgau.c:398-400
}

template <int FL>
int launch_topn2(psb_batch_t *b, const int32_t *d_klist, int n_k, const GroupTabs &tabs, int n_groups,
                 const int32_t *d_featoff)
{
    psb_model_t *m = b->m;
    constexpr int RECF2 = (2 + 4 * FL + 3) / 4 * 4;
    size_t smem = (size_t)(m->n_density / 2) * RECF2 * sizeof(float);
    auto kern = ptm_topn2_kernel<FL>;
    PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(n_k, (n_groups + TOPN_WARPS - 1) / TOPN_WARPS);
    kern<<<grid, TOPN_WARPS * 32, smem, b->stream>>>(m->d_rec2, m->d_rec2_off, d_klist, b->d_featT, tabs, b->d_topn, n_groups,
                                                    m->n_density, m->n_feat, m->sumlen, d_featoff, m->K, m->ds_ratio,
                                                    m->d_topn_beam);
    PSB_LAUNCH_CHECK();
    return PSB_OK;
}

template <int FL>
int launch_topnq(psb_batch_t *b, const int32_t *d_klist, int n_k, const GroupTabs &tabs, int n_groups,
                 const int32_t *d_featoff)
{
    psb_model_t *m = b->m;
    constexpr int RECF2 = (2 + 4 * FL + 3) / 4 * 4;
    const size_t smem = (size_t)(m->n_density / 2) * RECF2 * sizeof(float) + (size_t)QCAP * TOPN_WARPS * 32 * sizeof(float);
    auto kern = ptm_topnq_kernel<FL>;
    PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(n_k, (n_groups + TOPN_WARPS - 1) / TOPN_WARPS);
    kern<<<grid, TOPN_WARPS * 32, smem, b->stream>>>(m->d_rec2, m->d_rec2_off, d_klist, b->d_featT, tabs, b->d_topn, n_groups,
                                                    m->n_density, m->n_feat, m->sumlen, d_featoff, m->K, m->ds_ratio);
    PSB_LAUNCH_CHECK();
    return PSB_OK;
}

// The scan for the streams of length FL: the scalar kernel for fixed point (integer distances) and for streams longer
// than 16 dimensions (the packed kernels' register budget), else the packed kernels -- ptm_topnq_kernel for PTM,
// ptm_topn2_kernel for semi-continuous models.
template <int FL, bool SEMI>
int launch_topn(psb_batch_t *b, const int32_t *d_klist, int n_k, const GroupTabs &tabs, int n_groups,
                const int32_t *d_featoff)
{
    psb_model_t *m = b->m;
    constexpr int FLP = FL <= 16 ? FL : 1;
    if (FL <= 16 && !m->fixed_point)
        return SEMI ? launch_topn2<FLP>(b, d_klist, n_k, tabs, n_groups, d_featoff)
                    : launch_topnq<FLP>(b, d_klist, n_k, tabs, n_groups, d_featoff);
    size_t smem = (size_t)m->n_density * rec_floats(FL) * sizeof(float);
    auto kern = m->fixed_point ? ptm_topn_kernel<FL, SEMI, true> : ptm_topn_kernel<FL, SEMI, false>;
    PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // few (pair, group) items (semi-continuous models, small batches): one warp per CTA spreads
    // them over more SMs; otherwise 4 warps share one staged codebook
    const int warps = (long long)n_k * ((n_groups + TOPN_WARPS - 1) / TOPN_WARPS) >= 4 * 148 ? TOPN_WARPS : 1;
    dim3 grid(n_k, (n_groups + warps - 1) / warps);
    kern<<<grid, warps * 32, smem, b->stream>>>(m->d_rec, m->d_rec_off, d_klist, b->d_featT, tabs, b->d_topn, n_groups,
                                               m->n_density, m->n_feat, m->sumlen, d_featoff, m->K, m->ds_ratio,
                                               m->d_topn_beam);
    PSB_LAUNCH_CHECK();
    return PSB_OK;
}

// Semi-continuous senone evaluation, 8-bit weights: one CTA per frame, four senones per thread,
// two senones per 32-bit word (the 16x2 arithmetic of ptm_senone4_kernel).  get_scores_8b_feat_*
// (s2_semi_mgau.c:206-330): per stream the first n = mgau_norm count (at least one) listed codewords
// are log-added, streams are summed in int16 (:441), no best-score normalisation.
__global__ void __launch_bounds__(512)
semi_senone4_kernel(const int4 *__restrict__ topn, const uint8_t *__restrict__ mixw,
                    const uint8_t *__restrict__ logadd_tab, int16_t *__restrict__ senscr, int n_sen, int n_feat, int nd,
                    int mixw_stride)
{
    __shared__ uint4 rowoff[PSB_MAX_FEAT], nvp[PSB_MAX_FEAT], nsc[PSB_MAX_FEAT];
    __shared__ int cnt[PSB_MAX_FEAT];
    __shared__ uint8_t tab[PSB_LOGADD8_N];
    const long long frame = blockIdx.x;
    const int tid = threadIdx.x;
    for (int i = tid; i < PSB_LOGADD8_N; i += blockDim.x) tab[i] = logadd_tab[i];
    if (tid < n_feat) {
        const int4 r = topn[frame * n_feat + tid];
        const unsigned cwb = (unsigned)r.y, eb = (unsigned)r.z;
        unsigned ro[TOPN], nv[TOPN];
#pragma unroll
        for (int j = 0; j < TOPN; ++j) {
            ro[j] = ((unsigned)tid * nd + ((cwb >> (8 * j)) & 0xff)) * (unsigned)mixw_stride;
            nv[j] = (eb >> (8 * j)) & 0xff;
        }
        rowoff[tid] = make_uint4(ro[0], ro[1], ro[2], ro[3]);
        nsc[tid] = make_uint4(nv[0], nv[1], nv[2], nv[3]);
        nvp[tid] = make_uint4((nv[0] + SEN_BIAS) * 0x10001u, (nv[1] + SEN_BIAS) * 0x10001u,
                              (nv[2] + SEN_BIAS) * 0x10001u, (nv[3] + SEN_BIAS) * 0x10001u);
        cnt[tid] = r.x;
    }
    __syncthreads();
    int16_t *dst = senscr + frame * n_sen;
    const int n_quads = n_sen >> 2;
    for (int q = tid; q < n_quads; q += blockDim.x) {
        const int s0 = q << 2;
        const uint8_t *mw = mixw + s0;
        short a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        for (int f = 0; f < n_feat; ++f) {
            const uint4 ro = rowoff[f], nv = nvp[f];
            const int n = cnt[f];
            const unsigned w0 = *reinterpret_cast<const unsigned *>(mw + ro.x);
            unsigned x01 = __byte_perm(w0, 0u, 0x4140) + nv.x, x23 = __byte_perm(w0, 0u, 0x4342) + nv.x;
#define PSB_LADD2(x, w, sel, nvj)                                                               \
            {                                                                                   \
                const unsigned y = __byte_perm(w, 0u, sel);                                     \
                const unsigned mn = __viaddmin_u16x2(y, nvj, x);                                \
                const unsigned mx = __viaddmax_u16x2(y, nvj, x);                                \
                const unsigned d = mx - mn;                                                     \
                const unsigned t = (unsigned)tab[d & 0xffffu] | ((unsigned)tab[d >> 16] << 16); \
                x = mn - t;                                                                     \
            }
            if (n > 1) {
                const unsigned w1 = *reinterpret_cast<const unsigned *>(mw + ro.y);
                PSB_LADD2(x01, w1, 0x4140, nv.y) PSB_LADD2(x23, w1, 0x4342, nv.y)
            }
            if (n > 2) {
                const unsigned w2 = *reinterpret_cast<const unsigned *>(mw + ro.z);
                PSB_LADD2(x01, w2, 0x4140, nv.z) PSB_LADD2(x23, w2, 0x4342, nv.z)
            }
            if (n > 3) {
                const unsigned w3 = *reinterpret_cast<const unsigned *>(mw + ro.w);
                PSB_LADD2(x01, w3, 0x4140, nv.w) PSB_LADD2(x23, w3, 0x4342, nv.w)
            }
#undef PSB_LADD2
            a0 = (short)(a0 + (int)(x01 & 0xffffu) - SEN_BIAS);          // int16 += (s2_semi_mgau.c:441)
            a1 = (short)(a1 + (int)(x01 >> 16) - SEN_BIAS);
            a2 = (short)(a2 + (int)(x23 & 0xffffu) - SEN_BIAS);
            a3 = (short)(a3 + (int)(x23 >> 16) - SEN_BIAS);
        }
        if ((((uintptr_t)(dst + s0)) & 7) == 0)
            *reinterpret_cast<short4 *>(dst + s0) = make_short4(a0, a1, a2, a3);
        else { dst[s0] = a0; dst[s0 + 1] = a1; dst[s0 + 2] = a2; dst[s0 + 3] = a3; }
    }
    for (int s = (n_quads << 2) + tid; s < n_sen; s += blockDim.x) {       // tail senones one by one
        int16_t acc = 0;
        for (int f = 0; f < n_feat; ++f) {
            const uint4 ro = rowoff[f], nv = nsc[f];
            const unsigned rr[TOPN] = {ro.x, ro.y, ro.z, ro.w}, vv[TOPN] = {nv.x, nv.y, nv.z, nv.w};
            const int n = cnt[f];
            int tmp = 0;
#pragma unroll
            for (int k = 0; k < TOPN; ++k)
                if (k == 0 || k < n) {
                    const int v = mixw[rr[k] + (unsigned)s] + (int)vv[k];
                    tmp = k == 0 ? v : logadd8(tab, tmp, v);
                }
            acc = (int16_t)(acc + tmp);
        }
        dst[s] = acc;
    }
}

}  // namespace

// Host side of one batched scoring pass.  d_feats: [total][D] on the device.
int psb_launch_ptm_batch(psb_batch_t *b, const float *d_feats, const int32_t *utt_off, int32_t n_utt,
                         int16_t *d_senscr)
{
    psb_model_t *m = b->m;
    PSB_REQUIRE(m->kind == PSB_KIND_PTM || m->kind == PSB_KIND_SEMI, "psb_launch_ptm_batch: model is neither PTM nor semi-continuous");
    const bool semi = m->kind == PSB_KIND_SEMI;
    PSB_REQUIRE(m->topn == TOPN, "tied-mixture batch kernels are built for -topn 4 (got %d)", m->topn);
    PSB_REQUIRE(m->n_density % 32 == 0 && m->n_density <= 32 * MAX_NDW,
                "PTM batch kernels need n_density in {32..256, multiple of 32} (got %d)", m->n_density);
    const long long total = utt_off[n_utt];
    PSB_REQUIRE(n_utt <= b->max_utts && total <= b->max_frames, "batch too large for this psb_batch_t");
    b->last_frames = total;
    if (total == 0 || n_utt == 0) return PSB_OK;
    const int D = m->sumlen, K = m->K;

    // ---- group utterances 32 per warp, longest first (ragged batches stay dense) ----
    std::vector<int> perm(n_utt);
    std::iota(perm.begin(), perm.end(), 0);
    std::stable_sort(perm.begin(), perm.end(), [&](int a, int c) {
        return utt_off[a + 1] - utt_off[a] > utt_off[c + 1] - utt_off[c];
    });
    const int n_groups = (n_utt + 31) / 32;
    // table layout in one int32 buffer: lane_len[G*32] lane_off[G*32] grp_maxT[G] klist[K] featoff[8]
    //                                   then 8-byte aligned: grp_base[G] warp_base[G+1]
    size_t n32 = (size_t)n_groups * 64 + n_groups + K + PSB_MAX_FEAT;
    n32 = (n32 + 1) & ~(size_t)1;
    size_t need = n32 + 2 * (size_t)(2 * n_groups + 1);
    if (need > b->tab_cap) {
        if (b->d_tab) cudaFree(b->d_tab);
        if (b->h_tab) cudaFreeHost(b->h_tab);
        b->tab_cap = need * 2;
        PSB_CUDA(cudaMalloc(&b->d_tab, b->tab_cap * sizeof(int32_t)));
        PSB_CUDA(cudaMallocHost(&b->h_tab, b->tab_cap * sizeof(int32_t)));
    }
    int32_t *lane_len = b->h_tab, *lane_off = lane_len + n_groups * 32, *grp_maxT = lane_off + n_groups * 32;
    int32_t *klist = grp_maxT + n_groups, *featoff = klist + K;
    long long *grp_base = reinterpret_cast<long long *>(b->h_tab + n32), *warp_base = grp_base + n_groups;
    long long featT_floats = 0, items = 0;
    for (int g = 0; g < n_groups; ++g) {
        int mx = 0;
        for (int l = 0; l < 32; ++l) {
            int idx = g * 32 + l;
            if (idx < n_utt) {
                int u = perm[idx];
                lane_len[idx] = utt_off[u + 1] - utt_off[u];
                lane_off[idx] = utt_off[u];
                mx = std::max(mx, lane_len[idx]);
            }
            else { lane_len[idx] = 0; lane_off[idx] = 0; }
        }
        grp_maxT[g] = mx;
        grp_base[g] = featT_floats;
        warp_base[g] = items;
        featT_floats += (long long)mx * D * 32;
        items += mx;
    }
    warp_base[n_groups] = items;
    for (int f = 0; f < PSB_MAX_FEAT; ++f) featoff[f] = f < m->n_feat ? m->featoff[f] : 0;
    if ((size_t)featT_floats > b->featT_cap) {
        if (b->d_featT) cudaFree(b->d_featT);
        b->featT_cap = (size_t)featT_floats + (featT_floats >> 3);
        PSB_CUDA(cudaMalloc(&b->d_featT, b->featT_cap * sizeof(float)));
    }
    // k lists per distinct feature length
    std::vector<std::vector<int>> byfl;
    std::vector<int> fls;
    for (int f = 0; f < m->n_feat; ++f) {
        size_t i = std::find(fls.begin(), fls.end(), m->featlen[f]) - fls.begin();
        if (i == fls.size()) { fls.push_back(m->featlen[f]); byfl.emplace_back(); }
        for (int cb = 0; cb < m->n_mgau; ++cb) byfl[i].push_back(cb * m->n_feat + f);
    }
    {
        int pos = 0;
        for (auto &v : byfl) for (int k : v) klist[pos++] = k;
    }
    PSB_CUDA(cudaMemcpyAsync(b->d_tab, b->h_tab, need * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream));
    GroupTabs tabs;
    tabs.lane_len = b->d_tab;
    tabs.lane_off = b->d_tab + n_groups * 32;
    tabs.grp_maxT = b->d_tab + n_groups * 64;
    const int32_t *d_klist = b->d_tab + n_groups * 64 + n_groups, *d_featoff = d_klist + K;
    tabs.grp_base = reinterpret_cast<const long long *>(b->d_tab + n32);
    const long long *d_warp_base = tabs.grp_base + n_groups;

    // Top-N kernels, by model shape: the tensor-core filter where psb_tc_usable allows it; else, for semi-continuous
    // models with one codebook and n_density in {64, 128, 256}, the split path (semi_dist / semi_scan); else one scan
    // per stream length (launch_topn).
    const bool use_tc = !semi && psb_tc_usable(b);
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[0], b->stream));
    if (!use_tc) {
        int warps = 8;
        while (warps > 1 && (size_t)warps * 32 * (D + 1) * sizeof(float) > 48 * 1024) warps >>= 1;
        size_t smem = (size_t)warps * 32 * (D + 1) * sizeof(float);
        PSB_REQUIRE(smem <= 48 * 1024, "feature vectors of %d floats are too long for transpose_feats_kernel", D);
        long long blocks = (items + warps - 1) / warps;
        transpose_feats_kernel<<<(unsigned)blocks, warps * 32, smem, b->stream>>>(
            d_feats, b->d_featT, tabs, d_warp_base, n_groups, D);
        PSB_LAUNCH_CHECK();
    }
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[1], b->stream));
    // semi-continuous: distances out of the time loop, one warp per (utterance, stream)
    const bool semi_split = semi && !m->fixed_point && m->n_mgau == 1 &&
                            (m->n_density == 64 || m->n_density == 128 || m->n_density == 256);
    if (use_tc) {
        // no recurrence over time: tensor-core filter, exact rescoring of the survivors, tie fix-up (psb_ptm_tc.cu)
        int rc = psb_launch_ptm_tc(b, d_feats, utt_off, n_utt, d_klist, d_featoff);
        if (rc) return rc;
    }
    else if (semi_split) {
        const size_t need_d = (size_t)K * total * m->n_density;
        if (need_d > b->semi_cap) {
            if (b->d_semi_dist) cudaFree(b->d_semi_dist);
            b->d_semi_dist = nullptr;
            b->semi_cap = need_d + need_d / 8;
            PSB_CUDA(cudaMalloc(&b->d_semi_dist, b->semi_cap * sizeof(float2)));
        }
        if ((size_t)n_utt + 1 > b->uttoff_cap) {
            if (b->d_uttoff) cudaFree(b->d_uttoff);
            b->d_uttoff = nullptr;
            b->uttoff_cap = (size_t)n_utt + 1 + 64;
            PSB_CUDA(cudaMalloc(&b->d_uttoff, b->uttoff_cap * sizeof(int32_t)));
        }
        PSB_CUDA(cudaMemcpyAsync(b->d_uttoff, utt_off, ((size_t)n_utt + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream));
        PSB_REQUIRE(total <= 0x7fffffffLL, "too many frames for one launch");
        int pos = 0;
        for (size_t i = 0; i < fls.size(); ++i) {
            const int n_k = (int)byfl[i].size();
            const dim3 grid((unsigned)total, (unsigned)n_k);
            switch (fls[i]) {
#define CASE(FL) case FL: semi_dist_kernel<FL><<<grid, roundup(m->n_density, 32), 0, b->stream>>>(                     \
                    m->d_rec, m->d_rec_off, d_klist + pos, d_feats, b->d_semi_dist, total, m->n_density, m->n_feat, D, d_featoff); break;
                CASE(13) CASE(12) CASE(24) CASE(3) CASE(39) CASE(1) CASE(2) CASE(4) CASE(8) CASE(16) CASE(26) CASE(32)
#undef CASE
            default:
                psb_set_error("no semi_dist_kernel instantiation for stream length %d", fls[i]);
                return PSB_ERR_ARG;
            }
            PSB_LAUNCH_CHECK();
            pos += n_k;
        }
        const int warps = 4;
        const unsigned blocks = (unsigned)(((long long)n_utt * K + warps - 1) / warps);
        if (m->n_density == 256)
            semi_scan_kernel<8><<<blocks, warps * 32, 0, b->stream>>>(b->d_semi_dist, b->d_uttoff, n_utt, K, total, 256, m->ds_ratio, m->d_topn_beam, b->d_topn);
        else if (m->n_density == 128)
            semi_scan_kernel<4><<<blocks, warps * 32, 0, b->stream>>>(b->d_semi_dist, b->d_uttoff, n_utt, K, total, 128, m->ds_ratio, m->d_topn_beam, b->d_topn);
        else
            semi_scan_kernel<2><<<blocks, warps * 32, 0, b->stream>>>(b->d_semi_dist, b->d_uttoff, n_utt, K, total, 64, m->ds_ratio, m->d_topn_beam, b->d_topn);
        PSB_LAUNCH_CHECK();
    }
    else {
        int pos = 0;
        for (size_t i = 0; i < fls.size(); ++i) {
            int n_k = (int)byfl[i].size(), rc;
            switch (fls[i]) {
#define CASE(FL) case FL: rc = semi ? launch_topn<FL, true>(b, d_klist + pos, n_k, tabs, n_groups, d_featoff) \
                                   : launch_topn<FL, false>(b, d_klist + pos, n_k, tabs, n_groups, d_featoff); break;
                CASE(13) CASE(12) CASE(24) CASE(3) CASE(39) CASE(1) CASE(2) CASE(4) CASE(8) CASE(16) CASE(26) CASE(32)
#undef CASE
            default:
                psb_set_error("no ptm_topn_kernel instantiation for stream length %d", fls[i]);
                return PSB_ERR_ARG;
            }
            if (rc) return rc;
            pos += n_k;
        }
    }
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[2], b->stream));
    // Senone kernels: 8-bit weights take the 16x2 kernel (four senones per thread) when (TOPN - 1) times the largest
    // add-table entry stays below SEN_BIAS, else -- and for 4-bit weights -- the scalar kernel.
    if (semi) {
        size_t smem = (size_t)K * 32 + PSB_LOGADD8_N + 16;
        PSB_REQUIRE(K <= 512, "semi_senone_kernel handles at most 512 streams (got %d)", K);
        const int threads = 256;
        dim3 grid((m->n_sen + threads - 1) / threads, (unsigned)total);
        PSB_REQUIRE(total <= 65535LL * 32768, "too many frames for one launch");
        if (!m->mixw_4bit && (TOPN - 1) * m->logadd8_max < SEN_BIAS && m->mixw_stride % 4 == 0 && m->n_feat <= PSB_MAX_FEAT)
            semi_senone4_kernel<<<(unsigned)total, 512, 0, b->stream>>>(b->d_topn, m->d_mixw, m->d_logadd8, d_senscr, m->n_sen,
                                                                      m->n_feat, m->n_density, m->mixw_stride);
        else if (m->mixw_4bit)
            semi_senone_kernel<true><<<dim3((unsigned)total, (m->n_sen + threads - 1) / threads), threads, smem, b->stream>>>(
                b->d_topn, m->d_mixw, m->d_mixw_cb, m->d_logadd8, d_senscr, m->n_sen, m->n_feat, m->n_density, m->mixw_stride);
        else
            semi_senone_kernel<false><<<dim3((unsigned)total, (m->n_sen + threads - 1) / threads), threads, smem, b->stream>>>(
                b->d_topn, m->d_mixw, m->d_mixw_cb, m->d_logadd8, d_senscr, m->n_sen, m->n_feat, m->n_density, m->mixw_stride);
        (void)grid;
        PSB_LAUNCH_CHECK();
    }
    else {
        size_t smem = (size_t)K * 32 + 8 * 4 + 32 * 4 + PSB_LOGADD8_N + 16 + (size_t)m->n_sen * 2;
        PSB_REQUIRE(K <= 512, "ptm_senone_kernel handles at most 512 (codebook, stream) pairs (got %d)", K);
        PSB_REQUIRE((size_t)m->n_feat * m->n_density * m->mixw_stride < (1ull << 32), "mixture-weight table too large for 32-bit offsets");
        if (m->mixw_4bit) {
            PSB_CUDA(cudaFuncSetAttribute(ptm_senone_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ptm_senone_kernel<true><<<(unsigned)total, 512, smem, b->stream>>>(
                b->d_topn, m->d_mixw, m->d_mixw_cb, m->d_sen2cb, m->d_logadd8, d_senscr, m->n_sen, m->n_feat,
                m->n_density, K, m->mixw_stride);
        }
        else if ((TOPN - 1) * m->logadd8_max >= SEN_BIAS) {
            // the 16x2 arithmetic's bias would not cover the add table (a -logbase closer to 1 than the default)
            PSB_CUDA(cudaFuncSetAttribute(ptm_senone_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ptm_senone_kernel<false><<<(unsigned)total, 512, smem, b->stream>>>(
                b->d_topn, m->d_mixw, m->d_mixw_cb, m->d_sen2cb, m->d_logadd8, d_senscr, m->n_sen, m->n_feat,
                m->n_density, K, m->mixw_stride);
        }
        else {
            // four senones per thread; threads sized so that the quads divide evenly over the block
            const int n_quads = (m->n_sen + 3) / 4;
            const int iters = (n_quads + 511) / 512;
            // at least 256 threads (log-add table staging) and one thread per (codebook, stream) pair
            const int threads = std::min(512, std::max(std::max(256, roundup(K, 32)), roundup((n_quads + iters - 1) / iters, 32)));
            const size_t smem4 = smem + 8 + (size_t)K * 16;
            PSB_CUDA(cudaFuncSetAttribute(ptm_senone4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
            ptm_senone4_kernel<<<(unsigned)total, threads, smem4, b->stream>>>(
                b->d_topn, m->d_mixw, m->d_sen2cb, m->d_quadcb, m->d_bsen, m->n_bsen, m->d_logadd8, d_senscr, m->n_sen,
                m->n_feat, m->n_density, K, m->mixw_stride);
        }
        PSB_LAUNCH_CHECK();
    }
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[3], b->stream));
    return PSB_OK;
}
