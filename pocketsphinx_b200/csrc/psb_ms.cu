// psb_ms.cu -- batched senone evaluation for the generic multi-stream / continuous back-end
// (ms_cont_mgau_frame_eval, ms_mgau.c:192-282): per-codebook ordered top-N distances without
// seeding (gauden_dist / compute_dist, ms_gauden.c:378-509), per-senone mixture with the wide
// log-add table (senone_eval, ms_senone.c:358-407), best-score normalisation with int16 clamps.
//
// Frames are independent on this path (no top-N recurrence), so the grid is (codebook tile x
// frame tile).  Gaussians are stored codebook-minor ("transposed") so that a warp whose lanes are
// consecutive codebooks reads each (density, dimension) parameter pair with one coalesced
// transaction, and each thread carries FT frames through the parameter stream to divide the
// L2 traffic by FT.
#include "psb_internal.cuh"

#include <algorithm>

namespace {

constexpr int FT = 4;          // frames per thread in ms_dist_kernel
constexpr int MAXNT = 8;

struct MsDist { int id; float dist; };

// One thread = one codebook, all streams, FT frames.  out: [frame][cb][f][NT] {id, dist}
template <int NT>
__global__ void __launch_bounds__(128)
ms_dist_kernel(const float *__restrict__ gT, const float *__restrict__ detT, const float *__restrict__ feats,
               int2 *__restrict__ out, long long frame0, long long n_frames, int n_mgau, int n_feat, int nd,
               int sumlen, const int32_t *__restrict__ featlen, const int32_t *__restrict__ featoff)
{
    extern __shared__ float sx[];                     // [FT][sumlen]
    const long long fbase = (long long)blockIdx.y * FT;
    for (int i = threadIdx.x; i < FT * sumlen; i += blockDim.x) {
        const long long fr = fbase + i / sumlen;
        sx[i] = fr < n_frames ? feats[(frame0 + fr) * sumlen + i % sumlen] : 0.f;
    }
    __syncthreads();
    const int cb = blockIdx.x * blockDim.x + threadIdx.x;
    if (cb >= n_mgau) return;
    const bool all = NT >= nd;                        // compute_dist_all (ms_gauden.c:378-419)
    for (int f = 0; f < n_feat; ++f) {
        const int fl = featlen[f], fo = featoff[f];
        int id[FT][NT];
        float ds[FT][NT];
#pragma unroll
        for (int q = 0; q < FT; ++q)
#pragma unroll
            for (int i = 0; i < NT; ++i) { id[q][i] = 0; ds[q][i] = (float)INT_MIN; }     // WORST_DIST (:447-448)
        const float *gp = gT + ((size_t)fo * nd * 2) * n_mgau + cb;
        for (int d = 0; d < nd; ++d) {
            float dv[FT];
            const float det = detT[((size_t)f * nd + d) * n_mgau + cb];
#pragma unroll
            for (int q = 0; q < FT; ++q) dv[q] = det;
            for (int j = 0; j < fl; ++j) {
                const float m = gp[((size_t)(d * fl + j) * 2) * n_mgau];
                const float v = gp[((size_t)(d * fl + j) * 2 + 1) * n_mgau];
#pragma unroll
                for (int q = 0; q < FT; ++q) {
                    const float diff = __fsub_rn(sx[q * sumlen + fo + j], m);
                    dv[q] = __fsub_rn(dv[q], __fmul_rn(__fmul_rn(diff, diff), v));       // :467-470
                }
            }
#pragma unroll
            for (int q = 0; q < FT; ++q) {
                if (all) {
#pragma unroll
                    for (int i = 0; i < NT; ++i)
                        if (i == d) { id[q][i] = d; ds[q][i] = dv[q]; }
                }
                else if (dv[q] >= ds[q][NT - 1]) {     // early exit is result-neutral (:457,:474)
                    // insert before the first entry that is not better (strict '<' scan, :478-483)
                    int p = 0;
#pragma unroll
                    for (int i = 0; i < NT; ++i) p += (dv[q] < ds[q][i]) ? 1 : 0;
#pragma unroll
                    for (int i = NT - 1; i > 0; --i)
                        if (i > p) { ds[q][i] = ds[q][i - 1]; id[q][i] = id[q][i - 1]; }
#pragma unroll
                    for (int i = 0; i < NT; ++i)
                        if (i == p) { ds[q][i] = dv[q]; id[q][i] = d; }
                }
            }
        }
#pragma unroll
        for (int q = 0; q < FT; ++q) {
            const long long fr = fbase + q;
            if (fr >= n_frames) break;
            int2 *o = out + ((fr * n_mgau + cb) * n_feat + f) * NT;
#pragma unroll
            for (int i = 0; i < NT; ++i) o[i] = make_int2(id[q][i], __float_as_int(ds[q][i]));
        }
    }
}

// ---------------------------------------------------------------------------------------
// logmath_add with the shifted table (logmath.c:402-446)
__device__ __forceinline__ int logadd_wide(const uint32_t *__restrict__ tab, int size, int zero, int x, int y)
{
    if (x <= zero) return y;
    if (y <= zero) return x;
    int d, r;
    if (x > y) { d = x - y; r = x; }
    else { d = y - x; r = y; }
    if (d < 0 || d >= size) return r;
    return r + (int)tab[d];
}

// ms_dist_tile_kernel: the same distances with the parameter stream taken out of L2.  ms_dist_kernel
// re-reads every (density, dimension) parameter pair of its 128 codebooks from L2 for every 4 frames
// (2 loads per 16 floating-point operations: 25 % of the FP32 lane rate, L2-bound).  Here a CTA owns a
// tile of 32 codebooks (lane = codebook) and keeps ALL their Gaussians in shared memory -- rows of 32
// floats, one per (stream, density, dimension, {mean, variance term}), conflict-free -- for a whole
// range of frames; its eight warps take eight frames each of a 64-frame block whose feature vectors are
// staged transposed ([dimension][frame]), so that one warp-uniform LDS.128 pair feeds eight frames.
// Per (density, dimension): 2 LDS + 2 broadcast LDS.128 for 32 floating-point operations.  Same
// arithmetic, same order, same insertion rule as ms_dist_kernel: bit-identical lists.
// MS_TFT = 4 frames per thread: sixteen warps per CTA at 64 registers, 32 warps per SM -- against eight frames per
// thread (127 registers, 16 warps per SM), twice the shared-memory instructions per floating-point operation and twice
// the warps to hide them.
constexpr int MS_TCB = 32, MS_TFB = 64, MS_TFT = 4;      // codebooks per CTA, frames per block, frames per thread

// Frame PAIRS go through FADD2 / FMUL2 (x - m == x + (-m) exactly, the means are staged negated; every product and
// difference is rounded separately as before and the running sums stay scalar -- ptxas would contract a packed
// multiply-add): 3 packed + 2 scalar instructions per pair and (density, dimension) instead of 8 scalar.
// FUSE (continuous models: senone s owns codebook s): the lane that holds a codebook's list evaluates the senone on the spot --
// senone_eval (ms_senone.c:358-407) exactly as ms_senone_kernel does, first clamp, raw int16 score, per-frame minimum -- so
// the lists (16 MB per 64 frames at 5138 x 8) never travel to HBM and back and one launch per chunk goes away.
struct MsSenArgs {
    const uint8_t *pdf; const uint32_t *tab; int tab_size, tab_zero; int16_t *senscr; int32_t *best; int n_used, aw;
};

template <int NT, bool FUSE>
__global__ void __launch_bounds__(MS_TFB / MS_TFT * 32, 2)
ms_dist_tile_kernel(const float *__restrict__ gT, const float *__restrict__ detT, const float *__restrict__ feats,
                    int2 *__restrict__ out, long long frame0, long long n_frames, int n_mgau, int n_feat, int nd,
                    int sumlen, const int32_t *__restrict__ featlen, const int32_t *__restrict__ featoff, int frames_per_cta,
                    MsSenArgs sa)
{
    extern __shared__ __align__(16) float tsm[];
    const int n_rows = nd * sumlen * 2, n_det = n_feat * nd;
    float *par = tsm;                                   // [n_rows][32]
    float *dets = par + (size_t)n_rows * MS_TCB;        // [n_det][32]
    float *xs = dets + (size_t)n_det * MS_TCB;          // [sumlen][MS_TFB]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cb = blockIdx.x * MS_TCB + lane;
    const int cbr = cb < n_mgau ? cb : n_mgau - 1;      // padding lanes read the last codebook and write nothing
    for (int r = warp; r < n_rows; r += MS_TFB / MS_TFT) {
        const float g = gT[(size_t)r * n_mgau + cbr];
        par[r * MS_TCB + lane] = !(r & 1) ? -g : g;             // rows alternate mean, variance term
    }
    for (int r = warp; r < n_det; r += MS_TFB / MS_TFT) dets[r * MS_TCB + lane] = detT[(size_t)r * n_mgau + cbr];
    const bool all = NT >= nd;                          // compute_dist_all (ms_gauden.c:378-419)
    const long long f_begin = (long long)blockIdx.y * frames_per_cta;
    const long long f_end = f_begin + frames_per_cta < n_frames ? f_begin + frames_per_cta : n_frames;
    // the next block's features travel while this block is computed: each thread keeps its share in registers
    constexpr int PRE = 6, NTHR = MS_TFB / MS_TFT * 32;
    const bool prefetch = sumlen * MS_TFB <= PRE * NTHR;            // uniform; longer vectors are staged in place
    float pre[PRE];
    auto fetch = [&](long long fb) {
#pragma unroll
        for (int k = 0; k < PRE; ++k) {
            const int i = threadIdx.x + k * NTHR, fr = i & (MS_TFB - 1), j = i / MS_TFB;
            pre[k] = (i < sumlen * MS_TFB && fb + fr < n_frames) ? feats[(frame0 + fb + fr) * sumlen + j] : 0.f;
        }
    };
    if (prefetch && f_begin < f_end) fetch(f_begin);
    for (long long fb = f_begin; fb < f_end; fb += MS_TFB) {
        __syncthreads();                                // the previous block's features are no longer read
        if (prefetch) {
#pragma unroll
            for (int k = 0; k < PRE; ++k) {
                const int i = threadIdx.x + k * NTHR;
                if (i < sumlen * MS_TFB) xs[i] = pre[k];             // xs[j * MS_TFB + fr] with i = j * MS_TFB + fr
            }
        }
        else
            for (int i = threadIdx.x; i < sumlen * MS_TFB; i += blockDim.x) {
                const int fr = i & (MS_TFB - 1), j = i / MS_TFB;
                xs[j * MS_TFB + fr] = fb + fr < n_frames ? feats[(frame0 + fb + fr) * sumlen + j] : 0.f;
            }
        __syncthreads();
        if (prefetch && fb + MS_TFB < f_end) fetch(fb + MS_TFB);
        int sscr[MS_TFT];
#pragma unroll
        for (int q = 0; q < MS_TFT; ++q) sscr[q] = 0;
        for (int f = 0; f < n_feat; ++f) {
            const int fl = featlen[f], fo = featoff[f];
            int id[MS_TFT][NT];
            float ds[MS_TFT][NT];
#pragma unroll
            for (int q = 0; q < MS_TFT; ++q)
#pragma unroll
                for (int i = 0; i < NT; ++i) { id[q][i] = 0; ds[q][i] = (float)INT_MIN; }     // WORST_DIST (:447-448)
            const float *pp = par + (size_t)fo * nd * 2 * MS_TCB + lane;
            for (int d = 0; d < nd; ++d) {
                float dv[MS_TFT];
                const float det = dets[(f * nd + d) * MS_TCB + lane];
#pragma unroll
                for (int q = 0; q < MS_TFT; ++q) dv[q] = det;
                const float *pr = pp + (size_t)d * fl * 2 * MS_TCB;          // this density's (mean, variance term) rows
                const float *xp = xs + fo * MS_TFB + warp * MS_TFT;           // this warp's frames of dimension j
#pragma unroll 4
                for (int j = 0; j < fl; ++j, pr += 2 * MS_TCB, xp += MS_TFB) {
                    const float m = pr[0];
                    const float v = pr[MS_TCB];
                    float xv[MS_TFT];
#pragma unroll
                    for (int q = 0; q < MS_TFT; q += 4) {
                        const float4 xq = *reinterpret_cast<const float4 *>(xp + q);
                        xv[q] = xq.x; xv[q + 1] = xq.y; xv[q + 2] = xq.z; xv[q + 3] = xq.w;
                    }
                    const float2 nm2 = make_float2(m, m), vv = make_float2(v, v);            // m holds the negated mean
#pragma unroll
                    for (int q = 0; q < MS_TFT; q += 2) {
                        float2 t = __fadd2_rn(make_float2(xv[q], xv[q + 1]), nm2);
                        t = __fmul2_rn(t, t);
                        t = __fmul2_rn(t, vv);
                        dv[q] = __fsub_rn(dv[q], t.x);                                       // :467-470
                        dv[q + 1] = __fsub_rn(dv[q + 1], t.y);
                    }
                }
#pragma unroll
                for (int q = 0; q < MS_TFT; ++q) {
                    if (all) {
#pragma unroll
                        for (int i = 0; i < NT; ++i)
                            if (i == d) { id[q][i] = d; ds[q][i] = dv[q]; }
                    }
                    else if (dv[q] >= ds[q][NT - 1]) {     // early exit is result-neutral (:457,:474)
                        // insertion before the first entry that is not better (:478-483) as a swap chain down the sorted
                        // list: the carried element displaces every entry it is >= to, which is the same final list
                        float x = dv[q];
                        int xi = d;
#pragma unroll
                        for (int i = 0; i < NT; ++i) {
                            const bool sw = x >= ds[q][i];
                            const float tv = ds[q][i];
                            const int ti = id[q][i];
                            ds[q][i] = sw ? x : tv; id[q][i] = sw ? xi : ti;
                            x = sw ? tv : x; xi = sw ? ti : xi;
                        }
                    }
                }
            }
            if (FUSE) {
                const uint8_t *w8 = sa.pdf + ((size_t)cbr * n_feat + f) * nd;            // this senone's weights of stream f
#pragma unroll
                for (int q = 0; q < MS_TFT; ++q) {
                    int fscr = 0;
#pragma unroll
                    for (int i = 0; i < NT; ++i)
                        if (i < sa.n_used) {
                            const float dv = ds[q][i];
                            int fden;
                            if (dv < (float)INT_MIN) fden = INT_MIN >> PSB_SENSCR_SHIFT;
                            else fden = (__float2int_rz(dv) + ((1 << PSB_SENSCR_SHIFT) - 1)) >> PSB_SENSCR_SHIFT;
                            const int fw = fden - (int)w8[id[q][i]];
                            fscr = i == 0 ? fw : logadd_wide(sa.tab, sa.tab_size, sa.tab_zero, fscr, fw);
                        }
                    sscr[q] -= fscr;
                }
            }
            else if (cb < n_mgau) {
#pragma unroll
                for (int q = 0; q < MS_TFT; ++q) {
                    const long long fr = fb + warp * MS_TFT + q;
                    if (fr >= n_frames) break;
                    int2 *o = out + ((fr * n_mgau + cb) * n_feat + f) * NT;
#pragma unroll
                    for (int i = 0; i < NT; ++i) o[i] = make_int2(id[q][i], __float_as_int(ds[q][i]));
                }
            }
        }
        if (FUSE) {
#pragma unroll
            for (int q = 0; q < MS_TFT; ++q) {
                const long long fr = fb + warp * MS_TFT + q;                              // warp-uniform
                if (fr >= n_frames) break;
                int scr = sscr[q] / sa.aw;                                                // C division, truncation toward zero (:396)
                scr = min(32767, max(-32768, scr));                                       // :399-404
                if (cb < n_mgau) sa.senscr[(frame0 + fr) * n_mgau + cb] = (int16_t)scr;
                scr = __reduce_min_sync(0xffffffffu, cb < n_mgau ? scr : 0x7fffffff);     // per-frame minimum (ms_mgau.c:218-224)
                if (lane == 0 && scr != 0x7fffffff) atomicMin(&sa.best[fr], scr);
            }
        }
    }
}

// senone_eval (ms_senone.c:358-407) + the first clamp; raw scores and the per-frame minimum.
__global__ void __launch_bounds__(256)
ms_senone_kernel(const int2 *__restrict__ dist, const uint8_t *__restrict__ pdf, const int32_t *__restrict__ sen2cb,
                 const uint32_t *__restrict__ tab, int tab_size, int tab_zero, int16_t *__restrict__ senscr,
                 int32_t *__restrict__ best, long long frame0, int n_sen, int n_mgau, int n_feat, int nd, int nt,
                 int n_used, int aw, int transposed, const int32_t *__restrict__ list, int n_items)
{
    // list == nullptr: all senones (n_items == n_sen); else the absolute ids of the active list
    const long long fr = blockIdx.y;
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    const int s = it < n_items ? (list ? list[it] : it) : n_sen;
    int scr = 0x7fffffff;
    if (s < n_sen) {
        const int cb = sen2cb[s];
        scr = 0;
        for (int f = 0; f < n_feat; ++f) {
            const int2 *l = dist + ((fr * n_mgau + cb) * n_feat + f) * nt;
            int fscr = 0;
            for (int t = 0; t < n_used; ++t) {
                const int2 e = l[t];
                const float dv = __int_as_float(e.y);
                int fden;
                if (dv < (float)INT_MIN) fden = INT_MIN >> PSB_SENSCR_SHIFT;
                else fden = (__float2int_rz(dv) + ((1 << PSB_SENSCR_SHIFT) - 1)) >> PSB_SENSCR_SHIFT;
                const int w = transposed ? pdf[((size_t)f * nd + e.x) * n_sen + s]
                                         : pdf[((size_t)s * n_feat + f) * nd + e.x];
                const int fw = fden - w;
                fscr = t == 0 ? fw : logadd_wide(tab, tab_size, tab_zero, fscr, fw);
            }
            scr -= fscr;
        }
        scr /= aw;                                     // C division, truncation toward zero (:396)
        scr = min(32767, max(-32768, scr));            // :399-404
        senscr[(frame0 + fr) * n_sen + s] = (int16_t)scr;
    }
    // per-frame minimum (ms_mgau.c:218-224)
    scr = __reduce_min_sync(0xffffffffu, scr);
    if ((threadIdx.x & 31) == 0 && scr != 0x7fffffff) atomicMin(&best[fr], scr);
}

// normalise: senscr - best with the second clamp (ms_mgau.c:227-235)
__global__ void __launch_bounds__(256)
ms_norm_kernel(int16_t *__restrict__ senscr, const int32_t *__restrict__ best, long long frame0, int n_sen,
               const int32_t *__restrict__ list, int n_items)
{
    const long long fr = blockIdx.y;
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= n_items) return;
    const int s = list ? list[it] : it;
    int16_t *p = senscr + (frame0 + fr) * n_sen + s;
    int bs = (int)*p - best[fr];
    *p = (int16_t)min(32767, max(-32768, bs));
}

__global__ void fill_i32(int32_t *p, long long n, int32_t v)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace

int psb_launch_ms_batch(psb_batch_t *b, const float *d_feats, const int32_t *utt_off, int32_t n_utt, int16_t *d_senscr)
{
    psb_model_t *m = b->m;
    PSB_REQUIRE(m->kind == PSB_KIND_MS, "psb_launch_ms_batch: model is not ms");
    const long long total = utt_off[n_utt];
    b->last_frames = total;
    if (total == 0) return PSB_OK;
    int nt = 1;
    while (nt < m->topn) nt <<= 1;
    PSB_REQUIRE(nt <= MAXNT, "ms batch kernels support -topn up to %d (got %d)", MAXNT, m->topn);
    const int n_used = std::min(m->topn, m->n_density);     // ms_mgau_init clamps topn (ms_mgau.c:137-143)
    PSB_REQUIRE(m->topn >= m->n_density || nt == m->topn, "ms batch kernels need a power-of-two -topn (got %d)", m->topn);
    const size_t per_frame = (size_t)m->n_mgau * m->n_feat * nt * sizeof(int2);
    const size_t budget = (size_t)2 << 30;
    long long chunk = std::max<long long>(FT, std::min<long long>(total, (long long)(budget / per_frame) / FT * FT));
    chunk = std::min<long long>(chunk, 65535);              // gridDim.y
    if (b->ms_cap < (size_t)chunk * per_frame) {
        cudaFree(b->d_msdist); cudaFree(b->d_msbest);
        b->d_msdist = nullptr; b->d_msbest = nullptr;
        b->ms_cap = (size_t)chunk * per_frame;
        PSB_CUDA(cudaMalloc(&b->d_msdist, b->ms_cap));
        PSB_CUDA(cudaMalloc(&b->d_msbest, 65536 * sizeof(int32_t)));
    }
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[0], b->stream));
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[1], b->stream));
    for (long long f0 = 0; f0 < total; f0 += chunk) {
        const long long n = std::min(chunk, total - f0);
        dim3 g1((m->n_mgau + 127) / 128, (unsigned)((n + FT - 1) / FT));
        size_t smem = (size_t)FT * m->sumlen * sizeof(float);
        int2 *dist = reinterpret_cast<int2 *>(b->d_msdist);
        // the Gaussians of a 32-codebook tile in shared memory when they fit, else ms_dist_kernel (parameters from L2)
        const size_t tile_smem = ((size_t)m->n_density * m->sumlen * 2 + (size_t)m->n_feat * m->n_density) * MS_TCB * sizeof(float)
                                 + (size_t)m->sumlen * MS_TFB * sizeof(float);
        const bool tile = tile_smem <= 100 * 1024;
        // frames per CTA: enough CTAs for ~4 waves of two resident CTAs per SM, whole 32-frame blocks
        const int tiles_x = (m->n_mgau + MS_TCB - 1) / MS_TCB;
        long long fpc = (n * tiles_x + 148LL * 2 * 4 - 1) / (148LL * 2 * 4);
        fpc = std::max<long long>(MS_TFB, (fpc + MS_TFB - 1) / MS_TFB * MS_TFB);
        const dim3 gt((unsigned)tiles_x, (unsigned)((n + fpc - 1) / fpc));
        // continuous models: mixtures evaluated by the lane that holds the list (the kernel writes raw scores and minima)
        const bool fuse = tile && m->sen_is_cb && m->n_mgau > 1;
        MsSenArgs sa = {m->d_mixw, m->d_logadd_ms, m->logadd_ms_size, m->logadd_ms_zero, d_senscr, b->d_msbest, n_used, m->aw};
        if (fuse) {
            fill_i32<<<(unsigned)((n + 255) / 256), 256, 0, b->stream>>>(b->d_msbest, n, 0x7fffffff);
            PSB_LAUNCH_CHECK();
        }
#define PSB_MS_TILE(NT, FUSEV) do {                                                                                        \
            auto kern = ms_dist_tile_kernel<NT, FUSEV>;                                                                   \
            PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem));            \
            kern<<<gt, MS_TFB / MS_TFT * 32, tile_smem, b->stream>>>(m->d_msT, m->d_msdetT, d_feats, dist, f0, n,         \
                m->n_mgau, m->n_feat, m->n_density, m->sumlen, m->d_featlen, m->d_featoff, (int)fpc, sa); } while (0)
#define LAUNCH(NT) do {                                                                                                    \
            if (fuse) PSB_MS_TILE(NT, true);                                                                               \
            else if (tile) PSB_MS_TILE(NT, false);                                                                         \
            else ms_dist_kernel<NT><<<g1, 128, smem, b->stream>>>(m->d_msT, m->d_msdetT, d_feats, dist, f0, n,            \
                m->n_mgau, m->n_feat, m->n_density, m->sumlen, m->d_featlen, m->d_featoff); } while (0)
        switch (nt) {
        case 1: LAUNCH(1); break;
        case 2: LAUNCH(2); break;
        case 4: LAUNCH(4); break;
        default: LAUNCH(8); break;
        }
#undef LAUNCH
#undef PSB_MS_TILE
        PSB_LAUNCH_CHECK();
        dim3 g2((m->n_sen + 255) / 256, (unsigned)n);
        if (!fuse) {
            fill_i32<<<(unsigned)((n + 255) / 256), 256, 0, b->stream>>>(b->d_msbest, n, 0x7fffffff);
            PSB_LAUNCH_CHECK();
            ms_senone_kernel<<<g2, 256, 0, b->stream>>>(dist, m->d_mixw, m->d_sen2cb32, m->d_logadd_ms, m->logadd_ms_size,
                                                        m->logadd_ms_zero, d_senscr, b->d_msbest, f0, m->n_sen, m->n_mgau,
                                                        m->n_feat, m->n_density, nt, n_used, m->aw, m->n_mgau == 1, nullptr, m->n_sen);
            PSB_LAUNCH_CHECK();
        }
        ms_norm_kernel<<<g2, 256, 0, b->stream>>>(d_senscr, b->d_msbest, f0, m->n_sen, nullptr, m->n_sen);
        PSB_LAUNCH_CHECK();
    }
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[2], b->stream));
    if (b->have_ev) PSB_CUDA(cudaEventRecord(b->ev[3], b->stream));
    return PSB_OK;
}

// One frame for the per-frame scorer (psb_scorer.cu): distances for every codebook (results for
// codebooks no listed senone uses are simply not read, which equals the reference skipping them,
// ms_mgau.c:238-252), then only the listed senones are evaluated, normalised among themselves and
// written; d_senscr entries of unlisted senones are left untouched (:254-276).
int psb_ms_score_one(psb_model_t *m, cudaStream_t st, const float *d_feat, void *d_dist, int32_t *d_best,
                     int16_t *d_senscr, const int32_t *d_list, int n_items)
{
    int nt = 1;
    while (nt < m->topn) nt <<= 1;
    PSB_REQUIRE(nt <= MAXNT, "ms kernels support -topn up to %d (got %d)", MAXNT, m->topn);
    PSB_REQUIRE(m->topn >= m->n_density || nt == m->topn, "ms kernels need a power-of-two -topn (got %d)", m->topn);
    const int n_used = std::min(m->topn, m->n_density);
    dim3 g1((m->n_mgau + 127) / 128, 1);
    size_t smem = (size_t)FT * m->sumlen * sizeof(float);
    int2 *dist = reinterpret_cast<int2 *>(d_dist);
#define LAUNCH(NT) ms_dist_kernel<NT><<<g1, 128, smem, st>>>(m->d_msT, m->d_msdetT, d_feat, dist, 0, 1, \
        m->n_mgau, m->n_feat, m->n_density, m->sumlen, m->d_featlen, m->d_featoff)
    switch (nt) {
    case 1: LAUNCH(1); break;
    case 2: LAUNCH(2); break;
    case 4: LAUNCH(4); break;
    default: LAUNCH(8); break;
    }
#undef LAUNCH
    PSB_LAUNCH_CHECK();
    fill_i32<<<1, 32, 0, st>>>(d_best, 1, 0x7fffffff);
    PSB_LAUNCH_CHECK();
    if (n_items == 0) return PSB_OK;
    dim3 g2((n_items + 255) / 256, 1);
    ms_senone_kernel<<<g2, 256, 0, st>>>(dist, m->d_mixw, m->d_sen2cb32, m->d_logadd_ms, m->logadd_ms_size,
                                         m->logadd_ms_zero, d_senscr, d_best, 0, m->n_sen, m->n_mgau, m->n_feat,
                                         m->n_density, nt, n_used, m->aw, m->n_mgau == 1, d_list, n_items);
    PSB_LAUNCH_CHECK();
    ms_norm_kernel<<<g2, 256, 0, st>>>(d_senscr, d_best, 0, m->n_sen, d_list, n_items);
    PSB_LAUNCH_CHECK();
    return PSB_OK;
}

size_t psb_ms_dist_bytes(const psb_model_t *m)
{
    int nt = 1;
    while (nt < m->topn) nt <<= 1;
    return (size_t)m->n_mgau * m->n_feat * nt * sizeof(int2);
}
