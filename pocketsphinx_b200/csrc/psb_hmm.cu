// psb_hmm.cu -- batched hmm_vit_eval and the device-resident phone-loop Viterbi.
#include "psb_hmmctx.cuh"

#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include <vector>


struct psb_phoneloop_s {
    psb_hmmctx_t *c;
    int n_phones, window, beam, pbeam, pip;
    double penalty_weight;
    int32_t *d_ssid, *d_tmatid;
    uint16_t *d_senid;            // [n_emit][n_phones]
    cudaStream_t stream;
    int32_t *d_flags;             // [1] pathological-regime counter
};

namespace {

__device__ __forceinline__ void load_hmm(const psb_hmm_t *p, HmmReg &h, int n)
{
#pragma unroll
    for (int i = 0; i < PSB_HMM_MAX_NSTATE; ++i) {
        h.score[i] = i < n ? p->score[i] : PSB_WORST_SCORE;
        h.hist[i] = i < n ? p->history[i] : -1;
        h.senid[i] = i < n ? p->senid[i] : PSB_BAD_SSID;
    }
    h.out_score = p->out_score;
    h.out_hist = p->out_history;
    h.best = p->bestscore;
}

__device__ __forceinline__ void store_hmm(psb_hmm_t *p, const HmmReg &h, int n, bool mpx)
{
#pragma unroll
    for (int i = 0; i < PSB_HMM_MAX_NSTATE; ++i)
        if (i < n) {
            p->score[i] = h.score[i];
            p->history[i] = h.hist[i];
            if (mpx) p->senid[i] = (uint16_t)h.senid[i];
        }
    p->out_score = h.out_score;
    p->out_history = h.out_hist;
    p->bestscore = h.best;
}

// One thread per hmm_t record (array-of-structs, as the search modules keep them).
__global__ void __launch_bounds__(256)
hmm_eval_aos_kernel(psb_hmm_t *hmms, int n, HmmCtxDev c, const int16_t *__restrict__ senscr, int *best_out)
{
    __shared__ int red[8];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int best = PSB_WORST_SCORE;
    if (i < n) {
        psb_hmm_t *p = hmms + i;
        HmmReg h;
        load_hmm(p, h, c.n_emit);
        const bool mpx = p->mpx != 0;
        best = hmm_step(h, c, p->tmatid, mpx, senscr);
        store_hmm(p, h, c.n_emit, mpx);
    }
    best = __reduce_max_sync(0xffffffffu, best);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x < 32) {
        int v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : PSB_WORST_SCORE;
        v = __reduce_max_sync(0xffffffffu, v);
        if (threadIdx.x == 0) atomicMax(best_out, v);
    }
}

// ---------------------------------------------------------------------------------------
// Phone loop: one CTA per utterance, HMM state in shared memory (struct of arrays), threads
// stride over the HMMs; time is the sequential loop.  All phones are non-multiplexed
// (phone_loop_search.c:98-103).
struct PlParams {
    int n_phones, window, beam, pbeam, pip;
    double penalty_weight;
};

template <typename T>
__device__ __forceinline__ T block_reduce_max_pair(T v, int idx, int *sidx, T *sval, int &out_idx)
{
    // max value, smallest index among ties (first winner in ascending order)
    const unsigned full = 0xffffffffu;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        T ov = __shfl_xor_sync(full, v, o);
        int oi = __shfl_xor_sync(full, idx, o);
        if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) { sval[warp] = v; sidx[warp] = idx; }
    __syncthreads();
    v = sval[0]; idx = sidx[0];
    for (int w = 1; w < nw; ++w) {
        T ov = sval[w]; int oi = sidx[w];
        if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
    out_idx = idx;
    return v;
}

__global__ void __launch_bounds__(1024)
phoneloop_kernel(const int16_t *__restrict__ senscr, const int32_t *__restrict__ utt_off, HmmCtxDev c,
                 PlParams P, const uint16_t *__restrict__ senid_g, const int32_t *__restrict__ tmatid_g,
                 const int32_t *__restrict__ ssid_g,
                 int32_t *__restrict__ best_out, int32_t *__restrict__ pen_out,
                 psb_hmm_t *__restrict__ final_out, psb_hmm_t *__restrict__ trace_out, int32_t *flags)
{
    extern __shared__ int sm[];
    const int H = P.n_phones, N = c.n_emit, tid = threadIdx.x;
    int *score = sm;                       // [N][H]
    int *hist = score + N * H;             // [N][H]
    int *out_score = hist + N * H;         // [H]
    int *out_hist = out_score + H;         // [H]
    int *bestsc = out_hist + H;            // [H]
    int *frame = bestsc + H;               // [H]
    int *pen_buf = frame + H;              // [window][H]
    int *sval = pen_buf + P.window * H;    // [32]
    int *sidx = sval + 32;                 // [32]

    const int u = blockIdx.x;
    const long long f0 = utt_off[u];
    const int T = utt_off[u + 1] - utt_off[u];

    // phone_loop_search_start (:155-175): hmm_clear + hmm_enter(0, -1, 0)
    for (int i = tid; i < H; i += blockDim.x) {
        for (int s = 0; s < N; ++s) { score[s * H + i] = PSB_WORST_SCORE; hist[s * H + i] = -1; }
        out_score[i] = PSB_WORST_SCORE; out_hist[i] = -1; bestsc[i] = PSB_WORST_SCORE;
        score[i] = 0; hist[i] = -1; frame[i] = 0;
        for (int w = 0; w < P.window; ++w) pen_buf[w * H + i] = 0;
    }
    int best_score = 0, pen_ptr = 0;
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        const int16_t *row = senscr + (f0 + t) * c.n_sen;
        // renormalize_hmms (:177-191)
        const bool renorm = best_score + 2 * P.beam < PSB_WORST_SCORE;
        int bs = PSB_WORST_SCORE;
        // evaluate_hmms (:193-214)
        for (int i = tid; i < H; i += blockDim.x) {
            HmmReg h;
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s) {
                h.score[s] = s < N ? score[s * H + i] : PSB_WORST_SCORE;
                h.hist[s] = s < N ? hist[s * H + i] : -1;
                h.senid[s] = s < N ? senid_g[s * H + i] : PSB_BAD_SSID;
            }
            h.out_score = out_score[i]; h.out_hist = out_hist[i]; h.best = bestsc[i];
            if (renorm) {                                    // hmm_normalize (hmm.c:206-216)
#pragma unroll
                for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s)
                    if (s < N && h.score[s] > PSB_WORST_SCORE) h.score[s] -= best_score;
                if (h.out_score > PSB_WORST_SCORE) h.out_score -= best_score;
            }
            if (frame[i] >= t) {
                int b = hmm_step(h, c, tmatid_g[i], false, row);
                if (b > bs) bs = b;
            }
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s)
                if (s < N) { score[s * H + i] = h.score[s]; hist[s * H + i] = h.hist[s]; }
            out_score[i] = h.out_score; out_hist[i] = h.out_hist; bestsc[i] = h.best;
        }
        int dummy;
        bs = block_reduce_max_pair<int>(bs, 0, sidx, sval, dummy);
        best_score = bs;
        // store_scores (:216-239)
        if (P.window > 0) {
            for (int i = tid; i < H; i += blockDim.x)
                pen_buf[pen_ptr * H + i] = (int)((double)(bestsc[i] - best_score) * P.penalty_weight);
            pen_ptr = (pen_ptr + 1) % P.window;
            if (pen_out)
                for (int i = tid; i < H; i += blockDim.x) {
                    int pmax = PSB_WORST_SCORE;
                    for (int w = 0; w < P.window; ++w) pmax = max(pmax, pen_buf[w * H + i]);
                    pen_out[(f0 + t) * H + i] = pmax;
                }
        }
        // prune_hmms (:241-261)
        const int nf = t + 1;
        int thresh = best_score + P.beam;
        // phone_transition (:263-299): candidates among the survivors
        const int xthresh = best_score + P.pbeam;
        int cand = INT_MIN, cidx = 0x7fffffff;
        for (int i = tid; i < H; i += blockDim.x) {
            if (frame[i] < t) continue;
            if (bestsc[i] > thresh) {
                frame[i] = nf;
                const int ns = out_score[i] + P.pip;
                if (ns > xthresh && (ns > cand)) { cand = ns; cidx = i; }
            }
            else {                                           // hmm_clear_scores (hmm.c:167-178)
                for (int s = 0; s < N; ++s) score[s * H + i] = PSB_WORST_SCORE;
                out_score[i] = PSB_WORST_SCORE;
                bestsc[i] = PSB_WORST_SCORE;
            }
        }
        int widx;
        cand = block_reduce_max_pair<int>(cand, cidx, sidx, sval, widx);
        if (tid == 0) {
            if (best_out) best_out[f0 + t] = best_score;
            // sequential-order corner the max formulation does not cover (see DESIGN.md)
            if (cand != INT_MIN && PSB_WORST_SCORE + P.pip > xthresh) atomicAdd(flags, 1);
        }
        if (cand != INT_MIN) {
            const int whist = out_hist[widx];
            __syncthreads();
            for (int i = tid; i < H; i += blockDim.x)
                if (frame[i] < t || cand > score[i]) {       // hmm_enter (hmm.c:198-204)
                    score[i] = cand; hist[i] = whist; frame[i] = nf;
                }
        }
        __syncthreads();
        if (trace_out)
            for (int i = tid; i < H; i += blockDim.x) {
                psb_hmm_t *p = trace_out + (f0 + t) * H + i;
                for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s) {
                    p->score[s] = s < N ? score[s * H + i] : 0;
                    p->history[s] = s < N ? hist[s * H + i] : 0;
                    p->senid[s] = s < N ? senid_g[s * H + i] : 0;
                }
                p->ctx = nullptr; p->out_score = out_score[i]; p->out_history = out_hist[i];
                p->ssid = (uint16_t)ssid_g[i]; p->bestscore = bestsc[i]; p->tmatid = (int16_t)tmatid_g[i];
                p->frame = frame[i]; p->mpx = 0; p->n_emit_state = (uint8_t)N;
            }
    }
    if (final_out)
        for (int i = tid; i < H; i += blockDim.x) {
            psb_hmm_t *p = final_out + (size_t)u * H + i;
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s) {
                p->score[s] = s < N ? score[s * H + i] : 0;
                p->history[s] = s < N ? hist[s * H + i] : 0;
                p->senid[s] = s < N ? senid_g[s * H + i] : 0;
            }
            p->ctx = nullptr; p->out_score = out_score[i]; p->out_history = out_hist[i];
            p->ssid = (uint16_t)ssid_g[i]; p->bestscore = bestsc[i]; p->tmatid = (int16_t)tmatid_g[i];
            p->frame = frame[i]; p->mpx = 0; p->n_emit_state = (uint8_t)N;
        }
}

}  // namespace

// ---------------------------------------------------------------------------------------

extern "C" int psb_hmmctx_create(int32_t n_emit_state, const uint8_t *tp, int32_t n_tmat, const uint16_t *sseq,
                                 int32_t n_sseq, int32_t n_sen, int device, psb_hmmctx_t **out)
{
    PSB_REQUIRE(out && tp && n_emit_state >= 1 && n_emit_state <= PSB_HMM_MAX_NSTATE && n_tmat > 0 && n_sen > 0,
                "psb_hmmctx_create: bad argument");
    PSB_CUDA(cudaSetDevice(device));
    psb_hmmctx_t *c = new psb_hmmctx_t();
    memset(c, 0, sizeof(*c));
    c->device = device; c->n_emit = n_emit_state; c->n_tmat = n_tmat; c->n_sseq = n_sseq; c->n_sen = n_sen;
    size_t tpb = (size_t)n_tmat * n_emit_state * (n_emit_state + 1);
    cudaError_t e = cudaMalloc(&c->d_tp, tpb);
    if (e == cudaSuccess) e = cudaMemcpy(c->d_tp, tp, tpb, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_sseq, std::max<size_t>(2, (size_t)n_sseq * n_emit_state * 2));
    if (e == cudaSuccess && n_sseq > 0 && sseq)
        e = cudaMemcpy(c->d_sseq, sseq, (size_t)n_sseq * n_emit_state * 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_senscr, (size_t)n_sen * 2);
    if (e == cudaSuccess) e = cudaMallocHost(&c->h_senscr, (size_t)n_sen * 2);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_best, 4);
    if (e == cudaSuccess) e = cudaMallocHost(&c->h_best, 4);
    if (e != cudaSuccess) {
        psb_set_error("psb_hmmctx_create: %s", cudaGetErrorString(e));
        psb_hmmctx_free(c);
        return PSB_ERR_CUDA;
    }
    *out = c;
    return PSB_OK;
}

extern "C" void psb_hmmctx_free(psb_hmmctx_t *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    cudaFree(c->d_tp); cudaFree(c->d_sseq); cudaFree(c->d_hmms); cudaFree(c->d_senscr); cudaFree(c->d_best);
    cudaFree(c->d_al_i32); cudaFree(c->d_al_tok); cudaFree(c->d_al_senid); cudaFree(c->d_al_tokoff);
    for (void *p : c->d_srch) cudaFree(p);
    if (c->al_ev[0]) cudaEventDestroy(c->al_ev[0]);
    if (c->al_ev[1]) cudaEventDestroy(c->al_ev[1]);
    if (c->h_hmms) cudaFreeHost(c->h_hmms);
    if (c->h_senscr) cudaFreeHost(c->h_senscr);
    if (c->h_best) cudaFreeHost(c->h_best);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}


static int validate_hmm(const psb_hmmctx_t *c, const psb_hmm_t *h, int i)
{
    PSB_REQUIRE(h->n_emit_state == c->n_emit, "hmm[%d].n_emit_state %d != context %d", i, h->n_emit_state, c->n_emit);
    PSB_REQUIRE(h->tmatid >= 0 && h->tmatid < c->n_tmat, "hmm[%d].tmatid %d out of range", i, h->tmatid);
    for (int s = 0; s < c->n_emit; ++s) {
        if (h->mpx)
            PSB_REQUIRE(h->senid[s] == PSB_BAD_SSID || h->senid[s] < c->n_sseq, "hmm[%d] ssid out of range", i);
        else
            PSB_REQUIRE(h->senid[s] < c->n_sen || (h->senid[s] == PSB_BAD_SSID && c->n_emit != 3 && c->n_emit != 5),
                        "hmm[%d].senid[%d] = %d out of range", i, s, h->senid[s]);
    }
    return PSB_OK;
}

static int ensure_hmm_cap(psb_hmmctx_t *c, size_t n)
{
    if (n <= c->hmm_cap) return PSB_OK;
    if (c->d_hmms) cudaFree(c->d_hmms);
    if (c->h_hmms) cudaFreeHost(c->h_hmms);
    c->d_hmms = nullptr; c->h_hmms = nullptr;
    c->hmm_cap = n + n / 2 + 256;
    PSB_CUDA(cudaMalloc(&c->d_hmms, c->hmm_cap * sizeof(psb_hmm_t)));
    PSB_CUDA(cudaMallocHost(&c->h_hmms, c->hmm_cap * sizeof(psb_hmm_t)));
    return PSB_OK;
}

static int eval_staged(psb_hmmctx_t *c, int32_t n, const int16_t *senscr, int32_t *best)
{
    memcpy(c->h_senscr, senscr, (size_t)c->n_sen * 2);
    *c->h_best = PSB_WORST_SCORE;
    PSB_CUDA(cudaMemcpyAsync(c->d_hmms, c->h_hmms, (size_t)n * sizeof(psb_hmm_t), cudaMemcpyHostToDevice, c->stream));
    PSB_CUDA(cudaMemcpyAsync(c->d_senscr, c->h_senscr, (size_t)c->n_sen * 2, cudaMemcpyHostToDevice, c->stream));
    PSB_CUDA(cudaMemcpyAsync(c->d_best, c->h_best, 4, cudaMemcpyHostToDevice, c->stream));
    hmm_eval_aos_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(c->d_hmms, n, dev_ctx(c), c->d_senscr, c->d_best);
    PSB_LAUNCH_CHECK();
    PSB_CUDA(cudaMemcpyAsync(c->h_hmms, c->d_hmms, (size_t)n * sizeof(psb_hmm_t), cudaMemcpyDeviceToHost, c->stream));
    PSB_CUDA(cudaMemcpyAsync(c->h_best, c->d_best, 4, cudaMemcpyDeviceToHost, c->stream));
    PSB_CUDA(cudaStreamSynchronize(c->stream));
    if (best) *best = *c->h_best;
    return PSB_OK;
}

extern "C" int psb_hmm_vit_eval_batch(psb_hmmctx_t *c, psb_hmm_t *hmms, int32_t n, const int16_t *senscr, int32_t *best)
{
    PSB_REQUIRE(c && n >= 0 && (n == 0 || (hmms && senscr)), "psb_hmm_vit_eval_batch: bad argument");
    if (best) *best = PSB_WORST_SCORE;
    if (n == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(c->device));
    for (int i = 0; i < n; ++i) {
        int rc = validate_hmm(c, &hmms[i], i);
        if (rc) return rc;
    }
    int rc = ensure_hmm_cap(c, n);
    if (rc) return rc;
    memcpy(c->h_hmms, hmms, (size_t)n * sizeof(psb_hmm_t));
    rc = eval_staged(c, n, senscr, best);
    if (rc) return rc;
    for (int i = 0; i < n; ++i) {           // keep the caller's ctx pointers
        void *ctx = hmms[i].ctx;
        hmms[i] = c->h_hmms[i];
        hmms[i].ctx = ctx;
    }
    return PSB_OK;
}

extern "C" int psb_hmm_vit_eval_ptrs(psb_hmmctx_t *c, psb_hmm_t *const *hmms, int32_t n, const int16_t *senscr,
                                     int32_t *best)
{
    PSB_REQUIRE(c && n >= 0 && (n == 0 || (hmms && senscr)), "psb_hmm_vit_eval_ptrs: bad argument");
    if (best) *best = PSB_WORST_SCORE;
    if (n == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(c->device));
    int rc = ensure_hmm_cap(c, n);
    if (rc) return rc;
    for (int i = 0; i < n; ++i) {
        PSB_REQUIRE(hmms[i], "hmms[%d] is null", i);
        rc = validate_hmm(c, hmms[i], i);
        if (rc) return rc;
        c->h_hmms[i] = *hmms[i];
    }
    rc = eval_staged(c, n, senscr, best);
    if (rc) return rc;
    for (int i = 0; i < n; ++i) {
        void *ctx = hmms[i]->ctx;
        *hmms[i] = c->h_hmms[i];
        hmms[i]->ctx = ctx;
    }
    return PSB_OK;
}

// ---------------------------------------------------------------------------------------

extern "C" int psb_phoneloop_create(psb_hmmctx_t *c, int32_t n_phones, const int32_t *ssid, const int32_t *tmatid,
                                    int32_t window, int32_t beam, int32_t pbeam, int32_t pip, double penalty_weight,
                                    psb_phoneloop_t **out)
{
    PSB_REQUIRE(c && out && n_phones > 0 && ssid && tmatid && window >= 0, "psb_phoneloop_create: bad argument");
    PSB_CUDA(cudaSetDevice(c->device));
    std::vector<uint16_t> sseq((size_t)c->n_sseq * c->n_emit);
    PSB_CUDA(cudaMemcpy(sseq.data(), c->d_sseq, sseq.size() * 2, cudaMemcpyDeviceToHost));
    std::vector<uint16_t> senid((size_t)c->n_emit * n_phones);
    for (int i = 0; i < n_phones; ++i) {
        PSB_REQUIRE(ssid[i] >= 0 && ssid[i] < c->n_sseq, "ssid[%d] out of range", i);
        PSB_REQUIRE(tmatid[i] >= 0 && tmatid[i] < c->n_tmat, "tmatid[%d] out of range", i);
        for (int s = 0; s < c->n_emit; ++s) {
            uint16_t v = sseq[(size_t)ssid[i] * c->n_emit + s];         // hmm_init, non-mpx (hmm.c:99-102)
            PSB_REQUIRE(v < c->n_sen, "senone id %d out of range", v);
            senid[(size_t)s * n_phones + i] = v;
        }
    }
    psb_phoneloop_t *p = new psb_phoneloop_t();
    memset(p, 0, sizeof(*p));
    p->c = c; p->n_phones = n_phones; p->window = window; p->beam = beam; p->pbeam = pbeam; p->pip = pip;
    p->penalty_weight = penalty_weight;
    cudaError_t e = cudaMalloc(&p->d_senid, senid.size() * 2);
    if (e == cudaSuccess) e = cudaMemcpy(p->d_senid, senid.data(), senid.size() * 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_tmatid, (size_t)n_phones * 4);
    if (e == cudaSuccess) e = cudaMemcpy(p->d_tmatid, tmatid, (size_t)n_phones * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_ssid, (size_t)n_phones * 4);
    if (e == cudaSuccess) e = cudaMemcpy(p->d_ssid, ssid, (size_t)n_phones * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_flags, 4);
    if (e == cudaSuccess) e = cudaMemset(p->d_flags, 0, 4);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        psb_set_error("psb_phoneloop_create: %s", cudaGetErrorString(e));
        psb_phoneloop_free(p);
        return PSB_ERR_CUDA;
    }
    *out = p;
    return PSB_OK;
}

extern "C" void psb_phoneloop_free(psb_phoneloop_t *p)
{
    if (!p) return;
    cudaSetDevice(p->c->device);
    if (p->stream) cudaStreamSynchronize(p->stream);
    cudaFree(p->d_senid); cudaFree(p->d_tmatid); cudaFree(p->d_ssid); cudaFree(p->d_flags);
    if (p->stream) cudaStreamDestroy(p->stream);
    delete p;
}

int psb_phoneloop_launch(psb_phoneloop_t *p, const int16_t *d_senscr, const int32_t *d_utt_off, int32_t n_utt,
                         int32_t *d_best, int32_t *d_pen, psb_hmm_t *d_final, psb_hmm_t *d_trace, cudaStream_t st)
{
    const int H = p->n_phones, N = p->c->n_emit;
    size_t smem = ((size_t)(2 * N + 4 + p->window) * H + 64) * sizeof(int);
    PSB_REQUIRE(smem <= 227 * 1024, "phone loop with %d HMMs needs %zu bytes of shared memory (max 227 KB)", H, smem);
    PSB_CUDA(cudaFuncSetAttribute(phoneloop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int threads = std::min(1024, roundup(H, 32));
    PlParams P;
    P.n_phones = H; P.window = p->window; P.beam = p->beam; P.pbeam = p->pbeam; P.pip = p->pip;
    P.penalty_weight = p->penalty_weight;
    phoneloop_kernel<<<n_utt, threads, smem, st>>>(d_senscr, d_utt_off, dev_ctx(p->c), P, p->d_senid, p->d_tmatid, p->d_ssid,
                                                   d_best, d_pen, d_final, d_trace, p->d_flags);
    PSB_LAUNCH_CHECK();
    return PSB_OK;
}

int psb_phoneloop_n_phones(const psb_phoneloop_t *p) { return p->n_phones; }

extern "C" int psb_phoneloop_run_device(psb_phoneloop_t *p, const int16_t *d_senscr, const int32_t *utt_off,
                                        int32_t n_utt, int32_t *d_best, int32_t *d_pen, psb_hmm_t *final_hmms,
                                        void *batch)
{
    PSB_REQUIRE(p && d_senscr && utt_off && n_utt >= 0, "psb_phoneloop_run_device: bad argument");
    if (n_utt == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(p->c->device));
    cudaStream_t st = batch ? psb_batch_stream((psb_batch_t *)batch) : p->stream;
    int32_t *d_off = nullptr;
    psb_hmm_t *d_final = nullptr;
    PSB_CUDA(cudaMalloc(&d_off, (size_t)(n_utt + 1) * 4));
    PSB_CUDA(cudaMemcpyAsync(d_off, utt_off, (size_t)(n_utt + 1) * 4, cudaMemcpyHostToDevice, st));
    if (final_hmms) PSB_CUDA(cudaMalloc(&d_final, (size_t)n_utt * p->n_phones * sizeof(psb_hmm_t)));
    int rc = psb_phoneloop_launch(p, d_senscr, d_off, n_utt, d_best, d_pen, d_final, nullptr, st);
    if (!rc && final_hmms) {
        cudaError_t e = cudaMemcpyAsync(final_hmms, d_final, (size_t)n_utt * p->n_phones * sizeof(psb_hmm_t),
                                        cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) { psb_set_error("%s", cudaGetErrorString(e)); rc = PSB_ERR_CUDA; }
    }
    cudaStreamSynchronize(st);
    cudaFree(d_off);
    cudaFree(d_final);
    return rc;
}

extern "C" int psb_phoneloop_run_host(psb_phoneloop_t *p, const int16_t *senscr, const int32_t *utt_off, int32_t n_utt,
                                      int32_t *best, int32_t *pen, psb_hmm_t *hmm_trace)
{
    PSB_REQUIRE(p && senscr && utt_off && n_utt >= 0, "psb_phoneloop_run_host: bad argument");
    if (n_utt == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(p->c->device));
    const size_t total = utt_off[n_utt], H = p->n_phones;
    int16_t *d_scr = nullptr; int32_t *d_off = nullptr, *d_best = nullptr, *d_pen = nullptr; psb_hmm_t *d_tr = nullptr;
    int rc = PSB_OK;
    cudaError_t e = cudaMalloc(&d_scr, std::max<size_t>(2, total * p->c->n_sen * 2));
    if (e == cudaSuccess) e = cudaMemcpy(d_scr, senscr, total * p->c->n_sen * 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&d_off, (size_t)(n_utt + 1) * 4);
    if (e == cudaSuccess) e = cudaMemcpy(d_off, utt_off, (size_t)(n_utt + 1) * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && best) e = cudaMalloc(&d_best, std::max<size_t>(4, total * 4));
    if (e == cudaSuccess && pen) e = cudaMalloc(&d_pen, std::max<size_t>(4, total * H * 4));
    if (e == cudaSuccess && hmm_trace) e = cudaMalloc(&d_tr, std::max<size_t>(4, total * H * sizeof(psb_hmm_t)));
    if (e == cudaSuccess) {
        rc = psb_phoneloop_launch(p, d_scr, d_off, n_utt, d_best, d_pen, nullptr, d_tr, p->stream);
        if (!rc) e = cudaStreamSynchronize(p->stream);
        if (!rc && e == cudaSuccess && best) e = cudaMemcpy(best, d_best, total * 4, cudaMemcpyDeviceToHost);
        if (!rc && e == cudaSuccess && pen) e = cudaMemcpy(pen, d_pen, total * H * 4, cudaMemcpyDeviceToHost);
        if (!rc && e == cudaSuccess && hmm_trace)
            e = cudaMemcpy(hmm_trace, d_tr, total * H * sizeof(psb_hmm_t), cudaMemcpyDeviceToHost);
    }
    if (e != cudaSuccess) { psb_set_error("psb_phoneloop_run_host: %s", cudaGetErrorString(e)); rc = PSB_ERR_CUDA; }
    cudaFree(d_scr); cudaFree(d_off); cudaFree(d_best); cudaFree(d_pen); cudaFree(d_tr);
    return rc;
}

// ---------------------------------------------------------------------------------------
// Device-resident HMM sets (SURVEY 8 b5 at the reference's real activity level, first brick of
// row f-1): what evaluate_channels (ngram_search_fwdtree.c:702-715), fsg_search_hmm_eval
// (fsg_search.c:336-408), phmm_eval_all (allphone_search.c:349) iterate over every frame --
// ~6 000 hmm_t per utterance on en-us -- kept in HBM between frames as a structure of arrays so
// that one frame is one coalesced streaming pass: 41 B read + 36 B written per 3-state instance
// (SURVEY 8d counts 74 B), against 176 B for the 88-byte hmm_t records themselves.  Instances are
// grouped in segments (one per utterance); every segment has its own senone-score row per frame
// and its own best score, like one decoder each.  Inside the set every segment is padded to a
// multiple of four instances so that a thread owns four neighbours and moves them with 128-bit
// (state) and 64-bit (ids) accesses; padding instances are inert (WORST_SCORE, senone 0) and
// never reach the best score.
constexpr int HS_V = 4;                     // instances per thread
constexpr int HS_TS = 512;                  // storage tile: [tile][field][HS_TS], so a CTA's fields are one contiguous block
constexpr int HS_THREADS = 128;             // threads per CTA of hmmset_eval_kernel: 112.7 us against 118.2 us at 256 per 6.08 M-instance frame

struct psb_hmmset_s {
    psb_hmmctx_t *c;
    int64_t n_max, n, pitch;
    int32_t n_seg_max, n_seg;
    int64_t max_seg_len;
    bool any_mpx;                 // some instance is multiplexed (hmm_t.mpx): the fused sweep leaves those to the per-frame kernel
    int32_t *d_i32;               // [pitch / HS_TS][2*NS + 4][HS_TS]: score[NS] hist[NS] out_score out_hist best frame
    uint16_t *d_u16;              // [pitch / HS_TS][NS + 2][HS_TS]: senid[NS] ssid tmatid(int16)
    uint8_t *d_mpx;               // [pitch]
    int64_t *d_seg_off;           // [n_seg_max + 1] caller's offsets (AoS order)
    int64_t *d_seg_base;          // [n_seg_max + 1] padded offsets inside the set
    psb_hmm_t *d_aos;             // staging for upload / download
    int32_t *d_snap_i32;          // psb_hmmset_snapshot: copy of the mutable state (scores, histories, exits)
    cudaStream_t stream, own_stream;
    cudaEvent_t ev[2];
};

namespace {

struct HmmSetDev {
    int32_t *i32;
    uint16_t *u16;
    uint8_t *mpx;
    const int64_t *seg_off, *seg_base;
    int64_t pitch;
    int n_seg;
};

static HmmSetDev dev_set(const psb_hmmset_t *s)
{
    HmmSetDev d;
    d.i32 = s->d_i32; d.u16 = s->d_u16; d.mpx = s->d_mpx; d.seg_off = s->d_seg_off; d.seg_base = s->d_seg_base;
    d.pitch = s->pitch; d.n_seg = s->n_seg;
    return d;
}

template <bool TO_SOA>
__global__ void __launch_bounds__(256)
hmmset_convert_kernel(psb_hmm_t *aos, HmmSetDev s, int64_t n, int ns)
{
    const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // index in the caller's array
    if (a >= n) return;
    int lo = 0, hi = s.n_seg;                                           // segment of a: seg_off[lo] <= a < seg_off[lo+1]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (s.seg_off[mid] <= a) lo = mid; else hi = mid;
    }
    const int64_t i = s.seg_base[lo] + (a - s.seg_off[lo]);
    psb_hmm_t *p = aos + a;
    const int64_t b32 = (i / HS_TS) * (int64_t)(2 * ns + 4) * HS_TS + (i % HS_TS);
    const int64_t b16 = (i / HS_TS) * (int64_t)(ns + 2) * HS_TS + (i % HS_TS);
    int32_t *score = s.i32 + b32, *hist = score + ns * HS_TS, *tail = score + 2 * ns * HS_TS;
    uint16_t *senid = s.u16 + b16, *ids = senid + ns * HS_TS;
    if (TO_SOA) {
        for (int k = 0; k < ns; ++k) {
            score[k * HS_TS] = p->score[k];
            hist[k * HS_TS] = p->history[k];
            senid[k * HS_TS] = p->senid[k];
        }
        tail[0] = p->out_score; tail[HS_TS] = p->out_history; tail[2 * HS_TS] = p->bestscore; tail[3 * HS_TS] = p->frame;
        ids[0] = p->ssid; ids[HS_TS] = (uint16_t)p->tmatid;
        s.mpx[i] = p->mpx;
    }
    else {
        for (int k = 0; k < PSB_HMM_MAX_NSTATE; ++k) {
            p->score[k] = k < ns ? score[k * HS_TS] : 0;
            p->history[k] = k < ns ? hist[k * HS_TS] : 0;
            p->senid[k] = k < ns ? senid[k * HS_TS] : 0;
        }
        p->out_score = tail[0]; p->out_history = tail[HS_TS]; p->bestscore = tail[2 * HS_TS]; p->frame = tail[3 * HS_TS];
        p->ssid = ids[0]; p->tmatid = (int16_t)ids[HS_TS];
        p->mpx = s.mpx[i]; p->n_emit_state = (uint8_t)ns;
        p->ctx = nullptr;
    }
}

__global__ void fill_i32_kernel(int32_t *p, int64_t n, int32_t v)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

__device__ __forceinline__ int comp(const int4 &v, int q) { return q == 0 ? v.x : q == 1 ? v.y : q == 2 ? v.z : v.w; }
__device__ __forceinline__ void setc(int4 &v, int q, int x)
{
    if (q == 0) v.x = x; else if (q == 1) v.y = x; else if (q == 2) v.z = x; else v.w = x;
}

// mbarrier + TMA bulk copy (global -> shared, completion counted in bytes on the barrier): used by both set kernels
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(dst)),
                 "l"(src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
                 : "memory");
}

// One hmm_vit_eval per instance, four instances per thread, one CTA row (blockIdx.y) per
// segment.  row0[seg] + t is the segment's senone-score row of this frame (staged in shared
// memory: the gathers of a tile hit ~3 x HS_TILE random int16 of it); segments with
// n_rows[seg] <= t are finished.  NS = 3 or 5 (0: any topology, runtime count).
template <int NS>
__global__ void __launch_bounds__(HS_THREADS, (NS == 3 ? 3 : 2) * (256 / HS_THREADS))
hmmset_eval_kernel(HmmSetDev s, HmmCtxDev c, const int16_t *__restrict__ senscr, const int64_t *__restrict__ row0,
                   const int32_t *__restrict__ n_rows, int t, int32_t *__restrict__ best_out)
{
    extern __shared__ __align__(16) int16_t srow[];         // [n_sen] + 16 bytes
    __shared__ int red[HS_THREADS / 32];
    const int seg = blockIdx.y;
    if (n_rows && t >= n_rows[seg]) return;
    const int64_t n = s.seg_off[seg + 1] - s.seg_off[seg];
    const int64_t j0 = ((int64_t)blockIdx.x * HS_THREADS + threadIdx.x) * HS_V;   // first of this thread's four
    if ((int64_t)blockIdx.x * HS_THREADS * HS_V >= n) return;
    // issue this thread's state loads first: they are in flight while the CTA stages the score row
    constexpr int NL = NS > 0 ? NS : PSB_HMM_MAX_NSTATE;
    const int ns = NS > 0 ? NS : c.n_emit;
    const bool live = j0 < n;
    const int64_t i = s.seg_base[seg] + (live ? j0 : 0);              // multiple of four
    const int64_t b32 = (i / HS_TS) * (int64_t)(2 * ns + 4) * HS_TS + (i % HS_TS);
    const int64_t b16 = (i / HS_TS) * (int64_t)(ns + 2) * HS_TS + (i % HS_TS);
    int32_t *score = s.i32 + b32, *hist = score + ns * HS_TS, *tail = score + 2 * ns * HS_TS;
    uint16_t *senid = s.u16 + b16;
    const uint16_t *ids = senid + ns * HS_TS;
    int4 sc[NL], hi[NL], osc, ohi, bst;
    uint2 sid[NL], tm = make_uint2(0u, 0u);
    uchar4 mp = make_uchar4(0, 0, 0, 0);
    if (live) {
#pragma unroll
        for (int k = 0; k < NL; ++k)
            if (k < ns) {
                sc[k] = __ldcs(reinterpret_cast<const int4 *>(score + k * HS_TS));
                hi[k] = __ldcs(reinterpret_cast<const int4 *>(hist + k * HS_TS));
                sid[k] = __ldcs(reinterpret_cast<const uint2 *>(senid + k * HS_TS));
            }
        osc = __ldcs(reinterpret_cast<const int4 *>(tail));
        ohi = __ldcs(reinterpret_cast<const int4 *>(tail + HS_TS));
        tm = __ldcs(reinterpret_cast<const uint2 *>(ids + HS_TS));
        mp = __ldcs(reinterpret_cast<const uchar4 *>(s.mpx + i));
    }
    // The segment's score row: its 16-byte aligned interior by ONE TMA bulk copy (issued by thread 0, completion on an
    // mbarrier, in flight together with the state loads above), the few bytes before and after it by plain loads -- nothing
    // outside the row is touched.  In shared memory the row keeps its alignment within 16 bytes.
    __shared__ __align__(8) uint64_t row_bar;
    const int16_t *srow_al;
    {
        const int16_t *row = senscr + (row0 ? row0[seg] + t : (int64_t)t * gridDim.y + seg) * c.n_sen;
        const uintptr_t a = reinterpret_cast<uintptr_t>(row);
        const unsigned mis = (unsigned)(a & 15), nbytes = (unsigned)c.n_sen * 2;
        unsigned head = (16 - mis) & 15;
        if (head > nbytes) head = nbytes;
        const unsigned body = (nbytes - head) & ~15u, tail = nbytes - head - body;
        unsigned char *dst = reinterpret_cast<unsigned char *>(srow) + mis;           // srow is 16-byte aligned
        if (threadIdx.x == 0) {
            mbar_init(&row_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            if (body) {
                mbar_expect_tx(&row_bar, body);
                tma_bulk_g2s(dst + head, reinterpret_cast<const unsigned char *>(row) + head, body, &row_bar);
            }
        }
        const unsigned hn = head >> 1, tn = tail >> 1;                                  // int16 elements (rows are 2-byte aligned)
        if (threadIdx.x < hn) reinterpret_cast<int16_t *>(dst)[threadIdx.x] = row[threadIdx.x];
        if (threadIdx.x >= 32 && threadIdx.x < 32 + tn)
            reinterpret_cast<int16_t *>(dst + head + body)[threadIdx.x - 32] = row[((head + body) >> 1) + threadIdx.x - 32];
        srow_al = reinterpret_cast<const int16_t *>(dst);
        __syncthreads();                                                                // barrier initialised, head / tail written
        if (body) mbar_wait(&row_bar, 0u);
    }
    int best = PSB_WORST_SCORE;
    if (live) {
        bool any_mpx = false;
#pragma unroll
        for (int q = 0; q < HS_V; ++q) {
            HmmReg h;
#pragma unroll
            for (int k = 0; k < PSB_HMM_MAX_NSTATE; ++k) {
                const bool in = k < NL && k < ns;
                h.score[k] = in ? comp(sc[k < NL ? k : 0], q) : PSB_WORST_SCORE;
                h.hist[k] = in ? comp(hi[k < NL ? k : 0], q) : -1;
                const unsigned w = (q < 2) ? sid[k < NL ? k : 0].x : sid[k < NL ? k : 0].y;
                h.senid[k] = in ? (int)((q & 1) ? (w >> 16) : (w & 0xffffu)) : PSB_BAD_SSID;
            }
            h.out_score = comp(osc, q);
            h.out_hist = comp(ohi, q);
            h.best = PSB_WORST_SCORE;                 // every hmm_step variant overwrites it
            const unsigned tw = (q < 2) ? tm.x : tm.y;
            const int tmatid = (int16_t)((q & 1) ? (tw >> 16) : (tw & 0xffffu));
            const bool mpx = (q == 0 ? mp.x : q == 1 ? mp.y : q == 2 ? mp.z : mp.w) != 0;
            const int b = hmm_step(h, c, tmatid, mpx, srow_al);
            if (j0 + q < n) best = max(best, b);
#pragma unroll
            for (int k = 0; k < NL; ++k)
                if (k < ns) {
                    setc(sc[k], q, h.score[k]);
                    setc(hi[k], q, h.hist[k]);
                    if (mpx) {
                        unsigned &w = (q < 2) ? sid[k].x : sid[k].y;
                        w = (q & 1) ? ((w & 0xffffu) | ((unsigned)h.senid[k] << 16)) : ((w & 0xffff0000u) | ((unsigned)h.senid[k] & 0xffffu));
                        any_mpx = true;
                    }
                }
            setc(osc, q, h.out_score);
            setc(ohi, q, h.out_hist);
            setc(bst, q, h.best);
        }
#pragma unroll
        for (int k = 0; k < NL; ++k)
            if (k < ns) {
                __stcs(reinterpret_cast<int4 *>(score + k * HS_TS), sc[k]);
                __stcs(reinterpret_cast<int4 *>(hist + k * HS_TS), hi[k]);
                if (any_mpx) __stcs(reinterpret_cast<uint2 *>(senid + k * HS_TS), sid[k]);
            }
        __stcs(reinterpret_cast<int4 *>(tail), osc);
        __stcs(reinterpret_cast<int4 *>(tail + HS_TS), ohi);
        __stcs(reinterpret_cast<int4 *>(tail + 2 * HS_TS), bst);
    }
    best = __reduce_max_sync(0xffffffffu, best);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x < 32) {
        int v = threadIdx.x < (HS_THREADS >> 5) ? red[threadIdx.x] : PSB_WORST_SCORE;
        v = __reduce_max_sync(0xffffffffu, v);
        if (threadIdx.x == 0) atomicMax(best_out + seg, v);
    }
}

// ---------------------------------------------------------------------------------------
// hmmset_sweep_kernel: the same step fused over frames.  hmmset_eval_kernel streams every
// instance's state through HBM once per frame (77 B per 3-state instance and frame: the step is
// HBM-bound and needs one launch per frame).  When nothing else has to see the state between
// frames -- evaluate_channels over a fixed active set, ngram_search_fwdtree.c:702-715 -- a CTA can
// keep its slice of a segment (THREADS x V instances) in REGISTERS for the whole utterance and
// only the segment's int16 score row of each frame has to arrive: 2 * n_sen bytes per frame,
// staged by the TMA unit (cp.async.bulk global -> shared, completion on an mbarrier) two frames
// ahead into a double buffer, so that the copy of frame t+2 overlaps the arithmetic of frames t
// and t+1.  One elected thread arms the barrier and issues the copy; everybody waits on the
// barrier's phase.  Bulk copies need 16-byte aligned source, destination and size: the copy
// starts at the row's address rounded down to 16 and ends at its end rounded up, the row is read
// at its offset inside the buffer; the matrix's LAST row is copied by the threads themselves so
// that nothing past the allocation is touched.  Per frame one block-wide max (REDUX + one
// shared-memory hop) and one atomicMax per CTA into best[t][segment].  Results are bit-identical
// to n_frames calls of hmmset_eval_kernel (tests/test_gpu_parity.py).
//
// BEAM: the same sweep with the beam pruning of prune_channels between frames (ngram_search_fwdtree.c:1130-1181 and the
// keep-or-hmm_clear decision of prune_nonroot_chan, :811, :823-827, :872-874, without the lexicon-tree transitions): an instance is active
// in frame f iff its frame field == f (as for the channels evaluate_channels walks); after frame f the segment's best
// score and number of evaluated instances are known to every CTA of the segment, the -maxhmmpf histogram (256 bins of
// (best - bestscore) / (-beam / 256), walked until more than maxhmmpf instances are covered) narrows the beam, survivors
// (bestscore BETTER_THAN best + dynamic beam) move to frame f + 1 and the others are hmm_clear'ed (hmm.c:181-196) and
// never evaluated again.  The CTAs of one segment form ONE thread-block cluster: every frame each CTA sends its
// (maximum, count) into every peer's shared memory with st.async, whose completion is counted on the PEER's mbarrier
// (8 bytes per peer; the peer waits on its own barrier: one distributed-shared-memory store latency per frame -- a
// barrier.cluster per frame, ~380 cycles plus an L1 flush, measured 2.9x slower); only the rare histogram frames take
// a barrier.cluster and read the peers' bins (ld.shared::cluster).  No global-memory round trip, no launch per frame.
__device__ __forceinline__ unsigned cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cluster_nctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned mapa_shared(const void *p, unsigned rank)
{
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"((unsigned)__cvta_generic_to_shared(p)), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_u32(unsigned addr, unsigned v) { asm volatile("st.shared::cluster.u32 [%0], %1;" :: "r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned ld_cluster_u32(unsigned addr) { unsigned v; asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v; }
// remote store that signals: 8 bytes into a peer's shared memory, completion counted on the PEER's mbarrier (the peer
// waits on its own barrier -- one DSMEM store latency, no cluster-wide barrier, no L1 flush)
__device__ __forceinline__ void st_async_v2(unsigned remote_addr, unsigned a, unsigned b, unsigned remote_bar)
{
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];"
                 :: "r"(remote_addr), "r"(a), "r"(b), "r"(remote_bar) : "memory");
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int NS, int V, int THREADS, bool BEAM>
__global__ void __launch_bounds__(THREADS)
hmmset_sweep_kernel(HmmSetDev s, HmmCtxDev c, const int16_t *__restrict__ senscr, long long rows_total,
                    const int64_t *__restrict__ row0, const int32_t *__restrict__ n_rows, int n_frames,
                    int32_t *__restrict__ best_out, int n_tmat, int buf_bytes, int frame0, int beam, int maxhmmpf,
                    int32_t *__restrict__ n_active_out)
{
    static_assert(!BEAM || THREADS == 256, "the histogram walk maps one bin to one thread");
    // score rows in flight: two for the plain sweep (its frame is longer than half a bulk copy's latency), six under the
    // beam, where a CTA whose instances have mostly left runs ahead of the copies (measured: no difference, the floor of
    // the pruned sweep is the per-frame exchange, DESIGN 4.19)
    constexpr int NBUF = BEAM ? 6 : 2;
    extern __shared__ __align__(128) unsigned char sw_smem[];       // [NBUF][buf_bytes] score rows, then the transition matrices
    __shared__ __align__(8) uint64_t full[NBUF];
    __shared__ int red[2][THREADS / 32];
    __shared__ int redc[BEAM ? 2 : 1][THREADS / 32];
    __shared__ __align__(8) int2 cl_slot[BEAM ? 2 : 1][16];                 // [parity][rank in the cluster] {maximum, count}, written by the peers
    __shared__ __align__(8) uint64_t xbar[2];                               // ... whose arrival these count
    __shared__ unsigned hist[BEAM ? 2 : 1][BEAM ? 256 : 1];
    __shared__ unsigned scan_w[8];
    __shared__ int found;
    const int seg = blockIdx.y, tid = threadIdx.x;
    const int64_t n = s.seg_off[seg + 1] - s.seg_off[seg];
    const int64_t j_base = (int64_t)blockIdx.x * THREADS * V;
    const bool cta_empty = j_base >= n;                   // BEAM: stays for the cluster's barriers
    if (!BEAM && cta_empty) return;
    int T = n_frames;
    if (n_rows) T = min(T, n_rows[seg]);
    if (T <= 0) return;                                   // uniform over the segment's CTAs
    const unsigned my_rank = BEAM ? cluster_ctarank() : 0u, n_rank = BEAM ? cluster_nctarank() : 1u;
    if (BEAM) {
        hist[0][tid] = 0u;
        hist[1][tid] = 0u;
        if (tid == 0) {
            mbar_init(&xbar[0], 1);
            mbar_init(&xbar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    uint8_t *tps = sw_smem + NBUF * (size_t)buf_bytes;
    for (int q = tid; q < n_tmat * NS * (NS + 1); q += THREADS) tps[q] = c.tp[q];

    // this thread's V instances (THREADS apart: neighbouring threads read neighbouring words)
    int sc[V][NS], hi[V][NS], sid[V][NS], osc[V], ohi[V], tmo[V];
    unsigned tpk[V][3];                                   // 3-state: the instance's 12 transition bytes in registers
    int32_t *p32[V];
    bool live[V], act[V], touched[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int64_t j = j_base + (int64_t)v * THREADS + tid;
        live[v] = j < n;
        const int64_t i = s.seg_base[seg] + (live[v] ? j : 0);
        const int64_t b32 = (i / HS_TS) * (int64_t)(2 * NS + 4) * HS_TS + (i % HS_TS);
        const int64_t b16 = (i / HS_TS) * (int64_t)(NS + 2) * HS_TS + (i % HS_TS);
        p32[v] = s.i32 + b32;
        const uint16_t *p16 = s.u16 + b16;
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            sc[v][k] = live[v] ? p32[v][k * HS_TS] : PSB_WORST_SCORE;
            hi[v][k] = live[v] ? p32[v][(NS + k) * HS_TS] : -1;
            sid[v][k] = live[v] ? p16[k * HS_TS] : 0;
        }
        osc[v] = live[v] ? p32[v][2 * NS * HS_TS] : PSB_WORST_SCORE;
        ohi[v] = live[v] ? p32[v][(2 * NS + 1) * HS_TS] : -1;
        tmo[v] = live[v] ? (int)(int16_t)p16[(NS + 1) * HS_TS] * NS * (NS + 1) : 0;
        act[v] = BEAM ? (live[v] && p32[v][(2 * NS + 3) * HS_TS] == frame0) : live[v];
        touched[v] = act[v];
    }
    __syncthreads();                                      // the transition matrices are staged
    if (NS == 3) {
#pragma unroll
        for (int v = 0; v < V; ++v)
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const uint8_t *t4 = tps + tmo[v] + 4 * q;
                tpk[v][q] = (unsigned)t4[0] | ((unsigned)t4[1] << 8) | ((unsigned)t4[2] << 16) | ((unsigned)t4[3] << 24);
            }
    }
    const int64_t r0 = row0 ? row0[seg] : seg;
    const int64_t rstep = row0 ? 1 : gridDim.y;
    const size_t row_bytes = (size_t)c.n_sen * 2;
    auto row_addr = [&](int t) { return reinterpret_cast<uintptr_t>(senscr + (size_t)(r0 + (int64_t)t * rstep) * c.n_sen); };
    auto tma_ok = [&](int t) { return r0 + (int64_t)t * rstep + 1 < rows_total; };
    if (BEAM) cluster_sync_all();                         // every peer runs (its shared memory may be written) and has zeroed its histograms
    auto issue = [&](int t) {                                         // one thread: arm the barrier, start the copy
        const uintptr_t a = row_addr(t), a16 = a & ~(uintptr_t)15;
        const unsigned bytes = (unsigned)(((a - a16) + row_bytes + 15) & ~(size_t)15);
        mbar_expect_tx(&full[t % NBUF], bytes);
        tma_bulk_g2s(sw_smem + (size_t)(t % NBUF) * buf_bytes, reinterpret_cast<const void *>(a16), bytes, &full[t % NBUF]);
    };
    if (tid == 0) {
        for (int q = 0; q < NBUF; ++q) mbar_init(&full[q], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0 && !cta_empty)
        for (int q = 0; q < NBUF && q < T; ++q)
            if (tma_ok(q)) issue(q);
    int best_final[V];
#pragma unroll
    for (int v = 0; v < V; ++v) best_final[v] = PSB_WORST_SCORE;

    for (int t = 0; t < T; ++t) {
        const int b = t & 1, rb = t % NBUF;
        unsigned char *buf = sw_smem + (size_t)rb * buf_bytes;
        const uintptr_t a = row_addr(t);
        const int16_t *srow;
        if (BEAM && cta_empty)
            srow = reinterpret_cast<const int16_t *>(buf);            // nothing to evaluate
        else if (tma_ok(t)) {
            mbar_wait(&full[rb], (unsigned)(t / NBUF) & 1u);
            srow = reinterpret_cast<const int16_t *>(buf + (a & 15));
        }
        else {                                                        // last row of the matrix: plain copy
            const int16_t *g = reinterpret_cast<const int16_t *>(a);
            int16_t *d = reinterpret_cast<int16_t *>(buf);
            for (int q = tid; q < c.n_sen; q += THREADS) d[q] = g[q];
            __syncthreads();
            srow = d;
        }
        int best = PSB_WORST_SCORE, cnt = 0;
#pragma unroll
        for (int v = 0; v < V; ++v) {
            if (BEAM && !act[v]) continue;
            ++cnt;
            HmmReg h;
            int obs[PSB_HMM_MAX_NSTATE];
#pragma unroll
            for (int k = 0; k < PSB_HMM_MAX_NSTATE; ++k) {
                h.score[k] = k < NS ? sc[v][k < NS ? k : 0] : PSB_WORST_SCORE;
                h.hist[k] = k < NS ? hi[v][k < NS ? k : 0] : -1;
                h.senid[k] = 0;
                obs[k] = k < NS ? -(int)srow[sid[v][k < NS ? k : 0]] : 0;
            }
            h.out_score = osc[v]; h.out_hist = ohi[v]; h.best = PSB_WORST_SCORE;
            int bb;
            if (NS == 3) {
                uint8_t tl[12];                                       // byte extracts from registers, no shared-memory reads
#pragma unroll
                for (int q = 0; q < 12; ++q) tl[q] = (uint8_t)(tpk[v][q >> 2] >> (8 * (q & 3)));
                bb = hmm_step_3st(h, tl, obs);
            }
            else
                bb = hmm_step_5st(h, tps + tmo[v], obs);
            if (live[v]) best = max(best, bb);
#pragma unroll
            for (int k = 0; k < NS; ++k) { sc[v][k] = h.score[k]; hi[v][k] = h.hist[k]; }
            osc[v] = h.out_score; ohi[v] = h.out_hist;
            best_final[v] = bb;
        }
        best = __reduce_max_sync(0xffffffffu, best);
        if (BEAM) cnt = __reduce_add_sync(0xffffffffu, cnt);
        if ((tid & 31) == 0) {
            red[b][tid >> 5] = best;
            if (BEAM) redc[b][tid >> 5] = cnt;
        }
        __syncthreads();                                              // buf[b] and red[b] are complete / free
        if (tid == 0 && t + NBUF < T && tma_ok(t + NBUF) && !cta_empty) issue(t + NBUF);
        if (tid < 32) {
            int v = tid < THREADS / 32 ? red[b][tid] : PSB_WORST_SCORE;
            v = __reduce_max_sync(0xffffffffu, v);
            if (!BEAM) {
                if (tid == 0) atomicMax(best_out + (size_t)t * gridDim.y + seg, v);
            }
            else {
                int cc = tid < THREADS / 32 ? redc[b][tid] : 0;
                cc = __reduce_add_sync(0xffffffffu, cc);
                if (tid == 0) mbar_expect_tx(&xbar[b], n_rank * 8u);  // this frame's n_rank messages (own included)
                if ((unsigned)tid < n_rank)                           // lane r tells peer r
                    st_async_v2(mapa_shared(&cl_slot[b][my_rank], (unsigned)tid), (unsigned)v, (unsigned)cc,
                                mapa_shared(&xbar[b], (unsigned)tid));
            }
        }
        if (BEAM) {
            // A(t): every CTA's maximum and count have arrived.  A peer can only send frame t + 2 into the same slots
            // after it has seen this CTA's frame t + 1 message, i.e. after every thread here is done with frame t's.
            mbar_wait(&xbar[b], (unsigned)(t >> 1) & 1u);
            int seg_best = PSB_WORST_SCORE, seg_cnt = 0;
            for (unsigned r = 0; r < n_rank; ++r) {
                const int2 m = cl_slot[b][r];
                seg_best = max(seg_best, m.x);
                seg_cnt += m.y;
            }
            if (my_rank == 0 && tid == 0) {
                best_out[(size_t)t * gridDim.y + seg] = seg_best;
                if (n_active_out) n_active_out[(size_t)t * gridDim.y + seg] = seg_cnt;
            }
            hist[b ^ 1][tid] = 0u;                                    // the peers finished with it before they sent frame t's message
            int dyn = beam;
            if (maxhmmpf >= 0 && seg_cnt > maxhmmpf) {                // uniform over the cluster
                const int bw = -beam / 256;
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (act[v]) {
                        int bin = (seg_best - best_final[v]) / bw;
                        bin = bin > 255 ? 255 : bin;
                        atomicAdd(&hist[b][bin], 1u);
                    }
                if (tid == 0) found = 256;
                cluster_sync_all();                                   // B(t): every CTA's histogram is complete
                unsigned tot = 0;
                for (unsigned r = 0; r < n_rank; ++r) tot += ld_cluster_u32(mapa_shared(&hist[b][tid], r));
                unsigned incl = tot;                                  // running count over the bins, bin = thread
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned y = __shfl_up_sync(0xffffffffu, incl, o);
                    if ((tid & 31) >= o) incl += y;
                }
                if ((tid & 31) == 31) scan_w[tid >> 5] = incl;
                __syncthreads();
                for (int w = 0; w < (tid >> 5); ++w) incl += scan_w[w];
                if (incl > (unsigned)maxhmmpf) atomicMin(&found, tid);
                __syncthreads();
                dyn = -(found * bw);
            }
            const int thresh = seg_best + dyn;
#pragma unroll
            for (int v = 0; v < V; ++v)
                if (act[v] && !(best_final[v] > thresh)) {            // hmm_clear
#pragma unroll
                    for (int k = 0; k < NS; ++k) { sc[v][k] = PSB_WORST_SCORE; hi[v][k] = -1; }
                    osc[v] = PSB_WORST_SCORE; ohi[v] = -1; best_final[v] = PSB_WORST_SCORE;
                    act[v] = false;
                }
        }
    }
    if (BEAM) cluster_sync_all();                         // nobody leaves while a peer may still read its histogram
#pragma unroll
    for (int v = 0; v < V; ++v) {
        if (!live[v] || !touched[v]) continue;            // BEAM: instances that were never active stay as they are
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            p32[v][k * HS_TS] = sc[v][k];
            p32[v][(NS + k) * HS_TS] = hi[v][k];
        }
        p32[v][2 * NS * HS_TS] = osc[v];
        p32[v][(2 * NS + 1) * HS_TS] = ohi[v];
        p32[v][(2 * NS + 2) * HS_TS] = best_final[v];
        if (BEAM) p32[v][(2 * NS + 3) * HS_TS] = act[v] ? frame0 + T : -1;
    }
}

}  // namespace

extern "C" void psb_hmmset_free(psb_hmmset_t *s)
{
    if (!s) return;
    cudaSetDevice(s->c->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    cudaFree(s->d_i32); cudaFree(s->d_u16); cudaFree(s->d_mpx); cudaFree(s->d_seg_off); cudaFree(s->d_seg_base); cudaFree(s->d_aos);
    cudaFree(s->d_snap_i32);
    if (s->ev[0]) cudaEventDestroy(s->ev[0]);
    if (s->ev[1]) cudaEventDestroy(s->ev[1]);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    delete s;
}

extern "C" int psb_hmmset_create(psb_hmmctx_t *c, int64_t n_max, int32_t n_seg_max, psb_hmmset_t **out)
{
    PSB_REQUIRE(c && out && n_max > 0 && n_seg_max > 0 && n_seg_max <= 65535, "psb_hmmset_create: bad argument");
    PSB_CUDA(cudaSetDevice(c->device));
    psb_hmmset_t *s = new psb_hmmset_t();
    s->c = c; s->n_max = n_max; s->n_seg_max = n_seg_max;
    s->pitch = ((n_max + (int64_t)(HS_V - 1) * n_seg_max + HS_TS - 1) / HS_TS) * HS_TS;   // every segment may pad up to 3
    const int ns = c->n_emit;
    cudaError_t e = cudaMalloc(&s->d_i32, (size_t)(2 * ns + 4) * s->pitch * 4);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_u16, (size_t)(ns + 2) * s->pitch * 2);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_mpx, (size_t)s->pitch);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_seg_off, (size_t)(n_seg_max + 1) * 8);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_seg_base, (size_t)(n_seg_max + 1) * 8);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking);
    s->stream = s->own_stream;
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev[0]);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev[1]);
    if (e != cudaSuccess) {
        psb_set_error("psb_hmmset_create: %s", cudaGetErrorString(e));
        psb_hmmset_free(s);
        return PSB_ERR_CUDA;
    }
    *out = s;
    return PSB_OK;
}

// Run the set's kernels on a batch's stream (behind the kernels that produce the scores it reads).
extern "C" int psb_hmmset_use_batch_stream(psb_hmmset_t *s, psb_batch_t *b)
{
    PSB_REQUIRE(s, "psb_hmmset_use_batch_stream: null set");
    PSB_CUDA(cudaStreamSynchronize(s->stream));
    s->stream = b ? psb_batch_stream(b) : s->own_stream;
    return PSB_OK;
}

// Keep / bring back a copy of the mutable state: the same starting instances for the next batch of
// utterances without another upload (mpx sets also change senone-sequence ids: not snapshotted).
extern "C" int psb_hmmset_snapshot(psb_hmmset_t *s)
{
    PSB_REQUIRE(s && !s->any_mpx, "psb_hmmset_snapshot: null set or multiplexed instances");
    PSB_CUDA(cudaSetDevice(s->c->device));
    const size_t nb = (size_t)(2 * s->c->n_emit + 4) * s->pitch * 4;
    if (!s->d_snap_i32) PSB_CUDA(cudaMalloc(&s->d_snap_i32, nb));
    PSB_CUDA(cudaMemcpyAsync(s->d_snap_i32, s->d_i32, nb, cudaMemcpyDeviceToDevice, s->stream));
    return PSB_OK;
}

extern "C" int psb_hmmset_restore(psb_hmmset_t *s)
{
    PSB_REQUIRE(s && s->d_snap_i32, "psb_hmmset_restore: no snapshot");
    PSB_CUDA(cudaSetDevice(s->c->device));
    PSB_CUDA(cudaMemcpyAsync(s->d_i32, s->d_snap_i32, (size_t)(2 * s->c->n_emit + 4) * s->pitch * 4, cudaMemcpyDeviceToDevice, s->stream));
    return PSB_OK;
}

static int hmmset_staging(psb_hmmset_t *s)
{
    if (!s->d_aos) PSB_CUDA(cudaMalloc(&s->d_aos, (size_t)s->n_max * sizeof(psb_hmm_t)));
    return PSB_OK;
}

extern "C" int psb_hmmset_upload(psb_hmmset_t *s, const psb_hmm_t *hmms, int64_t n, const int64_t *seg_off, int32_t n_seg)
{
    PSB_REQUIRE(s && n >= 0 && n <= s->n_max && n_seg > 0 && n_seg <= s->n_seg_max && seg_off && (n == 0 || hmms),
                "psb_hmmset_upload: bad argument");
    PSB_REQUIRE(seg_off[0] == 0 && seg_off[n_seg] == n, "psb_hmmset_upload: seg_off must run from 0 to n");
    PSB_CUDA(cudaSetDevice(s->c->device));
    int64_t mx = 0;
    std::vector<int64_t> base((size_t)n_seg + 1);
    base[0] = 0;
    // large segments start on a storage-tile boundary when the capacity allows it (then every CTA
    // reads and writes whole contiguous tiles); otherwise segments are only padded to HS_V
    for (int pass = 0; pass < 2; ++pass) {
        const int big = pass == 0 ? HS_TS : HS_V;
        for (int i = 0; i < n_seg; ++i) {
            PSB_REQUIRE(seg_off[i + 1] >= seg_off[i], "psb_hmmset_upload: seg_off not monotone at %d", i);
            const int64_t len = seg_off[i + 1] - seg_off[i];
            const int pad = len >= HS_TS ? big : HS_V;
            mx = std::max<int64_t>(mx, len);
            base[(size_t)i + 1] = base[(size_t)i] + (len + pad - 1) / pad * pad;
        }
        if (base[(size_t)n_seg] <= s->pitch) break;
    }
    PSB_REQUIRE(base[(size_t)n_seg] <= s->pitch, "psb_hmmset_upload: internal capacity exceeded");
    s->any_mpx = false;
    for (int64_t i = 0; i < n; ++i) {
        int rc = validate_hmm(s->c, &hmms[i], (int)i);
        if (rc) return rc;
        s->any_mpx |= hmms[i].mpx != 0;
    }
    int rc = hmmset_staging(s);
    if (rc) return rc;
    s->n = n; s->n_seg = n_seg; s->max_seg_len = mx;
    PSB_CUDA(cudaMemcpyAsync(s->d_seg_off, seg_off, (size_t)(n_seg + 1) * 8, cudaMemcpyHostToDevice, s->stream));
    PSB_CUDA(cudaMemcpyAsync(s->d_seg_base, base.data(), (size_t)(n_seg + 1) * 8, cudaMemcpyHostToDevice, s->stream));
    // inert padding: WORST_SCORE everywhere, senone / transition matrix 0, not multiplexed
    const int ns = s->c->n_emit;
    const int64_t ni = (int64_t)(2 * ns + 4) * s->pitch;
    fill_i32_kernel<<<(unsigned)((ni + 255) / 256), 256, 0, s->stream>>>(s->d_i32, ni, PSB_WORST_SCORE);
    PSB_LAUNCH_CHECK();
    PSB_CUDA(cudaMemsetAsync(s->d_u16, 0, (size_t)(ns + 2) * s->pitch * 2, s->stream));
    PSB_CUDA(cudaMemsetAsync(s->d_mpx, 0, (size_t)s->pitch, s->stream));
    if (n) {
        PSB_CUDA(cudaMemcpyAsync(s->d_aos, hmms, (size_t)n * sizeof(psb_hmm_t), cudaMemcpyHostToDevice, s->stream));
        hmmset_convert_kernel<true><<<(unsigned)((n + 255) / 256), 256, 0, s->stream>>>(s->d_aos, dev_set(s), n, ns);
        PSB_LAUNCH_CHECK();
    }
    PSB_CUDA(cudaStreamSynchronize(s->stream));
    return PSB_OK;
}

extern "C" int psb_hmmset_download(psb_hmmset_t *s, psb_hmm_t *hmms)
{
    PSB_REQUIRE(s && (s->n == 0 || hmms), "psb_hmmset_download: bad argument");
    if (s->n == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(s->c->device));
    int rc = hmmset_staging(s);
    if (rc) return rc;
    hmmset_convert_kernel<false><<<(unsigned)((s->n + 255) / 256), 256, 0, s->stream>>>(s->d_aos, dev_set(s), s->n, s->c->n_emit);
    PSB_LAUNCH_CHECK();
    std::vector<psb_hmm_t> tmp((size_t)s->n);
    PSB_CUDA(cudaMemcpyAsync(tmp.data(), s->d_aos, (size_t)s->n * sizeof(psb_hmm_t), cudaMemcpyDeviceToHost, s->stream));
    PSB_CUDA(cudaStreamSynchronize(s->stream));
    for (int64_t i = 0; i < s->n; ++i) {        // keep the caller's ctx pointers
        void *ctx = hmms[i].ctx;
        hmms[i] = tmp[(size_t)i];
        hmms[i].ctx = ctx;
    }
    return PSB_OK;
}

extern "C" int psb_hmmset_eval_frames_device(psb_hmmset_t *s, const int16_t *d_senscr, const int64_t *d_row0,
                                             const int32_t *d_n_rows, int32_t n_frames, int32_t *d_best, float *ms)
{
    PSB_REQUIRE(s && d_senscr && d_best && n_frames >= 0, "psb_hmmset_eval_frames_device: bad argument");
    if (ms) *ms = 0.f;
    if (n_frames == 0 || s->n_seg == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(s->c->device));
    const int64_t nb = (int64_t)n_frames * s->n_seg;
    fill_i32_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, s->stream>>>(d_best, nb, PSB_WORST_SCORE);
    PSB_LAUNCH_CHECK();
    if (s->n == 0) {
        PSB_CUDA(cudaStreamSynchronize(s->stream));
        return PSB_OK;
    }
    const int tile = HS_THREADS * HS_V;
    const dim3 grid((unsigned)((s->max_seg_len + tile - 1) / tile), (unsigned)s->n_seg);
    const HmmSetDev sd = dev_set(s);
    const HmmCtxDev cd = dev_ctx(s->c);
    const size_t smem = (((size_t)cd.n_sen * 2 + 15) & ~(size_t)15) + 16;      // the row keeps its alignment within 16 bytes
    PSB_REQUIRE(smem <= 200 * 1024, "psb_hmmset: %d senones do not fit the shared-memory score row", cd.n_sen);
    auto launch = [&](auto kern, int t, int32_t *best) {
        kern<<<grid, HS_THREADS, smem, s->stream>>>(sd, cd, d_senscr, d_row0, d_n_rows, t, best);
    };
#define PSB_HS_ATTR(NS) PSB_CUDA(cudaFuncSetAttribute(hmmset_eval_kernel<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem))
    if (smem > 48 * 1024) {
        PSB_HS_ATTR(3); PSB_HS_ATTR(5); PSB_HS_ATTR(0);
    }
#undef PSB_HS_ATTR
    PSB_CUDA(cudaEventRecord(s->ev[0], s->stream));
    for (int t = 0; t < n_frames; ++t) {
        int32_t *best = d_best + (size_t)t * s->n_seg;
        if (cd.n_emit == 3) launch(hmmset_eval_kernel<3>, t, best);
        else if (cd.n_emit == 5) launch(hmmset_eval_kernel<5>, t, best);
        else launch(hmmset_eval_kernel<0>, t, best);
        PSB_LAUNCH_CHECK();
    }
    PSB_CUDA(cudaEventRecord(s->ev[1], s->stream));
    PSB_CUDA(cudaStreamSynchronize(s->stream));
    if (ms) PSB_CUDA(cudaEventElapsedTime(ms, s->ev[0], s->ev[1]));
    return PSB_OK;
}

extern "C" int psb_hmmset_sweep_device(psb_hmmset_t *s, const int16_t *d_senscr, int64_t rows_total, const int64_t *d_row0,
                                       const int32_t *d_n_rows, int32_t n_frames, int32_t *d_best, float *ms)
{
    PSB_REQUIRE(s && d_senscr && d_best && n_frames >= 0 && rows_total > 0, "psb_hmmset_sweep_device: bad argument");
    const HmmCtxDev cd = dev_ctx(s->c);
    if (s->any_mpx || (cd.n_emit != 3 && cd.n_emit != 5) || (cd.n_sen & 1))
        return psb_hmmset_eval_frames_device(s, d_senscr, d_row0, d_n_rows, n_frames, d_best, ms);   // per-frame launches
    if (ms) *ms = 0.f;
    if (n_frames == 0 || s->n_seg == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(s->c->device));
    const int64_t nb = (int64_t)n_frames * s->n_seg;
    fill_i32_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, s->stream>>>(d_best, nb, PSB_WORST_SCORE);
    PSB_LAUNCH_CHECK();
    if (s->n == 0) {
        if (ms) PSB_CUDA(cudaStreamSynchronize(s->stream));
        return PSB_OK;
    }
    const int buf_bytes = (int)(((size_t)cd.n_sen * 2 + 32 + 127) & ~(size_t)127);
    const int tp_bytes = s->c->n_tmat * cd.n_emit * (cd.n_emit + 1);
    const size_t smem = 2 * (size_t)buf_bytes + tp_bytes;
    PSB_REQUIRE(smem <= 200 * 1024, "psb_hmmset_sweep: %d senones / %d transition matrices do not fit shared memory", cd.n_sen, s->c->n_tmat);
    const HmmSetDev sd = dev_set(s);
    PSB_CUDA(cudaEventRecord(s->ev[0], s->stream));
#define PSB_SWEEP(NS, V, THREADS)                                                                                               \
    do {                                                                                                                       \
        auto kern = hmmset_sweep_kernel<NS, V, THREADS, false>;                                                                \
        PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                          \
        const dim3 grid((unsigned)((s->max_seg_len + THREADS * V - 1) / (THREADS * V)), (unsigned)s->n_seg);                   \
        kern<<<grid, THREADS, smem, s->stream>>>(sd, cd, d_senscr, (long long)rows_total, d_row0, d_n_rows, n_frames, d_best,  \
                                                s->c->n_tmat, buf_bytes, 0, 0, -1, nullptr);                                   \
    } while (0)
    // CTA shape: 256 threads x 4 instances per thread
    if (cd.n_emit == 3) PSB_SWEEP(3, 4, 256);
    else PSB_SWEEP(5, 4, 256);
#undef PSB_SWEEP
    PSB_LAUNCH_CHECK();
    PSB_CUDA(cudaEventRecord(s->ev[1], s->stream));
    if (ms) {                                               // ms == NULL: asynchronous on the set's stream
        PSB_CUDA(cudaStreamSynchronize(s->stream));
        PSB_CUDA(cudaEventElapsedTime(ms, s->ev[0], s->ev[1]));
    }
    return PSB_OK;
}

// The fused sweep with beam pruning between frames: one thread-block cluster per segment (hmmset_sweep_kernel<.., BEAM>).
extern "C" int psb_hmmset_sweep_beam_device(psb_hmmset_t *s, const int16_t *d_senscr, int64_t rows_total, const int64_t *d_row0,
                                            const int32_t *d_n_rows, int32_t n_frames, int32_t frame0, int32_t beam,
                                            int32_t maxhmmpf, int32_t *d_best, int32_t *d_n_active, float *ms)
{
    PSB_REQUIRE(s && d_senscr && d_best && n_frames >= 0 && rows_total > 0, "psb_hmmset_sweep_beam_device: bad argument");
    PSB_REQUIRE(beam < 0 && beam > -0x20000000, "psb_hmmset_sweep_beam_device: the beam is a negative log score (got %d)", beam);
    PSB_REQUIRE(maxhmmpf < 0 || beam <= -256, "psb_hmmset_sweep_beam_device: -maxhmmpf needs a beam of at least 256 score units (bin width -beam/256)");
    const HmmCtxDev cd = dev_ctx(s->c);
    PSB_REQUIRE(!s->any_mpx && (cd.n_emit == 3 || cd.n_emit == 5) && !(cd.n_sen & 1),
                "psb_hmmset_sweep_beam_device: plain 3- or 5-state instances and an even senone count (the fused kernel's shapes)");
    constexpr int THREADS = 256, V = 4;
    const int64_t per_seg = (s->max_seg_len + THREADS * V - 1) / (THREADS * V);
    PSB_REQUIRE(per_seg <= 16, "psb_hmmset_sweep_beam_device: a segment of %lld instances needs %lld CTAs, a cluster holds 16",
                (long long)s->max_seg_len, (long long)per_seg);
    if (ms) *ms = 0.f;
    if (n_frames == 0 || s->n_seg == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(s->c->device));
    const int64_t nb = (int64_t)n_frames * s->n_seg;
    fill_i32_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, s->stream>>>(d_best, nb, PSB_WORST_SCORE);
    PSB_LAUNCH_CHECK();
    if (d_n_active) PSB_CUDA(cudaMemsetAsync(d_n_active, 0, (size_t)nb * 4, s->stream));
    if (s->n == 0) {
        if (ms) PSB_CUDA(cudaStreamSynchronize(s->stream));
        return PSB_OK;
    }
    const int buf_bytes = (int)(((size_t)cd.n_sen * 2 + 32 + 127) & ~(size_t)127);
    const int tp_bytes = s->c->n_tmat * cd.n_emit * (cd.n_emit + 1);
    const size_t smem = 6 * (size_t)buf_bytes + tp_bytes;                 // NBUF of the BEAM instantiation
    PSB_REQUIRE(smem <= 200 * 1024, "psb_hmmset_sweep_beam: %d senones / %d transition matrices do not fit shared memory", cd.n_sen, s->c->n_tmat);
    const HmmSetDev sd = dev_set(s);
    const long long rows_ll = rows_total;
    const int n_tmat = s->c->n_tmat;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)std::max<int64_t>(per_seg, 1), (unsigned)s->n_seg);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cfg.gridDim.x; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    PSB_CUDA(cudaEventRecord(s->ev[0], s->stream));
#define PSB_SWEEPB(NS)                                                                                                         \
    do {                                                                                                                       \
        auto kern = hmmset_sweep_kernel<NS, V, THREADS, true>;                                                                 \
        PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                          \
        if (cfg.gridDim.x > 8) PSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));       \
        int n_clusters = 0;                                                                                                    \
        PSB_CUDA(cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg));                                                     \
        PSB_REQUIRE(n_clusters > 0, "psb_hmmset_sweep_beam: a cluster of %u CTAs with %zu bytes of shared memory each does not fit the device", \
                    cfg.gridDim.x, smem);                                                                                      \
        PSB_CUDA(cudaLaunchKernelEx(&cfg, kern, sd, cd, d_senscr, rows_ll, d_row0, d_n_rows, (int)n_frames, d_best, n_tmat,   \
                                    buf_bytes, (int)frame0, (int)beam, (int)maxhmmpf, d_n_active));                            \
        PSB_LAUNCH_CHECK();                                                                                                    \
    } while (0)
    if (cd.n_emit == 3) PSB_SWEEPB(3);
    else PSB_SWEEPB(5);
#undef PSB_SWEEPB
    PSB_CUDA(cudaEventRecord(s->ev[1], s->stream));
    if (ms) {
        PSB_CUDA(cudaStreamSynchronize(s->stream));
        PSB_CUDA(cudaEventElapsedTime(ms, s->ev[0], s->ev[1]));
    }
    return PSB_OK;
}

extern "C" int psb_hmmset_eval_host(psb_hmmset_t *s, const int16_t *senscr, int32_t *best)
{
    // one frame, host rows [n_seg][n_sen] in, host best[n_seg] out (tests and small callers)
    PSB_REQUIRE(s && senscr && best, "psb_hmmset_eval_host: bad argument");
    PSB_CUDA(cudaSetDevice(s->c->device));
    int16_t *d_scr = nullptr;
    int32_t *d_best = nullptr;
    const size_t nb = (size_t)s->n_seg * s->c->n_sen * 2;
    PSB_CUDA(cudaMalloc(&d_scr, nb));
    cudaError_t e = cudaMalloc(&d_best, (size_t)s->n_seg * 4);
    if (e == cudaSuccess) e = cudaMemcpy(d_scr, senscr, nb, cudaMemcpyHostToDevice);
    int rc = PSB_OK;
    if (e == cudaSuccess) {
        rc = psb_hmmset_eval_frames_device(s, d_scr, nullptr, nullptr, 1, d_best, nullptr);
        if (!rc) e = cudaMemcpy(best, d_best, (size_t)s->n_seg * 4, cudaMemcpyDeviceToHost);
    }
    cudaFree(d_scr); cudaFree(d_best);
    if (e != cudaSuccess) {
        psb_set_error("psb_hmmset_eval_host: %s", cudaGetErrorString(e));
        return PSB_ERR_CUDA;
    }
    return rc;
}

// ---------------------------------------------------------------------------------------
// Forced alignment: state_align_search.c on the device for whole batches (SURVEY 8 row b5 lists
// its evaluate_hmms, state_align_search.c:65).  One CTA per utterance, the utterance's phone
// chain in shared memory (SoA), time is the loop inside the kernel: renormalise (:199-203),
// evaluate_hmms (:64-86), prune_hmms (:88-107), phone_transition (:109-136, a left-to-right
// scan whose hmm_enter can cascade through not-yet-active successors: one warp resolves it as a
// carry chain, see below), record_transitions (:153-182) into a token table in HBM, and at the end
// the backtrace of state_align_search_finish (:221-279).
namespace {

__global__ void __launch_bounds__(128)
align_kernel(const int16_t *__restrict__ senscr, const int32_t *__restrict__ utt_off, HmmCtxDev c,
             const int32_t *__restrict__ ph_off, const uint16_t *__restrict__ senid_g,
             const int32_t *__restrict__ tmatid_g, const int32_t *__restrict__ sf_g, const int32_t *__restrict__ ef_g,
             int32_t *__restrict__ tok_id, int32_t *__restrict__ tok_sc, const int64_t *__restrict__ tok_off,
             int32_t *__restrict__ st_start, int32_t *__restrict__ st_dur, int32_t *__restrict__ st_score,
             int32_t *__restrict__ status)
{
    extern __shared__ int sm[];
    const int u = blockIdx.x, tid = threadIdx.x, N = c.n_emit;
    const int p0 = ph_off[u], H = ph_off[u + 1] - p0;
    const long long f0 = utt_off[u];
    const int T = utt_off[u + 1] - utt_off[u];
    const int n_st = H * N;
    int *score = sm;                       // [N][H]
    int *hist = score + N * H;             // [N][H]
    int *out_score = hist + N * H;         // [H]
    int *out_hist = out_score + H;         // [H]
    int *frame = out_hist + H;             // [H]
    int *sval = frame + H;                 // [32]
    int *sidx = sval + 32;                 // [32]
    int32_t *tid_u = tok_id + tok_off[u], *tsc_u = tok_sc + tok_off[u];
    int32_t *ss = st_start + (size_t)p0 * N, *sd = st_dur + (size_t)p0 * N, *sc = st_score + (size_t)p0 * N;

    for (int i = tid; i < n_st; i += blockDim.x) { ss[i] = -1; sd[i] = -1; sc[i] = -1; }
    if (H == 0) { if (tid == 0) status[u] = -1; return; }
    // hmm_init -> hmm_clear (hmm.c:85-105, 180-196), then state_align_search_start: hmm_enter(hmms, 0, 0, 0)
    for (int i = tid; i < H; i += blockDim.x) {
        for (int s = 0; s < N; ++s) { score[s * H + i] = PSB_WORST_SCORE; hist[s * H + i] = -1; }
        out_score[i] = PSB_WORST_SCORE; out_hist[i] = -1; frame[i] = -1;
    }
    __syncthreads();
    if (tid == 0) { score[0] = 0; hist[0] = 0; frame[0] = 0; }
    int best_score = 0;
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        const int16_t *row = senscr + (f0 + t) * c.n_sen;
        const int nf = t + 1;
        const bool renorm = best_score - 0x300000 < PSB_WORST_SCORE;
        int bs = PSB_WORST_SCORE;
        for (int i = tid; i < H; i += blockDim.x) {
            HmmReg h;
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s) {
                h.score[s] = s < N ? score[s * H + i] : PSB_WORST_SCORE;
                h.hist[s] = s < N ? hist[s * H + i] : -1;
                h.senid[s] = s < N ? senid_g[(size_t)(p0 + i) * N + s] : PSB_BAD_SSID;
            }
            h.out_score = out_score[i]; h.out_hist = out_hist[i]; h.best = PSB_WORST_SCORE;
            if (renorm) {                                    // hmm_normalize, every phone
#pragma unroll
                for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s)
                    if (s < N && h.score[s] > PSB_WORST_SCORE) h.score[s] -= best_score;
                if (h.out_score > PSB_WORST_SCORE) h.out_score -= best_score;
            }
            if (frame[i] >= t) {
                const int b = hmm_step(h, c, tmatid_g[p0 + i], false, row);
                if (b > bs) bs = b;
            }
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s)
                if (s < N) { score[s * H + i] = h.score[s]; hist[s * H + i] = h.hist[s]; }
            out_score[i] = h.out_score; out_hist[i] = h.out_hist;
            // prune_hmms: stays active unless the alignment constraint ends it
            if (frame[i] >= t && !(nf > (ef_g ? ef_g[p0 + i] : INT_MAX))) frame[i] = nf;
        }
        int dummy;
        bs = block_reduce_max_pair<int>(bs, 0, sidx, sval, dummy);      // (contains the barriers)
        best_score = bs;
        __syncthreads();
        // phone_transition.  Reference order: for i = 0..H-2, if phone i is active in nf (by pruning
        // OR because iteration i-1 just entered it) and the window of phone i+1 is open and
        // (phone i+1 is idle or out_score[i] beats its state-0 score): hmm_enter(i+1).  With
        //   P[i] = frame[i] == nf after pruning,  G[j] = window(j) && (idle(j) || out[j-1] > score0[j])
        // (G reads nothing an earlier iteration writes), "active" is A[i] = P[i] | (G[i] & A[i-1]):
        // a carry chain.  One warp resolves 32 phones per step with a 64-bit add
        // (generate = P, propagate = G & ~P), the carry links the steps; E[j] = A[j-1] & G[j].
        if (tid < 32) {
            unsigned carry = 0u;
            for (int base = 0; base < H; base += 32) {
                const int j = base + tid;
                const bool in = j < H;
                const bool P = in && frame[j] == nf;
                const bool G = in && j >= 1 && nf >= (sf_g ? sf_g[p0 + j] : 0) &&
                               (frame[j] < t || out_score[j - 1] > score[j]);
                const unsigned g = __ballot_sync(0xffffffffu, P);
                const unsigned pp = __ballot_sync(0xffffffffu, G) & ~g;
                const unsigned long long x = (unsigned long long)(g | pp), y = (unsigned long long)g;
                const unsigned long long cin = (x + y + carry) ^ x ^ y;  // bit k = A[base + k - 1]
                if (G && ((cin >> tid) & 1ull)) {                        // hmm_enter(phone j, out_score[j-1], out_hist[j-1], nf)
                    score[j] = out_score[j - 1]; hist[j] = out_hist[j - 1]; frame[j] = nf;
                }
                carry = (unsigned)(cin >> 32) & 1u;
                __syncwarp();
            }
        }
        __syncthreads();
        // record_transitions
        int32_t *ti = tid_u + (size_t)t * n_st, *ts = tsc_u + (size_t)t * n_st;
        for (int i = tid; i < H; i += blockDim.x) {
            const bool on = frame[i] >= t;
            for (int s = 0; s < N; ++s) {
                const int idx = i * N + s;
                ti[idx] = on ? hist[s * H + i] : -1;
                ts[idx] = on ? score[s * H + i] : -1;
                if (on) hist[s * H + i] = idx;
            }
        }
        __syncthreads();
    }
    // state_align_search_finish
    if (tid == 0) {
        int rc = 0;
        int last_id = out_hist[H - 1], last_sc = out_score[H - 1], cur_id = last_id, cur_sc;
        if (last_id == -1 || T == 0) rc = -1;
        else {
            int last_frame = T;
            for (int cf = T - 2; cf >= 0; --cf) {
                const int prev = cur_id;
                cur_id = tid_u[(size_t)cf * n_st + prev];
                cur_sc = tsc_u[(size_t)cf * n_st + prev];
                if (cur_id == -1) { rc = -2 - cf; break; }
                if (cur_id != last_id) {
                    ss[last_id] = cf + 1;
                    sd[last_id] = last_frame - (cf + 1);
                    sc[last_id] = last_sc - cur_sc;
                    last_id = cur_id; last_sc = cur_sc;
                    last_frame = cf + 1;
                }
            }
            if (rc == 0) { ss[0] = 0; sd[0] = last_frame; sc[0] = 0; }
        }
        status[u] = rc;
    }
}

}  // namespace

extern "C" int psb_align_batch_device(psb_hmmctx_t *c, const int16_t *d_senscr, const int32_t *utt_off, int32_t n_utt,
                                      const int32_t *ph_off, const int32_t *ssid, const int32_t *tmatid,
                                      const int32_t *sf, const int32_t *ef,
                                      int32_t *st_start, int32_t *st_dur, int32_t *st_score, int32_t *status)
{
    PSB_REQUIRE(c && utt_off && ph_off && n_utt >= 0 && st_start && st_dur && st_score && status,
                "psb_align_batch_device: bad argument");
    if (n_utt == 0) return PSB_OK;
    PSB_REQUIRE(utt_off[0] == 0 && ph_off[0] == 0, "psb_align_batch_device: offsets must start at 0");
    const int N = c->n_emit;
    const int total_ph = ph_off[n_utt];
    PSB_REQUIRE(total_ph == 0 || (ssid && tmatid), "psb_align_batch_device: phones missing");
    PSB_REQUIRE(d_senscr || utt_off[n_utt] == 0, "psb_align_batch_device: scores missing");
    PSB_CUDA(cudaSetDevice(c->device));
    std::vector<uint16_t> sseq((size_t)c->n_sseq * N);
    PSB_CUDA(cudaMemcpy(sseq.data(), c->d_sseq, sseq.size() * 2, cudaMemcpyDeviceToHost));
    std::vector<uint16_t> senid((size_t)std::max(total_ph, 1) * N);
    std::vector<int64_t> tok_off((size_t)n_utt + 1);
    int max_h = 0;
    tok_off[0] = 0;
    for (int u = 0; u < n_utt; ++u) {
        const int H = ph_off[u + 1] - ph_off[u], T = utt_off[u + 1] - utt_off[u];
        PSB_REQUIRE(H >= 0 && T >= 0, "psb_align_batch_device: offsets not monotone at %d", u);
        max_h = std::max(max_h, H);
        tok_off[(size_t)u + 1] = tok_off[(size_t)u] + (int64_t)T * H * N;
    }
    for (int i = 0; i < total_ph; ++i) {
        PSB_REQUIRE(ssid[i] >= 0 && ssid[i] < c->n_sseq, "ssid[%d] out of range", i);
        PSB_REQUIRE(tmatid[i] >= 0 && tmatid[i] < c->n_tmat, "tmatid[%d] out of range", i);
        for (int s = 0; s < N; ++s) {
            const uint16_t v = sseq[(size_t)ssid[i] * N + s];           // hmm_init, non-mpx (hmm.c:99-102)
            PSB_REQUIRE(v < c->n_sen, "senone id %d out of range", v);
            senid[(size_t)i * N + s] = v;
        }
    }
    const size_t smem = ((size_t)(2 * N + 3) * max_h + 64) * sizeof(int);
    PSB_REQUIRE(smem <= 200 * 1024, "psb_align_batch_device: %d phones in one utterance do not fit shared memory", max_h);
    // grow-only workspace in the context: one int32 block
    //   utt_off | ph_off | tmatid | sf | ef | start | dur | score | status
    // plus the token table (2 x frames x states), the senone ids and the token offsets
    const size_t n_state = (size_t)total_ph * N;
    const size_t o_utt = 0, o_ph = o_utt + n_utt + 1, o_tm = o_ph + n_utt + 1, o_sf = o_tm + total_ph, o_ef = o_sf + total_ph,
                 o_ss = o_ef + total_ph, o_sd = o_ss + n_state, o_sc = o_sd + n_state, o_st = o_sc + n_state,
                 n_i32 = o_st + n_utt;
    const size_t n_tok = (size_t)tok_off[(size_t)n_utt] * 2;
    auto grow = [](void **p, size_t *cap, size_t need, size_t elem) -> cudaError_t {
        if (need <= *cap) return cudaSuccess;
        if (*p) cudaFree(*p);
        *p = nullptr; *cap = 0;
        const size_t want = need + need / 8 + 256;
        cudaError_t e = cudaMalloc(p, want * elem);
        if (e == cudaSuccess) *cap = want;
        return e;
    };
    cudaError_t e = grow((void **)&c->d_al_i32, &c->al_i32_cap, n_i32, 4);
    if (e == cudaSuccess) e = grow((void **)&c->d_al_tok, &c->al_tok_cap, std::max<size_t>(n_tok, 1), 4);
    if (e == cudaSuccess) e = grow((void **)&c->d_al_senid, &c->al_senid_cap, senid.size(), 2);
    if (e == cudaSuccess) e = grow((void **)&c->d_al_tokoff, &c->al_tokoff_cap, tok_off.size(), 8);
    if (e == cudaSuccess && !c->al_ev[0]) e = cudaEventCreate(&c->al_ev[0]);
    if (e == cudaSuccess && !c->al_ev[1]) e = cudaEventCreate(&c->al_ev[1]);
    int32_t *d_i32 = c->d_al_i32, *d_tok = c->d_al_tok;
    cudaStream_t st = c->stream;
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_i32 + o_utt, utt_off, ((size_t)n_utt + 1) * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_i32 + o_ph, ph_off, ((size_t)n_utt + 1) * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && total_ph) e = cudaMemcpyAsync(d_i32 + o_tm, tmatid, (size_t)total_ph * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && total_ph && sf) e = cudaMemcpyAsync(d_i32 + o_sf, sf, (size_t)total_ph * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && total_ph && ef) e = cudaMemcpyAsync(d_i32 + o_ef, ef, (size_t)total_ph * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_al_senid, senid.data(), senid.size() * 2, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_al_tokoff, tok_off.data(), tok_off.size() * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(align_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaEventRecord(c->al_ev[0], st);
    if (e == cudaSuccess) {
        align_kernel<<<(unsigned)n_utt, 128, smem, st>>>(d_senscr, d_i32 + o_utt, dev_ctx(c), d_i32 + o_ph, c->d_al_senid, d_i32 + o_tm,
                                                        sf ? d_i32 + o_sf : nullptr, ef ? d_i32 + o_ef : nullptr, d_tok,
                                                        d_tok + tok_off[(size_t)n_utt], c->d_al_tokoff, d_i32 + o_ss, d_i32 + o_sd,
                                                        d_i32 + o_sc, d_i32 + o_st);
        g_psb_launches.fetch_add(1, std::memory_order_relaxed);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaEventRecord(c->al_ev[1], st);
    if (e == cudaSuccess && n_state) e = cudaMemcpyAsync(st_start, d_i32 + o_ss, n_state * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && n_state) e = cudaMemcpyAsync(st_dur, d_i32 + o_sd, n_state * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && n_state) e = cudaMemcpyAsync(st_score, d_i32 + o_sc, n_state * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(status, d_i32 + o_st, (size_t)n_utt * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&c->last_align_ms, c->al_ev[0], c->al_ev[1]);
    if (e != cudaSuccess) {
        psb_set_error("psb_align_batch_device: %s", cudaGetErrorString(e));
        return PSB_ERR_CUDA;
    }
    return PSB_OK;
}

extern "C" float psb_align_last_kernel_ms(const psb_hmmctx_t *c)
{
    return c ? c->last_align_ms : 0.f;
}

extern "C" int psb_align_batch_host(psb_hmmctx_t *c, const int16_t *senscr, const int32_t *utt_off, int32_t n_utt,
                                    const int32_t *ph_off, const int32_t *ssid, const int32_t *tmatid,
                                    const int32_t *sf, const int32_t *ef,
                                    int32_t *st_start, int32_t *st_dur, int32_t *st_score, int32_t *status)
{
    PSB_REQUIRE(c && utt_off && n_utt >= 0, "psb_align_batch_host: bad argument");
    if (n_utt == 0) return PSB_OK;
    PSB_CUDA(cudaSetDevice(c->device));
    const size_t nb = (size_t)utt_off[n_utt] * c->n_sen * 2;
    PSB_REQUIRE(nb == 0 || senscr, "psb_align_batch_host: scores missing");
    int16_t *d = nullptr;
    PSB_CUDA(cudaMalloc((void **)&d, std::max<size_t>(nb, 2)));
    cudaError_t e = nb ? cudaMemcpy(d, senscr, nb, cudaMemcpyHostToDevice) : cudaSuccess;
    int rc = PSB_OK;
    if (e == cudaSuccess)
        rc = psb_align_batch_device(c, d, utt_off, n_utt, ph_off, ssid, tmatid, sf, ef, st_start, st_dur, st_score, status);
    cudaFree(d);
    if (e != cudaSuccess) {
        psb_set_error("psb_align_batch_host: %s", cudaGetErrorString(e));
        return PSB_ERR_CUDA;
    }
    return rc;
}

// ---------------------------------------------------------------------------------------
// Keyword spotting: kws_search.c on the device for whole batches (SURVEY 8 row b5 lists its
// kws_search_hmm_eval, kws_search.c:194).  One CTA per utterance; the phone loop (all CI phones)
// and the keyphrases' HMM chains sit side by side in shared memory (SoA); per frame
// kws_search_hmm_eval (:194-229), kws_search_hmm_prune (:234-251) and kws_search_trans (:256-348):
// first-best exit score of the phone loop, detections, phone-loop re-entry, chain transitions
// (decided from the state BEFORE any entry of this frame, which is what the reference's reverse
// loop order achieves) and the chains' start from the phone loop.  Every detection the reference
// would pass to kws_detections_add comes back as a row (frame, keyphrase, start frame, prob, ascr)
// in the reference's order; the host applies the unchanged list logic (kws_detections.c:55-80).
namespace {

constexpr int KWS_MAX_SCORE = 1500;         // KWS_MAX, kws_search.c:59

__global__ void __launch_bounds__(128)
kws_kernel(const int16_t *__restrict__ senscr, const int32_t *__restrict__ utt_off, HmmCtxDev c,
           int n_pl, int n_kp, const int32_t *__restrict__ kp_off, const int32_t *__restrict__ kp_thresh,
           const uint16_t *__restrict__ senid_g, const int32_t *__restrict__ tmatid_g, const int32_t *__restrict__ kp_of,
           int beam, int plp, int32_t *__restrict__ hits, int cap, int32_t *__restrict__ n_hits)
{
    extern __shared__ int sm[];
    const int u = blockIdx.x, tid = threadIdx.x, N = c.n_emit;
    const int H = n_pl + kp_off[n_kp];
    const long long f0 = utt_off[u];
    const int T = utt_off[u + 1] - utt_off[u];
    int *score = sm;                       // [N][H]
    int *hist = score + N * H;             // [N][H]
    int *out_score = hist + N * H;         // [H]
    int *out_hist = out_score + H;         // [H]
    int *bestsc = out_hist + H;            // [H]
    int *frame = bestsc + H;               // [H]
    int *sval = frame + H;                 // [32]
    int *sidx = sval + 32;                 // [32]
    int32_t *my_hits = hits + (size_t)u * cap * 5;
    int nh = 0;

    // kws_search_reinit: hmm_init (= hmm_clear); kws_search_start: phone loop hmm_clear + hmm_enter(0, -1, 0)
    for (int i = tid; i < H; i += blockDim.x) {
        for (int s = 0; s < N; ++s) { score[s * H + i] = PSB_WORST_SCORE; hist[s * H + i] = -1; }
        out_score[i] = PSB_WORST_SCORE; out_hist[i] = -1; bestsc[i] = PSB_WORST_SCORE; frame[i] = -1;
        if (i < n_pl) { score[i] = 0; hist[i] = -1; frame[i] = 0; }
    }
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        const int16_t *row = senscr + (f0 + t) * c.n_sen;
        int bs = PSB_WORST_SCORE;
        // kws_search_hmm_eval: the phone loop always, keyphrase HMMs when active (frame > 0)
        for (int i = tid; i < H; i += blockDim.x) {
            if (i >= n_pl && !(frame[i] > 0)) continue;
            HmmReg h;
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s) {
                h.score[s] = s < N ? score[s * H + i] : PSB_WORST_SCORE;
                h.hist[s] = s < N ? hist[s * H + i] : -1;
                h.senid[s] = s < N ? senid_g[(size_t)i * N + s] : PSB_BAD_SSID;
            }
            h.out_score = out_score[i]; h.out_hist = out_hist[i]; h.best = bestsc[i];
            const int b = hmm_step(h, c, tmatid_g[i], false, row);
            if (b > bs) bs = b;
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s)
                if (s < N) { score[s * H + i] = h.score[s]; hist[s * H + i] = h.hist[s]; }
            out_score[i] = h.out_score; out_hist[i] = h.out_hist; bestsc[i] = h.best;
        }
        int dummy;
        bs = block_reduce_max_pair<int>(bs, 0, sidx, sval, dummy);
        // kws_search_hmm_prune: hmm_clear on active keyphrase HMMs below the beam
        const int thresh = bs + beam;
        int cand = PSB_WORST_SCORE, cidx = 0x7fffffff;
        for (int i = tid; i < H; i += blockDim.x) {
            if (i >= n_pl) {
                if (frame[i] > 0 && bestsc[i] < thresh) {
                    for (int s = 0; s < N; ++s) { score[s * H + i] = PSB_WORST_SCORE; hist[s * H + i] = -1; }
                    out_score[i] = PSB_WORST_SCORE; out_hist[i] = -1; bestsc[i] = PSB_WORST_SCORE; frame[i] = -1;
                }
            }
            else if (out_score[i] > cand) { cand = out_score[i]; cidx = i; }   // first best exit of the phone loop
        }
        int plb;
        cand = block_reduce_max_pair<int>(cand, cidx, sidx, sval, plb);   // ties -> smallest index = first in scan order
        __syncthreads();
        if (cand > PSB_WORST_SCORE) {                                     // else "out probs are not ready yet"
            const int plb_out = cand, plb_hist = out_hist[plb];
            // detections, in keyphrase order
            if (tid == 0)
                for (int k = 0; k < n_kp; ++k) {
                    if (kp_off[k + 1] - kp_off[k] < 1) continue;
                    const int last = n_pl + kp_off[k + 1] - 1;
                    if (frame[last] > 0 && out_score[last] - plb_out >= kp_thresh[k]) {
                        if (nh < cap) {
                            int32_t *hrow = my_hits + (size_t)nh * 5;
                            hrow[0] = t; hrow[1] = k; hrow[2] = out_hist[last];
                            hrow[3] = out_score[last] - plb_out - KWS_MAX_SCORE; hrow[4] = out_score[last];
                        }
                        ++nh;
                    }
                }
            // transitions: decide from the pre-entry state, then apply
            int e_sc[4], e_hi[4];
            bool e_on[4];
            int q = 0;
            for (int i = tid; i < H; i += blockDim.x, ++q) {
                bool on = false; int sc = 0, hi = 0;
                if (i < n_pl) {                                            // phone-loop re-entry (:303-311)
                    if (plb_out + plp > score[i]) { on = true; sc = plb_out + plp; hi = plb_hist; }
                }
                else {
                    const int j = i - n_pl, k = kp_of[j];
                    if (j > kp_off[k]) {                                   // inside a chain (:320-332)
                        if (frame[i - 1] > 0 && (!(frame[i] > 0) || out_score[i - 1] > score[i])) {
                            on = true; sc = out_score[i - 1]; hi = out_hist[i - 1];
                        }
                    }
                    else if (plb_out > score[i]) { on = true; sc = plb_out; hi = t; }   // chain start (:335-340)
                }
                if (q < 4) { e_on[q] = on; e_sc[q] = sc; e_hi[q] = hi; }
            }
            __syncthreads();
            q = 0;
            for (int i = tid; i < H; i += blockDim.x, ++q)
                if (q < 4 && e_on[q]) { score[i] = e_sc[q]; hist[i] = e_hi[q]; frame[i] = t + 1; }   // hmm_enter
        }
        __syncthreads();
    }
    if (tid == 0) n_hits[u] = nh;
}

}  // namespace

extern "C" int psb_kws_batch_device(psb_hmmctx_t *c, const int16_t *d_senscr, const int32_t *utt_off, int32_t n_utt,
                                    int32_t n_pl, const int32_t *pl_ssid, const int32_t *pl_tmat, int32_t n_kp,
                                    const int32_t *kp_off, const int32_t *kp_thresh, const int32_t *kp_ssid,
                                    const int32_t *kp_tmat, int32_t beam, int32_t plp, int32_t *hits,
                                    int32_t cap_per_utt, int32_t *n_hits)
{
    PSB_REQUIRE(c && utt_off && n_utt >= 0 && n_pl > 0 && pl_ssid && pl_tmat && n_kp >= 0 && kp_off && hits && n_hits &&
                cap_per_utt > 0, "psb_kws_batch_device: bad argument");
    if (n_utt == 0) return PSB_OK;
    PSB_REQUIRE(utt_off[0] == 0 && kp_off[0] == 0, "psb_kws_batch_device: offsets must start at 0");
    PSB_REQUIRE(d_senscr || utt_off[n_utt] == 0, "psb_kws_batch_device: scores missing");
    const int N = c->n_emit, n_k = kp_off[n_kp], H = n_pl + n_k;
    PSB_REQUIRE(n_k == 0 || (kp_ssid && kp_tmat && kp_thresh), "psb_kws_batch_device: keyphrase tables missing");
    PSB_REQUIRE(H <= 4 * 128, "psb_kws_batch_device: %d HMMs exceed the 512 this kernel keeps per utterance", H);
    PSB_CUDA(cudaSetDevice(c->device));
    std::vector<uint16_t> sseq((size_t)c->n_sseq * N);
    PSB_CUDA(cudaMemcpy(sseq.data(), c->d_sseq, sseq.size() * 2, cudaMemcpyDeviceToHost));
    std::vector<uint16_t> senid((size_t)H * N);
    std::vector<int32_t> ibuf;                       // utt_off | kp_off | kp_thresh | tmatid[H] | kp_of[n_k]
    ibuf.insert(ibuf.end(), utt_off, utt_off + n_utt + 1);
    const size_t o_kpoff = ibuf.size();
    ibuf.insert(ibuf.end(), kp_off, kp_off + n_kp + 1);
    const size_t o_thr = ibuf.size();
    for (int k = 0; k < n_kp; ++k) ibuf.push_back(kp_thresh[k]);
    const size_t o_tm = ibuf.size();
    for (int i = 0; i < H; ++i) {
        const int ss = i < n_pl ? pl_ssid[i] : kp_ssid[i - n_pl], tm = i < n_pl ? pl_tmat[i] : kp_tmat[i - n_pl];
        PSB_REQUIRE(ss >= 0 && ss < c->n_sseq, "kws: ssid %d out of range", ss);
        PSB_REQUIRE(tm >= 0 && tm < c->n_tmat, "kws: tmatid %d out of range", tm);
        for (int s = 0; s < N; ++s) {
            const uint16_t v = sseq[(size_t)ss * N + s];
            PSB_REQUIRE(v < c->n_sen, "senone id %d out of range", v);
            senid[(size_t)i * N + s] = v;
        }
        ibuf.push_back(tm);
    }
    const size_t o_of = ibuf.size();
    for (int k = 0; k < n_kp; ++k) {
        PSB_REQUIRE(kp_off[k + 1] >= kp_off[k], "psb_kws_batch_device: kp_off not monotone at %d", k);
        for (int j = kp_off[k]; j < kp_off[k + 1]; ++j) ibuf.push_back(k);
    }
    const size_t o_nh = ibuf.size();
    ibuf.resize(o_nh + (size_t)n_utt, 0);
    const size_t smem = ((size_t)(2 * N + 4) * H + 64) * sizeof(int);
    int32_t *d_i = nullptr, *d_hits = nullptr;
    uint16_t *d_senid = nullptr;
    const size_t hits_n = (size_t)n_utt * cap_per_utt * 5;
    cudaError_t e = cudaMalloc((void **)&d_i, ibuf.size() * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&d_hits, hits_n * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&d_senid, senid.size() * 2);
    cudaStream_t st = c->stream;
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_i, ibuf.data(), ibuf.size() * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_senid, senid.data(), senid.size() * 2, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        kws_kernel<<<(unsigned)n_utt, 128, smem, st>>>(d_senscr, d_i, dev_ctx(c), n_pl, n_kp, d_i + o_kpoff, d_i + o_thr, d_senid,
                                                      d_i + o_tm, d_i + o_of, beam, plp, d_hits, cap_per_utt, d_i + o_nh);
        g_psb_launches.fetch_add(1, std::memory_order_relaxed);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(hits, d_hits, hits_n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(n_hits, d_i + o_nh, (size_t)n_utt * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_i); cudaFree(d_hits); cudaFree(d_senid);
    if (e != cudaSuccess) {
        psb_set_error("psb_kws_batch_device: %s", cudaGetErrorString(e));
        return PSB_ERR_CUDA;
    }
    return PSB_OK;
}

// ---------------------------------------------------------------------------------------
// Phone decoding: allphone_search.c without a phone LM, for whole batches (SURVEY 8 row b5 lists
// its phmm_eval_all, allphone_search.c:349).  One CTA per utterance, the PHMM graph's state in
// shared memory (SoA): per frame phmm_eval_all (:349-378), phmm_exit (:380-456: every active node
// whose best score is inside pbeam appends a history entry -- numbered in node order by a block
// prefix sum -- the others are cleared) and phmm_trans (:458-524).  The reference pushes the new
// history entries to their successors one by one, each entering its target if it beats the
// beam and the target's state-0 score so far; per target that is "the first maximum over its
// exited predecessors", so the kernel pulls: every node scans its predecessor list (CSR, node
// order = history order).  The history table (ef, node, predecessor entry, score) goes back to
// the host, whose unchanged allphone_backtrace (:765-840) turns it into the phone segmentation.
namespace {

// LM = true: every transition carries its own phone-LM score from dense tables (bg [n_ci][n_ci],
// tg [n_ci][n_ci][n_ci], scores >> SENSCR_SHIFT tabulated by the host with the argument positions of
// phmm_exit / phmm_trans, allphone_search.c:416-441, 497-513); history rows get a fifth column.
template <bool LM>
__global__ void __launch_bounds__(128)
allphone_kernel(const int16_t *__restrict__ senscr, const int32_t *__restrict__ utt_off, HmmCtxDev c, int H,
                const uint16_t *__restrict__ senid_g, const int32_t *__restrict__ tmatid_g,
                const int32_t *__restrict__ pred_off, const int32_t *__restrict__ pred, int start,
                int beam, int pbeam, int inspen, int32_t *__restrict__ hist_out, int cap, int32_t *__restrict__ n_hist,
                int n_ci, const int32_t *__restrict__ node_ci, const int32_t *__restrict__ bg, const int32_t *__restrict__ tg)
{
    constexpr int ROW = LM ? 5 : 4;
    extern __shared__ int sm[];
    const int u = blockIdx.x, tid = threadIdx.x, N = c.n_emit, nt = blockDim.x;
    const long long f0 = utt_off[u];
    const int T = utt_off[u + 1] - utt_off[u];
    int *score = sm;                       // [N][H]
    int *hist = score + N * H;             // [N][H]
    int *out_score = hist + N * H;         // [H]
    int *out_hist = out_score + H;         // [H]
    int *bestsc = out_hist + H;            // [H]
    int *frame = bestsc + H;               // [H]
    int *ex_idx = frame + H;               // [H] history index of the entry this node appended this frame, or -1
    int *sval = ex_idx + H;                // [32]
    int *sidx = sval + 32;                 // [32]
    int *wsum = sidx + 32;                 // [32]
    int *pci = wsum + 32;                  // [H] (LM) CI phone of the predecessor entry of this node's new entry, or -1
    int32_t *my_hist = hist_out + (size_t)u * cap * ROW;
    int nh = 0;                                                   // uniform across the block
    const int chunk = (H + nt - 1) / nt, c0 = min(H, tid * chunk), c1 = min(H, c0 + chunk);

    // allphone_search_start: hmm_clear everything, hmm_enter(silence, 0, 0, 0)
    for (int i = tid; i < H; i += nt) {
        for (int s = 0; s < N; ++s) { score[s * H + i] = PSB_WORST_SCORE; hist[s * H + i] = -1; }
        out_score[i] = PSB_WORST_SCORE; out_hist[i] = -1; bestsc[i] = PSB_WORST_SCORE; frame[i] = -1; ex_idx[i] = -1;
    }
    __syncthreads();
    if (tid == 0) { score[start] = 0; hist[start] = 0; frame[start] = 0; }
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        const int16_t *row = senscr + (f0 + t) * c.n_sen;
        const int nf = t + 1;
        int bs = PSB_WORST_SCORE;
        for (int i = tid; i < H; i += nt) {                       // phmm_eval_all
            if (frame[i] != t) continue;
            HmmReg h;
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s) {
                h.score[s] = s < N ? score[s * H + i] : PSB_WORST_SCORE;
                h.hist[s] = s < N ? hist[s * H + i] : -1;
                h.senid[s] = s < N ? senid_g[(size_t)i * N + s] : PSB_BAD_SSID;
            }
            h.out_score = out_score[i]; h.out_hist = out_hist[i]; h.best = bestsc[i];
            const int b = hmm_step(h, c, tmatid_g[i], false, row);
            if (b > bs) bs = b;
#pragma unroll
            for (int s = 0; s < PSB_HMM_MAX_NSTATE; ++s)
                if (s < N) { score[s * H + i] = h.score[s]; hist[s * H + i] = h.hist[s]; }
            out_score[i] = h.out_score; out_hist[i] = h.out_hist; bestsc[i] = h.best;
        }
        int dummy;
        const int best = block_reduce_max_pair<int>(bs, 0, sidx, sval, dummy);
        __syncthreads();
        // phmm_exit: history entries numbered in node order (contiguous chunk per thread + block scan)
        const int th = best + pbeam;
        int cnt = 0;
        for (int i = c0; i < c1; ++i) cnt += (frame[i] == t && bestsc[i] >= th) ? 1 : 0;
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if ((tid & 31) >= o) incl += v;
        }
        if ((tid & 31) == 31) wsum[tid >> 5] = incl;
        __syncthreads();
        int base = nh, total = 0;
        for (int w = 0; w < (nt >> 5); ++w) {
            if (w < (tid >> 5)) base += wsum[w];
            total += wsum[w];
        }
        int k = base + incl - cnt;
        for (int i = c0; i < c1; ++i) {
            if (frame[i] != t) { ex_idx[i] = -1; continue; }
            if (bestsc[i] >= th) {
                if (LM) {
                    // phmm_exit's tscore (:416-441); it reads the SAME entry as pred and pred_pred
                    const int hh = out_hist[i];
                    int tscore = 0, pc = -1;
                    if (hh > 0 && hh < cap) {
                        pc = node_ci[my_hist[(size_t)hh * ROW + 1]];
                        tscore = my_hist[(size_t)hh * ROW + 2] > 0 ? tg[((size_t)pc * n_ci + pc) * n_ci + node_ci[i]]
                                                                  : bg[(size_t)pc * n_ci + node_ci[i]];
                    }
                    pci[i] = pc;
                    if (k < cap) my_hist[(size_t)k * ROW + 4] = tscore;
                }
                if (k < cap) {
                    int32_t *r = my_hist + (size_t)k * ROW;
                    r[0] = t; r[1] = i; r[2] = out_hist[i]; r[3] = out_score[i];
                }
                ex_idx[i] = k++;
                frame[i] = nf;
            }
            else {                                                // hmm_clear
                for (int s = 0; s < N; ++s) { score[s * H + i] = PSB_WORST_SCORE; hist[s * H + i] = -1; }
                out_score[i] = PSB_WORST_SCORE; out_hist[i] = -1; bestsc[i] = PSB_WORST_SCORE; frame[i] = -1;
                ex_idx[i] = -1;
            }
        }
        nh += total;
        __syncthreads();
        // phmm_trans, pulled per target: first maximum over the exited predecessors
        const int floor_ = best + beam;
        for (int i = tid; i < H; i += nt) {
            int cand = INT_MIN, ck = -1;
            for (int l = pred_off[i]; l < pred_off[i + 1]; ++l) {
                const int p = pred[l];
                if (ex_idx[p] < 0) continue;
                int ns;
                if (LM) {
                    const int fc = node_ci[p], tc = node_ci[i];
                    ns = out_score[p] + (pci[p] >= 0 ? tg[((size_t)pci[p] * n_ci + fc) * n_ci + tc] : bg[(size_t)fc * n_ci + tc]);
                }
                else
                    ns = out_score[p] + inspen;
                if (ns > cand) { cand = ns; ck = ex_idx[p]; }
            }
            if (ck >= 0 && cand > floor_ && cand > score[i]) { score[i] = cand; hist[i] = ck; frame[i] = nf; }   // hmm_enter
        }
        __syncthreads();
    }
    if (tid == 0) n_hist[u] = nh;
}

}  // namespace

static int allphone_common(psb_hmmctx_t *c, const int16_t *d_senscr, const int32_t *utt_off, int32_t n_utt,
                           int32_t n_nodes, const int32_t *ssid, const int32_t *tmatid,
                           const int32_t *succ_off, const int32_t *succ, int32_t start, int32_t beam,
                           int32_t pbeam, int32_t inspen, int32_t *hist, int32_t cap_per_utt, int32_t *n_hist,
                           int32_t n_ci, const int32_t *node_ci, const int32_t *bg, const int32_t *tg)
{
    const bool lm = bg != nullptr;
    const int ROW = lm ? 5 : 4;
    PSB_REQUIRE(c && utt_off && n_utt >= 0 && n_nodes > 0 && ssid && tmatid && succ_off && hist && n_hist && cap_per_utt > 0 &&
                start >= 0 && start < n_nodes, "psb_allphone_batch_device: bad argument");
    if (n_utt == 0) return PSB_OK;
    PSB_REQUIRE(utt_off[0] == 0 && succ_off[0] == 0, "psb_allphone_batch_device: offsets must start at 0");
    PSB_REQUIRE(d_senscr || utt_off[n_utt] == 0, "psb_allphone_batch_device: scores missing");
    const int N = c->n_emit, H = n_nodes, n_links = succ_off[n_nodes];
    PSB_REQUIRE(n_links == 0 || succ, "psb_allphone_batch_device: successor lists missing");
    const size_t smem = ((size_t)(2 * N + 6) * H + 96) * sizeof(int);
    PSB_REQUIRE(smem <= 200 * 1024, "psb_allphone_batch_device: a graph of %d PHMMs does not fit shared memory "
                "(context-independent graphs, -allphone_ci yes, have one node per phone)", H);
    PSB_CUDA(cudaSetDevice(c->device));
    std::vector<uint16_t> sseq((size_t)c->n_sseq * N);
    PSB_CUDA(cudaMemcpy(sseq.data(), c->d_sseq, sseq.size() * 2, cudaMemcpyDeviceToHost));
    std::vector<uint16_t> senid((size_t)H * N);
    // predecessor lists in node order (= the order the reference appends and walks history entries)
    std::vector<int32_t> ibuf;                       // utt_off | tmatid[H] | pred_off[H+1] | pred[n_links] | n_hist[n_utt]
    ibuf.insert(ibuf.end(), utt_off, utt_off + n_utt + 1);
    const size_t o_tm = ibuf.size();
    for (int i = 0; i < H; ++i) {
        PSB_REQUIRE(ssid[i] >= 0 && ssid[i] < c->n_sseq, "allphone: ssid[%d] out of range", i);
        PSB_REQUIRE(tmatid[i] >= 0 && tmatid[i] < c->n_tmat, "allphone: tmatid[%d] out of range", i);
        for (int s = 0; s < N; ++s) {
            const uint16_t v = sseq[(size_t)ssid[i] * N + s];
            PSB_REQUIRE(v < c->n_sen, "senone id %d out of range", v);
            senid[(size_t)i * N + s] = v;
        }
        ibuf.push_back(tmatid[i]);
    }
    std::vector<int32_t> pcount((size_t)H + 1, 0);
    for (int i = 0; i < H; ++i) {
        PSB_REQUIRE(succ_off[i + 1] >= succ_off[i], "psb_allphone_batch_device: succ_off not monotone at %d", i);
        for (int l = succ_off[i]; l < succ_off[i + 1]; ++l) {
            PSB_REQUIRE(succ[l] >= 0 && succ[l] < H, "allphone: successor %d out of range", succ[l]);
            ++pcount[(size_t)succ[l] + 1];
        }
    }
    for (int i = 0; i < H; ++i) pcount[(size_t)i + 1] += pcount[(size_t)i];
    const size_t o_poff = ibuf.size();
    ibuf.insert(ibuf.end(), pcount.begin(), pcount.end());
    const size_t o_pred = ibuf.size();
    ibuf.resize(o_pred + (size_t)n_links);
    {
        std::vector<int32_t> fill(pcount.begin(), pcount.end() - 1);
        for (int i = 0; i < H; ++i)                               // ascending `from` => ascending inside every list
            for (int l = succ_off[i]; l < succ_off[i + 1]; ++l) ibuf[o_pred + (size_t)fill[(size_t)succ[l]]++] = i;
    }
    const size_t o_nh = ibuf.size();
    ibuf.resize(o_nh + (size_t)n_utt, 0);
    size_t o_ci = 0, o_bg = 0, o_tg = 0;
    if (lm) {
        PSB_REQUIRE(n_ci > 0 && node_ci && tg, "psb_allphone_lm_batch_device: LM tables missing");
        o_ci = ibuf.size();
        for (int i = 0; i < H; ++i) {
            PSB_REQUIRE(node_ci[i] >= 0 && node_ci[i] < n_ci, "allphone: node_ci[%d] out of range", i);
            ibuf.push_back(node_ci[i]);
        }
        o_bg = ibuf.size();
        ibuf.insert(ibuf.end(), bg, bg + (size_t)n_ci * n_ci);
        o_tg = ibuf.size();
        ibuf.insert(ibuf.end(), tg, tg + (size_t)n_ci * n_ci * n_ci);
    }
    int32_t *d_i = nullptr, *d_hist = nullptr;
    uint16_t *d_senid = nullptr;
    const size_t hist_n = (size_t)n_utt * cap_per_utt * ROW;
    cudaError_t e = cudaMalloc((void **)&d_i, ibuf.size() * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&d_hist, hist_n * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&d_senid, senid.size() * 2);
    cudaStream_t st = c->stream;
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_i, ibuf.data(), ibuf.size() * 4, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_senid, senid.data(), senid.size() * 2, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(allphone_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(allphone_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        if (lm)
            allphone_kernel<true><<<(unsigned)n_utt, 128, smem, st>>>(d_senscr, d_i, dev_ctx(c), H, d_senid, d_i + o_tm, d_i + o_poff,
                                                                     d_i + o_pred, start, beam, pbeam, inspen, d_hist, cap_per_utt,
                                                                     d_i + o_nh, n_ci, d_i + o_ci, d_i + o_bg, d_i + o_tg);
        else
            allphone_kernel<false><<<(unsigned)n_utt, 128, smem, st>>>(d_senscr, d_i, dev_ctx(c), H, d_senid, d_i + o_tm, d_i + o_poff,
                                                                      d_i + o_pred, start, beam, pbeam, inspen, d_hist, cap_per_utt,
                                                                      d_i + o_nh, 0, nullptr, nullptr, nullptr);
        g_psb_launches.fetch_add(1, std::memory_order_relaxed);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(hist, d_hist, hist_n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(n_hist, d_i + o_nh, (size_t)n_utt * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_i); cudaFree(d_hist); cudaFree(d_senid);
    if (e != cudaSuccess) {
        psb_set_error("psb_allphone_batch_device: %s", cudaGetErrorString(e));
        return PSB_ERR_CUDA;
    }
    return PSB_OK;
}

extern "C" int psb_allphone_batch_device(psb_hmmctx_t *c, const int16_t *d_senscr, const int32_t *utt_off, int32_t n_utt,
                                         int32_t n_nodes, const int32_t *ssid, const int32_t *tmatid,
                                         const int32_t *succ_off, const int32_t *succ, int32_t start, int32_t beam,
                                         int32_t pbeam, int32_t inspen, int32_t *hist, int32_t cap_per_utt, int32_t *n_hist)
{
    return allphone_common(c, d_senscr, utt_off, n_utt, n_nodes, ssid, tmatid, succ_off, succ, start, beam, pbeam, inspen, hist,
                           cap_per_utt, n_hist, 0, nullptr, nullptr, nullptr);
}

extern "C" int psb_allphone_lm_batch_device(psb_hmmctx_t *c, const int16_t *d_senscr, const int32_t *utt_off, int32_t n_utt,
                                            int32_t n_nodes, const int32_t *ssid, const int32_t *tmatid,
                                            const int32_t *succ_off, const int32_t *succ, int32_t start, int32_t beam,
                                            int32_t pbeam, int32_t n_ci, const int32_t *node_ci, const int32_t *bg,
                                            const int32_t *tg, int32_t *hist, int32_t cap_per_utt, int32_t *n_hist)
{
    PSB_REQUIRE(bg && tg && node_ci && n_ci > 0, "psb_allphone_lm_batch_device: LM tables missing");
    return allphone_common(c, d_senscr, utt_off, n_utt, n_nodes, ssid, tmatid, succ_off, succ, start, beam, pbeam, 0, hist,
                           cap_per_utt, n_hist, n_ci, node_ci, bg, tg);
}

