// psb_api.cu -- extern "C" entry points of libpsb200.so: model upload and batched scoring.
#include "psb_internal.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

std::atomic<long long> g_psb_launches{0};

static thread_local char g_err[512] = "";

void psb_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *psb_last_error(void) { return g_err; }
extern "C" int psb_abi_version(void) { return PSB_ABI_VERSION; }
extern "C" int64_t psb_kernel_launch_count(void) { return g_psb_launches.load(); }

extern "C" int psb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ---------------------------------------------------------------------------------------
// model

static int upload(void **dst, const void *src, size_t bytes, bool src_on_device)
{
    PSB_CUDA(cudaMalloc(dst, bytes ? bytes : 1));
    if (bytes)
        PSB_CUDA(cudaMemcpy(*dst, src, bytes, src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    return PSB_OK;
}

// Gaussians -> per-(codebook, stream) record blocks {det, mean0, var0, mean1, var1, ...}.
static int build_records(psb_model_t *m, const float *mean, const float *var, const float *det,
                         bool on_device)
{
    const size_t n_gau = (size_t)m->n_mgau * m->n_density * m->sumlen;
    const size_t n_det = (size_t)m->n_mgau * m->n_feat * m->n_density;
    std::vector<float> hm(n_gau), hv(n_gau), hd(n_det);
    cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost;
    PSB_CUDA(cudaMemcpy(hm.data(), mean, n_gau * sizeof(float), kind));
    PSB_CUDA(cudaMemcpy(hv.data(), var, n_gau * sizeof(float), kind));
    PSB_CUDA(cudaMemcpy(hd.data(), det, n_det * sizeof(float), kind));
    size_t total = 0;
    m->rec_off.assign(m->K, 0);
    for (int cb = 0; cb < m->n_mgau; ++cb)
        for (int f = 0; f < m->n_feat; ++f) {
            m->rec_off[cb * m->n_feat + f] = total;
            total += (size_t)m->n_density * rec_floats(m->featlen[f]);
        }
    std::vector<float> rec(total, 0.f);
    for (int cb = 0; cb < m->n_mgau; ++cb)
        for (int f = 0; f < m->n_feat; ++f) {
            const int fl = m->featlen[f], rf = rec_floats(fl);
            const size_t src = ((size_t)cb * m->sumlen + m->featoff[f]) * m->n_density;
            float *r = rec.data() + m->rec_off[cb * m->n_feat + f];
            for (int c = 0; c < m->n_density; ++c) {
                r[(size_t)c * rf] = hd[((size_t)cb * m->n_feat + f) * m->n_density + c];
                for (int j = 0; j < fl; ++j) {
                    r[(size_t)c * rf + 1 + 2 * j] = hm[src + (size_t)c * fl + j];
                    r[(size_t)c * rf + 2 + 2 * j] = hv[src + (size_t)c * fl + j];
                }
            }
        }
    if (!m->d_rec) {
        PSB_CUDA(cudaMalloc(&m->d_rec, total * sizeof(float)));
        PSB_CUDA(cudaMalloc(&m->d_rec_off, m->K * sizeof(size_t)));
        PSB_CUDA(cudaMemcpy(m->d_rec_off, m->rec_off.data(), m->K * sizeof(size_t), cudaMemcpyHostToDevice));
    }
    PSB_CUDA(cudaMemcpy(m->d_rec, rec.data(), total * sizeof(float), cudaMemcpyHostToDevice));
    if (m->kind != PSB_KIND_MS && m->n_density % 2 == 0 && !m->fixed_point) {
        // pair-interleaved, negated copy for ptm_topn2_kernel: per (cb, f) nd/2 pair records
        // {detA, detB, -muA_0, -muB_0, -vA_0, -vB_0, ...} padded to a multiple of 4 floats
        size_t total2 = 0;
        std::vector<size_t> off2(m->K);
        for (int cb = 0; cb < m->n_mgau; ++cb)
            for (int f = 0; f < m->n_feat; ++f) {
                off2[cb * m->n_feat + f] = total2;
                total2 += (size_t)(m->n_density / 2) * roundup(2 + 4 * m->featlen[f], 4);
            }
        std::vector<float> rec2(total2, 0.f);
        for (int cb = 0; cb < m->n_mgau; ++cb)
            for (int f = 0; f < m->n_feat; ++f) {
                const int fl = m->featlen[f], rf2 = roundup(2 + 4 * fl, 4);
                const size_t src = ((size_t)cb * m->sumlen + m->featoff[f]) * m->n_density;
                float *r = rec2.data() + off2[cb * m->n_feat + f];
                for (int c = 0; c < m->n_density; ++c) {
                    float *rp = r + (size_t)(c >> 1) * rf2 + (c & 1);
                    rp[0] = hd[((size_t)cb * m->n_feat + f) * m->n_density + c];
                    for (int j = 0; j < fl; ++j) {
                        rp[2 + 4 * j] = -hm[src + (size_t)c * fl + j];
                        rp[4 + 4 * j] = -hv[src + (size_t)c * fl + j];
                    }
                }
            }
        if (!m->d_rec2) {
            PSB_CUDA(cudaMalloc(&m->d_rec2, total2 * sizeof(float)));
            PSB_CUDA(cudaMalloc(&m->d_rec2_off, m->K * sizeof(size_t)));
            PSB_CUDA(cudaMemcpy(m->d_rec2_off, off2.data(), m->K * sizeof(size_t), cudaMemcpyHostToDevice));
        }
        PSB_CUDA(cudaMemcpy(m->d_rec2, rec2.data(), total2 * sizeof(float), cudaMemcpyHostToDevice));
    }
    {
        int rc = psb_tc_prepare(m, hm.data(), hv.data(), hd.data());
        if (rc) return rc;
    }
    if (m->kind == PSB_KIND_MS) {
        // codebook-minor copy for ms_dist_kernel: per stream f (at float offset featoff[f]*nd*2*n_mgau)
        // [(d*fl + j)*2 + {mean,var}][cb]; determinants [f][d][cb]
        std::vector<float> gT(n_gau * 2), dT(n_det);
        for (int cb = 0; cb < m->n_mgau; ++cb)
            for (int f = 0; f < m->n_feat; ++f) {
                const int fl = m->featlen[f];
                const size_t src = ((size_t)cb * m->sumlen + m->featoff[f]) * m->n_density;
                const size_t dst = (size_t)m->featoff[f] * m->n_density * 2 * m->n_mgau;
                for (int c = 0; c < m->n_density; ++c) {
                    dT[((size_t)f * m->n_density + c) * m->n_mgau + cb] = hd[((size_t)cb * m->n_feat + f) * m->n_density + c];
                    for (int j = 0; j < fl; ++j) {
                        gT[dst + ((size_t)(c * fl + j) * 2) * m->n_mgau + cb] = hm[src + (size_t)c * fl + j];
                        gT[dst + ((size_t)(c * fl + j) * 2 + 1) * m->n_mgau + cb] = hv[src + (size_t)c * fl + j];
                    }
                }
            }
        if (!m->d_msT) {
            PSB_CUDA(cudaMalloc(&m->d_msT, gT.size() * sizeof(float)));
            PSB_CUDA(cudaMalloc(&m->d_msdetT, dT.size() * sizeof(float)));
        }
        PSB_CUDA(cudaMemcpy(m->d_msT, gT.data(), gT.size() * sizeof(float), cudaMemcpyHostToDevice));
        PSB_CUDA(cudaMemcpy(m->d_msdetT, dT.data(), dT.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    return PSB_OK;
}

extern "C" int psb_model_create(const psb_model_desc_t *d, int device, psb_model_t **out)
{
    PSB_REQUIRE(d && out, "psb_model_create: null argument");
    PSB_REQUIRE(d->kind >= PSB_KIND_PTM && d->kind <= PSB_KIND_MS, "unknown model kind %d", d->kind);
    PSB_REQUIRE(d->n_feat >= 1 && d->n_feat <= PSB_MAX_FEAT, "n_feat %d out of range", d->n_feat);
    PSB_REQUIRE(d->n_sen > 0 && d->n_mgau > 0 && d->n_density > 0, "empty model");
    PSB_REQUIRE(d->topn >= 1 && d->topn <= PSB_MAX_TOPN, "topn %d out of range", d->topn);
    PSB_REQUIRE(d->mean && d->var && d->det && d->mixw && d->sen2cb, "missing model array");
    PSB_CUDA(cudaSetDevice(device));
    psb_model_t *m = new psb_model_t();
    m->device = device;
    m->kind = d->kind; m->n_sen = d->n_sen; m->n_mgau = d->n_mgau; m->n_feat = d->n_feat;
    m->n_density = d->n_density; m->topn = d->topn;
    m->ds_ratio = d->ds_ratio > 0 ? d->ds_ratio : 1;
    m->aw = d->aw != 0 ? d->aw : 1;
    m->sumlen = 0;
    for (int f = 0; f < d->n_feat; ++f) {
        m->featlen[f] = d->featlen[f];
        m->featoff[f] = m->sumlen;
        m->sumlen += d->featlen[f];
    }
    m->K = m->n_mgau * m->n_feat;
    m->mixw_4bit = d->mixw_cb != nullptr;
    m->fixed_point = d->fixed_point != 0;
    if (m->fixed_point && d->kind == PSB_KIND_MS) {
        psb_set_error("fixed-point arithmetic is implemented for ptm and semi-continuous models only");
        delete m;
        return PSB_ERR_ARG;
    }
    m->logadd_ms_size = d->logadd_ms_size;
    m->logadd_ms_zero = d->logadd_ms_zero;
    m->d_rec = nullptr; m->d_rec_off = nullptr; m->d_rec2 = nullptr; m->d_rec2_off = nullptr; m->d_mixw = nullptr; m->d_mixw_cb = nullptr;
    m->d_sen2cb = nullptr; m->d_sen2cb32 = nullptr; m->d_quadcb = nullptr; m->d_bsen = nullptr; m->n_bsen = 0; m->d_logadd8 = nullptr; m->d_logadd_ms = nullptr;
    m->has_topn_beam = false;
    m->d_topn_beam = nullptr;
    m->tc_ok = false;
    m->d_tc_wumma = m->d_tc_cen = m->d_tc_bnd = nullptr;
    m->d_msT = m->d_msdetT = nullptr; m->d_featlen = m->d_featoff = nullptr;
    for (int f = 0; f < PSB_MAX_FEAT; ++f) m->topn_beam[f] = 0;
    const bool dev = d->on_device != 0;
    int rc = build_records(m, d->mean, d->var, d->det, dev);
    if (!rc) rc = upload((void **)&m->d_featlen, m->featlen, sizeof(m->featlen), false);
    if (!rc) rc = upload((void **)&m->d_featoff, m->featoff, sizeof(m->featoff), false);
    if (rc) { psb_model_free(m); return rc; }

    // senone -> codebook map
    std::vector<int32_t> s2c(m->n_sen);
    if (cudaMemcpy(s2c.data(), d->sen2cb, m->n_sen * sizeof(int32_t),
                   dev ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost) != cudaSuccess) {
        psb_set_error("copying sen2cb failed");
        psb_model_free(m);
        return PSB_ERR_CUDA;
    }
    std::vector<uint16_t> s2c16(m->n_sen);
    for (int i = 0; i < m->n_sen; ++i) {
        if (s2c[i] < 0 || s2c[i] >= m->n_mgau) {
            psb_set_error("sen2cb[%d] = %d out of range", i, s2c[i]);
            psb_model_free(m);
            return PSB_ERR_ARG;
        }
        s2c16[i] = (uint16_t)s2c[i];
    }
    {
        const int nq = (m->n_sen + 3) / 4;
        std::vector<int16_t> quadcb(nq, -1);
        std::vector<int32_t> bsen;
        for (int q = 0; q < nq; ++q) {
            const int s0 = 4 * q;
            bool uni = s0 + 3 < m->n_sen && m->n_mgau <= 32767;
            for (int i = 1; uni && i < 4; ++i) uni = s2c[s0 + i] == s2c[s0];
            if (uni) quadcb[q] = (int16_t)s2c[s0];
            else for (int i = 0; i < 4 && s0 + i < m->n_sen; ++i) bsen.push_back(s0 + i);
        }
        m->n_bsen = (int)bsen.size();
        if ((rc = upload((void **)&m->d_quadcb, quadcb.data(), nq * sizeof(int16_t), false)) ||
            (rc = upload((void **)&m->d_bsen, bsen.data(), bsen.size() * sizeof(int32_t), false))) {
            psb_model_free(m);
            return rc;
        }
    }
    m->sen_is_cb = m->n_mgau == m->n_sen;
    for (int i = 0; m->sen_is_cb && i < m->n_sen; ++i) m->sen_is_cb = s2c[i] == i;
    if ((rc = upload((void **)&m->d_sen2cb, s2c16.data(), m->n_sen * sizeof(uint16_t), false)) ||
        (rc = upload((void **)&m->d_sen2cb32, s2c.data(), m->n_sen * sizeof(int32_t), false))) {
        psb_model_free(m);
        return rc;
    }

    // mixture weights
    if (m->kind == PSB_KIND_MS) {
        m->mixw_row = m->n_sen;
        m->mixw_stride = m->n_sen;
        rc = upload((void **)&m->d_mixw, d->mixw, (size_t)m->n_sen * m->n_feat * m->n_density, dev);
    }
    else {
        m->mixw_row = m->mixw_4bit ? (m->n_sen + 1) / 2 : m->n_sen;
        m->mixw_stride = roundup(m->mixw_row, 128);
        const size_t rows = (size_t)m->n_feat * m->n_density;
        rc = upload((void **)&m->d_mixw, nullptr, 0, false);
        if (!rc) {
            cudaFree(m->d_mixw);
            m->d_mixw = nullptr;
            if (cudaMalloc(&m->d_mixw, rows * m->mixw_stride) != cudaSuccess ||
                cudaMemset(m->d_mixw, 0, rows * m->mixw_stride) != cudaSuccess ||
                cudaMemcpy2D(m->d_mixw, m->mixw_stride, d->mixw, m->mixw_row, m->mixw_row, rows,
                             dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice) != cudaSuccess) {
                psb_set_error("uploading mixture weights failed: %s", cudaGetErrorString(cudaGetLastError()));
                rc = PSB_ERR_CUDA;
            }
        }
    }
    if (!rc && m->mixw_4bit) rc = upload((void **)&m->d_mixw_cb, d->mixw_cb, 16, dev);
    if (!rc && d->logadd8) {
        // 256 entries from the caller (logmath.c:116-120), continued with zeros: see logadd8()
        if (cudaMalloc((void **)&m->d_logadd8, PSB_LOGADD8_N) != cudaSuccess ||
            cudaMemset(m->d_logadd8, 0, PSB_LOGADD8_N) != cudaSuccess ||
            cudaMemcpy(m->d_logadd8, d->logadd8, 256, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice) != cudaSuccess) {
            psb_set_error("uploading the log-add table failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = PSB_ERR_CUDA;
        }
        else {
            uint8_t t[256];
            if (cudaMemcpy(t, m->d_logadd8, 256, cudaMemcpyDeviceToHost) == cudaSuccess)
                for (int i = 0; i < 256; ++i) m->logadd8_max = std::max<int>(m->logadd8_max, t[i]);
        }
    }
    if (!rc && m->kind != PSB_KIND_MS && !d->logadd8) {
        psb_set_error("logadd8 table required for ptm/semi models");
        rc = PSB_ERR_ARG;
    }
    if (!rc && m->kind == PSB_KIND_MS) {
        if (!d->logadd_ms || d->logadd_ms_size <= 0) {
            psb_set_error("logadd_ms table required for ms models");
            rc = PSB_ERR_ARG;
        }
        else
            rc = upload((void **)&m->d_logadd_ms, d->logadd_ms, (size_t)d->logadd_ms_size * sizeof(uint32_t), dev);
    }
    if (!rc && d->topn_beam) {
        uint8_t tb[PSB_MAX_FEAT] = {0};
        if (cudaMemcpy(tb, d->topn_beam, m->n_feat, dev ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost) != cudaSuccess)
            rc = PSB_ERR_CUDA;
        for (int f = 0; f < m->n_feat; ++f) {
            m->topn_beam[f] = tb[f];
            if (tb[f]) m->has_topn_beam = true;
        }
    }
    if (!rc) {
        int32_t tb[PSB_MAX_FEAT] = {0};
        for (int f = 0; f < m->n_feat; ++f) tb[f] = m->has_topn_beam ? m->topn_beam[f] : 0;
        rc = upload((void **)&m->d_topn_beam, tb, sizeof(tb), false);
    }
    if (rc) { psb_model_free(m); return rc; }
    *out = m;
    return PSB_OK;
}

extern "C" void psb_model_free(psb_model_t *m)
{
    if (!m) return;
    cudaSetDevice(m->device);
    cudaFree(m->d_rec); cudaFree(m->d_rec_off); cudaFree(m->d_rec2); cudaFree(m->d_rec2_off); cudaFree(m->d_mixw); cudaFree(m->d_mixw_cb);
    cudaFree(m->d_sen2cb); cudaFree(m->d_sen2cb32); cudaFree(m->d_quadcb); cudaFree(m->d_bsen); cudaFree(m->d_logadd8); cudaFree(m->d_logadd_ms);
    cudaFree(m->d_topn_beam); cudaFree(m->d_msT); cudaFree(m->d_msdetT); cudaFree(m->d_featlen); cudaFree(m->d_featoff);
    cudaFree(m->d_tc_wumma); cudaFree(m->d_tc_cen); cudaFree(m->d_tc_bnd);
    delete m;
}

extern "C" int psb_model_update_gaussians(psb_model_t *m, const float *mean, const float *var, const float *det)
{
    PSB_REQUIRE(m && mean && var && det, "psb_model_update_gaussians: null argument");
    PSB_CUDA(cudaSetDevice(m->device));
    PSB_CUDA(cudaDeviceSynchronize());
    return build_records(m, mean, var, det, false);
}

extern "C" int psb_model_n_sen(const psb_model_t *m) { return m ? m->n_sen : 0; }
extern "C" int psb_model_device(const psb_model_t *m) { return m ? m->device : -1; }

// ---------------------------------------------------------------------------------------
// batch

extern "C" int psb_batch_create(psb_model_t *m, int32_t max_utts, int64_t max_frames, psb_batch_t **out)
{
    PSB_REQUIRE(m && out && max_utts > 0 && max_frames > 0, "psb_batch_create: bad argument");
    PSB_CUDA(cudaSetDevice(m->device));
    psb_batch_t *b = new psb_batch_t();      // value-initialised: all pointers null, counters zero
    b->m = m;
    b->max_utts = max_utts;
    b->max_frames = max_frames;
    {
        // 6 (default): tensor-core filter + exact rescoring (psb_ptm_tc.cu) where the model allows it, else the scan
        // kernels (psb_ptm.cu); 5: the scan kernels everywhere, the reference the filter is tested against
        const char *v = getenv("PSB_TOPN_VARIANT");
        if (v && strcmp(v, "5") && strcmp(v, "6")) {
            psb_set_error("psb_batch_create: PSB_TOPN_VARIANT=%s is not supported (accepted: 5 = scan kernels, 6 = default)", v);
            delete b;
            return PSB_ERR_ARG;
        }
        b->force_scan = v && !strcmp(v, "5");
        const char *p = getenv("PSB_PIPELINE");         // sub-batches in flight for psb_decode_batch_*
        b->n_pipe = p ? atoi(p) : 0;                   // 0 = auto (see decode_common)
        if (b->n_pipe < 0) b->n_pipe = 0;
        if (b->n_pipe > 8) b->n_pipe = 8;
    }
    cudaError_t e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&b->d_feats, (size_t)max_frames * m->sumlen * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_senscr, (size_t)max_frames * m->n_sen * sizeof(int16_t));
    if (e == cudaSuccess && m->kind != PSB_KIND_MS) e = cudaMalloc(&b->d_topn, (size_t)max_frames * m->K * sizeof(int4));
    for (int i = 0; i < 4 && e == cudaSuccess; ++i) e = cudaEventCreate(&b->ev[i]);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) e = cudaEventCreate(&b->tev[i]);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->fork_ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->join_ev, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        psb_set_error("psb_batch_create: %s", cudaGetErrorString(e));
        psb_batch_free(b);
        return e == cudaErrorMemoryAllocation ? PSB_ERR_NOMEM : PSB_ERR_CUDA;
    }
    b->have_ev = true;
    *out = b;
    return PSB_OK;
}

extern "C" void psb_batch_free(psb_batch_t *b)
{
    if (!b) return;
    cudaSetDevice(b->m->device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    for (psb_batch_t *k : b->kids) {            // sub-batches own only their stream, tables, featT, events
        cudaStreamSynchronize(k->stream);
        if (k->h_off) cudaFreeHost(k->h_off);
        cudaFree(k->d_featT); cudaFree(k->d_tab); cudaFree(k->d_off); cudaFree(k->d_msdist); cudaFree(k->d_msbest);
        cudaFree(k->d_uttoff); cudaFree(k->d_semi_dist); cudaFree(k->d_tc_flags); cudaFree(k->d_tc_check); cudaFree(k->d_tc_items); cudaFree(k->d_tc_nitems);
        if (k->h_tab) cudaFreeHost(k->h_tab);
        for (int i = 0; i < 4; ++i) cudaEventDestroy(k->ev[i]);
        cudaEventDestroy(k->join_ev);
        cudaStreamDestroy(k->stream);
        delete k;
    }
    if (b->fork_ev) cudaEventDestroy(b->fork_ev);
    if (b->join_ev) cudaEventDestroy(b->join_ev);
    cudaFree(b->d_feats); cudaFree(b->d_senscr); cudaFree(b->d_featT); cudaFree(b->d_topn); cudaFree(b->d_tab); cudaFree(b->d_semi_dist); cudaFree(b->d_uttoff);
    cudaFree(b->d_best); cudaFree(b->d_pen); cudaFree(b->d_off); cudaFree(b->d_msdist); cudaFree(b->d_msbest);
    cudaFree(b->d_tc_flags); cudaFree(b->d_tc_check); cudaFree(b->d_tc_items); cudaFree(b->d_tc_nitems);
    if (b->h_tab) cudaFreeHost(b->h_tab);
    if (b->h_feats) cudaFreeHost(b->h_feats);
    if (b->h_senscr) cudaFreeHost(b->h_senscr);
    if (b->h_best) cudaFreeHost(b->h_best);
    if (b->h_pen) cudaFreeHost(b->h_pen);
    if (b->have_ev) for (int i = 0; i < 4; ++i) cudaEventDestroy(b->ev[i]);
    if (b->have_ev) for (int i = 0; i < 2; ++i) cudaEventDestroy(b->tev[i]);
    if (b->stream) cudaStreamDestroy(b->stream);
    delete b;
}

static int score_dispatch(psb_batch_t *b, const float *d_feats, const int32_t *utt_off, int32_t n_utt,
                          int16_t *d_senscr)
{
    switch (b->m->kind) {
    case PSB_KIND_PTM:
    case PSB_KIND_SEMI:
        return psb_launch_ptm_batch(b, d_feats, utt_off, n_utt, d_senscr);
    case PSB_KIND_MS:
        return psb_launch_ms_batch(b, d_feats, utt_off, n_utt, d_senscr);
    default:
        psb_set_error("batched scoring for model kind %d is not built yet", b->m->kind);
        return PSB_ERR_ARG;
    }
}

static int check_offsets(const psb_batch_t *b, const int32_t *utt_off, int32_t n_utt)
{
    PSB_REQUIRE(utt_off && n_utt >= 0, "bad utt_off / n_utt");
    PSB_REQUIRE(utt_off[0] == 0, "utt_off[0] must be 0");
    for (int u = 0; u < n_utt; ++u)
        PSB_REQUIRE(utt_off[u + 1] >= utt_off[u], "utt_off must be non-decreasing");
    PSB_REQUIRE(n_utt <= b->max_utts && utt_off[n_utt] <= b->max_frames, "batch exceeds psb_batch_create limits");
    return PSB_OK;
}

extern "C" int psb_batch_score_device(psb_batch_t *b, const float *d_feats, const int32_t *utt_off,
                                      int32_t n_utt, int16_t *d_senscr)
{
    PSB_REQUIRE(b, "psb_batch_score_device: null batch");
    int rc = check_offsets(b, utt_off, n_utt);
    if (rc) return rc;
    PSB_REQUIRE(utt_off[n_utt] == 0 || d_feats, "psb_batch_score_device: null buffer");
    PSB_CUDA(cudaSetDevice(b->m->device));
    b->last_pipelined = false;
    return score_dispatch(b, d_feats, utt_off, n_utt, d_senscr ? d_senscr : b->d_senscr);
}

extern "C" int psb_batch_score_host(psb_batch_t *b, const float *feats, const int32_t *utt_off,
                                    int32_t n_utt, int16_t *senscr)
{
    PSB_REQUIRE(b, "psb_batch_score_host: null batch");
    int rc = check_offsets(b, utt_off, n_utt);
    if (rc) return rc;
    PSB_REQUIRE(utt_off[n_utt] == 0 || (feats && senscr), "psb_batch_score_host: null buffer");
    PSB_CUDA(cudaSetDevice(b->m->device));
    const size_t total = utt_off[n_utt];
    if (total == 0) return PSB_OK;
    b->last_pipelined = false;
    PSB_CUDA(cudaMemcpyAsync(b->d_feats, feats, total * b->m->sumlen * sizeof(float), cudaMemcpyHostToDevice, b->stream));
    rc = score_dispatch(b, b->d_feats, utt_off, n_utt, b->d_senscr);
    if (rc) return rc;
    PSB_CUDA(cudaMemcpyAsync(senscr, b->d_senscr, total * b->m->n_sen * sizeof(int16_t), cudaMemcpyDeviceToHost, b->stream));
    PSB_CUDA(cudaStreamSynchronize(b->stream));
    return PSB_OK;
}

extern "C" int psb_batch_sync(psb_batch_t *b)
{
    PSB_REQUIRE(b, "psb_batch_sync: null");
    PSB_CUDA(cudaSetDevice(b->m->device));
    PSB_CUDA(cudaStreamSynchronize(b->stream));
    return PSB_OK;
}

extern "C" int16_t *psb_batch_senscr_device(psb_batch_t *b) { return b ? b->d_senscr : nullptr; }

extern "C" int psb_batch_last_kernel_ms(psb_batch_t *b, float *out3)
{
    PSB_REQUIRE(b && out3, "psb_batch_last_kernel_ms: null");
    PSB_CUDA(cudaSetDevice(b->m->device));
    PSB_CUDA(cudaStreamSynchronize(b->stream));
    out3[0] = out3[1] = out3[2] = 0.f;
    if (b->last_pipelined) {
        // pipelined decode: sum of the sub-batches' own kernel intervals (they overlap in time)
        for (int q = 0; q < b->last_kids && q < (int)b->kids.size(); ++q)
            for (int i = 0; i < 3; ++i) {
                psb_batch_t *k = b->kids[q];
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, k->ev[i], k->ev[i + 1]) == cudaSuccess) out3[i] += ms;
                else cudaGetLastError();
            }
        return PSB_OK;
    }
    for (int i = 0; i < 3; ++i) PSB_CUDA(cudaEventElapsedTime(&out3[i], b->ev[i], b->ev[i + 1]));
    return PSB_OK;
}

extern "C" int psb_batch_get_topn(psb_batch_t *b, int32_t *rec, int64_t n_frames)
{
    PSB_REQUIRE(b && rec && n_frames >= 0 && n_frames <= b->max_frames, "psb_batch_get_topn: bad argument");
    PSB_REQUIRE(b->d_topn, "psb_batch_get_topn: this model kind keeps no top-N records");
    PSB_CUDA(cudaSetDevice(b->m->device));
    PSB_CUDA(cudaStreamSynchronize(b->stream));
    PSB_CUDA(cudaMemcpy(rec, b->d_topn, (size_t)n_frames * b->m->K * sizeof(int4), cudaMemcpyDeviceToHost));
    return PSB_OK;
}

cudaStream_t psb_batch_stream(psb_batch_t *b) { return b->stream; }

// One sub-batch of the pipelined decode: a light psb_batch_t with its own stream, tables and
// lane-major feature copy, pointing into the parent's big buffers.
static int get_kid(psb_batch_t *b, int i, psb_batch_t **out)
{
    while ((int)b->kids.size() <= i) {
        psb_batch_t *k = new psb_batch_t();
        k->m = b->m; k->max_utts = b->max_utts; k->max_frames = b->max_frames; k->force_scan = b->force_scan;
        k->is_kid = true; k->n_pipe = 1;
        cudaError_t e = cudaStreamCreateWithFlags(&k->stream, cudaStreamNonBlocking);
        for (int j = 0; j < 4 && e == cudaSuccess; ++j) e = cudaEventCreate(&k->ev[j]);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&k->join_ev, cudaEventDisableTiming);
        if (e != cudaSuccess) {
            psb_set_error("pipelined decode: %s", cudaGetErrorString(e));
            delete k;
            return PSB_ERR_CUDA;
        }
        k->have_ev = true;
        b->kids.push_back(k);
    }
    *out = b->kids[i];
    return PSB_OK;
}

// Shared by the host and device decode entry points.  The batch is cut into n_pipe contiguous
// utterance ranges of about equal frame counts; each range runs copy-in -> transpose -> top-N ->
// senone -> phone loop -> copy-out on its own stream, so the FP32-bound top-N kernel of one
// range overlaps the integer/LSU-bound senone kernel and the PCIe copies of the others.  The
// parent's stream forks into and joins the sub-streams with events, so psb_batch_event_record /
// psb_batch_sync on the parent still bracket all the work.
static int decode_common_body(psb_batch_t *b, psb_phoneloop_t *p, const float *feats, bool feats_on_host,
                              const int32_t *utt_off, int32_t n_utt, int32_t *h_best, int32_t *h_pen, int16_t *h_senscr,
                              bool want_best, bool want_pen);

// An error in the middle of the loop over sub-batches leaves earlier sub-streams with copies into the
// caller's host buffers in flight: drain every stream before handing the error back.
static int decode_common(psb_batch_t *b, psb_phoneloop_t *p, const float *feats, bool feats_on_host,
                         const int32_t *utt_off, int32_t n_utt, int32_t *h_best, int32_t *h_pen, int16_t *h_senscr,
                         bool want_best, bool want_pen)
{
    const int rc = decode_common_body(b, p, feats, feats_on_host, utt_off, n_utt, h_best, h_pen, h_senscr, want_best, want_pen);
    if (rc != PSB_OK) {
        for (psb_batch_t *k : b->kids) cudaStreamSynchronize(k->stream);
        cudaStreamSynchronize(b->stream);
    }
    return rc;
}

static int decode_common_body(psb_batch_t *b, psb_phoneloop_t *p, const float *feats, bool feats_on_host,
                              const int32_t *utt_off, int32_t n_utt, int32_t *h_best, int32_t *h_pen, int16_t *h_senscr,
                              bool want_best, bool want_pen)
{
    psb_model_t *m = b->m;
    const size_t H = psb_phoneloop_n_phones(p);
    const long long total = utt_off[n_utt];
    if ((size_t)b->max_frames * H > b->pen_cap) {
        cudaFree(b->d_best); cudaFree(b->d_pen);
        b->d_best = b->d_pen = nullptr;
        b->pen_cap = (size_t)b->max_frames * H;
        PSB_CUDA(cudaMalloc(&b->d_best, (size_t)b->max_frames * 4));
        PSB_CUDA(cudaMalloc(&b->d_pen, b->pen_cap * 4));
    }
    // auto: two ranges when the features come from the host (the copies of one overlap the
    // kernels of the other), one when they are resident (measured on B200 at 1000 x 10 s: two
    // concurrent top-N kernels only add launch/tail overhead, 110 ms vs 105 ms per step)
    const int want = b->n_pipe > 0 ? b->n_pipe : (feats_on_host ? 2 : 1);
    const int S = std::max(1, std::min<int>(want, n_utt));
    PSB_CUDA(cudaEventRecord(b->fork_ev, b->stream));
    int u0 = 0;
    for (int s = 0; s < S; ++s) {
        // utterances [u0, u1) with about total/S frames
        int u1 = u0;
        const long long target = total * (s + 1) / S;
        while (u1 < n_utt && (utt_off[u1 + 1] <= target || u1 == u0)) ++u1;
        if (s == S - 1) u1 = n_utt;
        if (u1 == u0) continue;
        psb_batch_t *k;
        int rc = get_kid(b, s, &k);
        if (rc) return rc;
        const long long f0 = utt_off[u0], nf = utt_off[u1] - f0;
        const int nu = u1 - u0;
        if ((size_t)nu + 1 > k->off_cap) {
            cudaFree(k->d_off);
            if (k->h_off) cudaFreeHost(k->h_off);
            k->d_off = nullptr; k->h_off = nullptr;
            k->off_cap = (size_t)nu + 1 + 256;
            PSB_CUDA(cudaMalloc(&k->d_off, k->off_cap * 4));
            PSB_CUDA(cudaMallocHost(&k->h_off, k->off_cap * 4));
        }
        PSB_CUDA(cudaStreamSynchronize(k->stream));          // the previous call's copy from h_off is done
        int32_t *off = k->h_off;
        for (int i = 0; i <= nu; ++i) off[i] = utt_off[u0 + i] - (int32_t)f0;
        PSB_CUDA(cudaStreamWaitEvent(k->stream, b->fork_ev, 0));
        const float *d_f = feats + f0 * m->sumlen;
        if (feats_on_host) {
            PSB_CUDA(cudaMemcpyAsync(b->d_feats + f0 * m->sumlen, feats + f0 * m->sumlen, (size_t)nf * m->sumlen * sizeof(float),
                                     cudaMemcpyHostToDevice, k->stream));
            d_f = b->d_feats + f0 * m->sumlen;
        }
        PSB_CUDA(cudaMemcpyAsync(k->d_off, off, (size_t)(nu + 1) * 4, cudaMemcpyHostToDevice, k->stream));
        k->d_topn = b->d_topn ? b->d_topn + f0 * m->K : nullptr;
        rc = score_dispatch(k, d_f, off, nu, b->d_senscr + f0 * m->n_sen);
        if (rc) return rc;
        rc = psb_phoneloop_launch(p, b->d_senscr + f0 * m->n_sen, k->d_off, nu, want_best ? b->d_best + f0 : nullptr,
                                  want_pen ? b->d_pen + f0 * H : nullptr, nullptr, nullptr, k->stream);
        if (rc) return rc;
        if (h_best) PSB_CUDA(cudaMemcpyAsync(h_best + f0, b->d_best + f0, (size_t)nf * 4, cudaMemcpyDeviceToHost, k->stream));
        if (h_pen) PSB_CUDA(cudaMemcpyAsync(h_pen + f0 * H, b->d_pen + f0 * H, (size_t)nf * H * 4, cudaMemcpyDeviceToHost, k->stream));
        if (h_senscr)
            PSB_CUDA(cudaMemcpyAsync(h_senscr + f0 * m->n_sen, b->d_senscr + f0 * m->n_sen, (size_t)nf * m->n_sen * 2,
                                     cudaMemcpyDeviceToHost, k->stream));
        PSB_CUDA(cudaEventRecord(k->join_ev, k->stream));
        PSB_CUDA(cudaStreamWaitEvent(b->stream, k->join_ev, 0));
        u0 = u1;
    }
    b->last_frames = total;
    b->last_pipelined = true;
    b->last_kids = S;
    return PSB_OK;
}

// End-to-end: host features -> senone scores -> phone-loop Viterbi -> host results.
extern "C" int psb_decode_batch_host(psb_batch_t *b, psb_phoneloop_t *p, const float *feats, const int32_t *utt_off,
                                     int32_t n_utt, int32_t *best, int32_t *pen, int16_t *senscr)
{
    PSB_REQUIRE(b && p, "psb_decode_batch_host: null handle");
    int rc = check_offsets(b, utt_off, n_utt);
    if (rc) return rc;
    PSB_REQUIRE(utt_off[n_utt] == 0 || feats, "psb_decode_batch_host: null buffer");
    PSB_CUDA(cudaSetDevice(b->m->device));
    if (utt_off[n_utt] == 0) return PSB_OK;
    rc = decode_common(b, p, feats, true, utt_off, n_utt, best, pen, senscr, best != nullptr, pen != nullptr);
    if (rc) return rc;
    PSB_CUDA(cudaStreamSynchronize(b->stream));
    return PSB_OK;
}

extern "C" int psb_decode_batch_device(psb_batch_t *b, psb_phoneloop_t *p, const float *d_feats, const int32_t *utt_off,
                                       int32_t n_utt, int32_t **d_best, int32_t **d_pen)
{
    PSB_REQUIRE(b && p, "psb_decode_batch_device: null handle");
    int rc = check_offsets(b, utt_off, n_utt);
    if (rc) return rc;
    PSB_REQUIRE(utt_off[n_utt] == 0 || d_feats, "psb_decode_batch_device: null buffer");
    PSB_CUDA(cudaSetDevice(b->m->device));
    if (utt_off[n_utt] == 0) return PSB_OK;
    rc = decode_common(b, p, d_feats, false, utt_off, n_utt, nullptr, nullptr, nullptr, true, true);
    if (d_best) *d_best = b->d_best;
    if (d_pen) *d_pen = b->d_pen;
    return rc;
}

// From audio: int16 PCM -> device front end (psb_fe.cu) -> senone scores -> phone loop, host results.
// The features never leave the device.
extern "C" int psb_decode_batch_pcm_host(psb_batch_t *b, psb_fe_t *fe, psb_phoneloop_t *p, const int16_t *pcm,
                                         const int64_t *samp_off, int32_t n_utt, int32_t *frame_off, int32_t *best,
                                         int32_t *pen, int16_t *senscr)
{
    PSB_REQUIRE(b && fe && p && samp_off && frame_off && n_utt >= 0, "psb_decode_batch_pcm_host: bad argument");
    PSB_REQUIRE(psb_fe_feat_dim(fe) == b->m->sumlen, "psb_decode_batch_pcm_host: the front end makes %d-dimensional features, the model wants %d",
                psb_fe_feat_dim(fe), b->m->sumlen);
    int rc = psb_fe_process_host(fe, pcm, samp_off, n_utt, nullptr, nullptr, frame_off);
    if (rc) return rc;
    rc = check_offsets(b, frame_off, n_utt);
    if (rc) return rc;
    PSB_CUDA(cudaSetDevice(b->m->device));
    if (frame_off[n_utt] == 0) return PSB_OK;
    rc = decode_common(b, p, psb_fe_device_feats(fe), false, frame_off, n_utt, best, pen, senscr, best != nullptr, pen != nullptr);
    if (rc) return rc;
    PSB_CUDA(cudaStreamSynchronize(b->stream));
    return PSB_OK;
}

extern "C" int psb_batch_event_record(psb_batch_t *b, int slot)
{
    PSB_REQUIRE(b && (slot == 0 || slot == 1), "psb_batch_event_record: bad argument");
    PSB_CUDA(cudaSetDevice(b->m->device));
    PSB_CUDA(cudaEventRecord(b->tev[slot], b->stream));
    return PSB_OK;
}

extern "C" int psb_batch_event_elapsed_ms(psb_batch_t *b, float *ms)
{
    PSB_REQUIRE(b && ms, "psb_batch_event_elapsed_ms: bad argument");
    PSB_CUDA(cudaSetDevice(b->m->device));
    PSB_CUDA(cudaEventSynchronize(b->tev[1]));
    PSB_CUDA(cudaEventElapsedTime(ms, b->tev[0], b->tev[1]));
    return PSB_OK;
}

extern "C" int psb_batch_set_pipeline(psb_batch_t *b, int n)
{
    PSB_REQUIRE(b && n >= 0 && n <= 8, "psb_batch_set_pipeline: n must be 0 (auto) or 1..8");
    b->n_pipe = n;
    return PSB_OK;
}
