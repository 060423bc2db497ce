#!/usr/bin/env python
"""bench.py -- frames/sec of the PocketSphinx hot path (senone evaluation + Viterbi) on B200.

One "step" = one pass of the hot path over one batch of synthetic utterances: GMM senone
evaluation of every frame (all senones, like `-compallsen yes`), the phone-loop Viterbi
(phone_loop_search.c: every CI-phone HMM through hmm_vit_eval each frame, beam pruning, phone
transitions, look-ahead penalties) and the SEARCH-SCALE Viterbi over the freshly computed scores:
every utterance keeps N_ACTIVE = 6 081 hmm_t instances alive (what SURVEY 8d measured per frame for
the en-us fwdtree search at default beams) and all of them take one hmm_vit_eval step per frame
with a per-frame best-score reduction -- evaluate_channels (ngram_search_fwdtree.c:702-715).  Both
arms run all three stages: ours on the device, the reference arm through the compiled reference's
ptm_mgau_frame_eval and hmm_vit_eval on the host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--model baseline|en-us] [--utts U] [--secs S] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for what each key means.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from pocketsphinx_b200.model import PackedModel, synth_feats, synth_ms, synth_ptm, synth_semi  # noqa: E402

FRAMES_PER_SEC_AUDIO = 100          # 10 ms frames
PL = dict(window=5, beam=-225, pbeam=-225, pip=0, weight=3.0)   # pl_beam 1e-10 etc. >> 10
N_ACTIVE = 6081                     # active HMMs per frame, en-us fwdtree at default beams (SURVEY 8d)


def channel_template(pm, HMM_DTYPE, n_active=N_ACTIVE):
    """The search-scale Viterbi's active set, the same on both arms: n_active non-multiplexed hmm_t drawn
    from the model's senone sequences and transition matrices, all entered at frame 0 with score 0
    (hmm_enter).  Returns None when the model has no 3-/5-state topology to evaluate."""
    if pm.n_emit_state not in (3, 5) or len(pm.sseq) == 0:
        return None
    ns = pm.n_emit_state
    rng = np.random.default_rng(99)
    hm = np.zeros(n_active, HMM_DTYPE)
    ssid = rng.integers(0, len(pm.sseq), n_active)
    hm["score"][:, :] = -0x20000000
    hm["score"][:, 0] = 0
    hm["history"][:, :] = -1
    hm["out_score"] = -0x20000000
    hm["out_history"] = -1
    hm["bestscore"] = -0x20000000
    hm["ssid"] = ssid
    hm["senid"][:, :ns] = pm.sseq[ssid]
    hm["tmatid"] = rng.integers(0, pm.tp.shape[0], n_active)
    hm["n_emit_state"] = ns
    return hm


def frames_for(secs):
    # fe/ with 25.6 ms windows and 10 ms shift: 10 s of 16 kHz audio -> 998 frames
    return max(1, int(secs * FRAMES_PER_SEC_AUDIO) - 2)


def load_model(name):
    """Returns (PackedModel, description, raw parameters or None)."""
    if name == "baseline":
        pm, raw = synth_ptm(seed=0, n_density=256, n_sen=5138, return_raw=True)
        return pm, "synthetic PTM 42x3x256x13, 5138 senones (BASELINE.json shape)", raw
    if name == "en-us":
        pm = PackedModel.load(os.path.join(ROOT, "tests", "golden", "en_us_ptm_model.npz"))
        return pm, "shipped en-us PTM 42x3x128x13, 5126 senones (packed fixture)", None
    if name == "semi":       # BASELINE.json config 3: semi-continuous, 1 codebook x 4 streams x 256, 5138 senones
        pm, raw = synth_semi(seed=0, n_density=256, n_sen=5138, return_raw=True)
        pm.n_ciphone, pm.n_ci_sen = 42, 126
        pm.sseq = np.arange(126, dtype=np.uint16).reshape(42, 3)
        pm.phone_ssid, pm.phone_tmat = np.arange(42, dtype=np.int32), np.arange(42, dtype=np.int32) % 10
        return pm, "synthetic semi-continuous 1x4x256x{12,24,3,12}, 5138 senones (BASELINE.json config 3 shape)", raw
    if name == "cont":       # BASELINE.json config 4: continuous, 8 Gaussians/senone x 39 dims, 5138 senones
        pm, raw = synth_ms(seed=0, n_sen=5138, n_density=8, featlens=(39,), topn=4, return_raw=True)
        pm.n_ciphone, pm.n_ci_sen = 42, 126
        pm.sseq = np.arange(126, dtype=np.uint16).reshape(42, 3)
        pm.phone_ssid, pm.phone_tmat = np.arange(42, dtype=np.int32), np.arange(42, dtype=np.int32) % 10
        return pm, "synthetic continuous ms 5138 senones x 8 Gaussians x 39 dims, topn 4 (BASELINE.json config 4 shape)", raw
    raise SystemExit("unknown --model " + name)


_REF_DIR = None


def reference_model_dir(name, pm, raw):
    """A model directory the compiled reference (oracle/_ref/libpsref.so) can load, or None."""
    global _REF_DIR
    from oracle import refdrv
    if not refdrv.available():
        return None
    if name == "en-us":
        d = os.path.join(ROOT, "oracle", "_ref", "model", "en-us")
        return d if os.path.isdir(d) else None
    if _REF_DIR is None:
        import tempfile
        from pocketsphinx_b200 import s3io
        _REF_DIR = tempfile.mkdtemp(prefix="psb200_model_")
        if pm.kind == "ptm":
            sen2ci, n_ci = pm.sen2cb, pm.n_mgau
            fp = "-feat 1s_c_d_dd\n-svspec 0-12/13-25/26-38\n-cmn batch\n-agc none\n"
        else:                            # semi-continuous / continuous: 42 CI phones x 3 states, the rest tied round-robin
            sen2ci = np.concatenate([np.repeat(np.arange(42), 3), np.arange(pm.n_sen - 126) % 42]).astype(np.int32)
            n_ci = 42
            fp = "-feat s2_4x\n-cmn batch\n-agc none\n" if pm.kind == "s2_semi" else "-feat 1s_c_d_dd\n-cmn batch\n-agc none\n"
        s3io.write_model_dir(_REF_DIR, kind=pm.kind, n_mgau=pm.n_mgau, n_feat=pm.n_feat, n_density=pm.n_density,
                             featlen=pm.featlen, mean=raw["mean"], var_raw=raw["var_raw"], tp_float=raw["tp_float"],
                             sen2ci=sen2ci, n_ci=n_ci, n_emit=3, n_ci_sen=n_ci * 3,
                             mixw_q=raw.get("mixw_q"), mixw_cb=raw.get("mixw_cb"), mixw_float=raw.get("mixw_float"),
                             feat_params=fp)
    return _REF_DIR


def ncu_traffic(kernel, workload):
    """DRAM bytes per launch of `kernel` at `workload` from a committed ncu capture, or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as f:
            return json.load(f).get(kernel + "|" + workload)
    except (OSError, ValueError):
        return None


def tensor_peak_bf16():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["bf16_tflops"])
    except (OSError, ValueError, KeyError):
        return 2250.0                                          # nominal dense bf16 (B200_PROFILING.md)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def viterbi_stage(api, torch, ctx, batch, pm, off, U, T, hbm_peak, n_active=6081, n_frames=48):
    """Stage-wise Viterbi number (SURVEY 8d): every utterance keeps n_active hmm_t instances alive
    (the survey measured 6 081 active HMMs per frame for en-us fwdtree at default beams), all of
    them take one hmm_vit_eval step per frame against that frame's senone scores (the ones the
    GMM stage just left in HBM) with a per-utterance best-score reduction: evaluate_channels
    (ngram_search_fwdtree.c:702-715) for a whole batch, state resident in HBM as SoA.  Which HMMs
    are active is the search's business (row f-1, not built): instances are drawn at random from
    the model's senone sequences, all entered at frame 0."""
    if pm.n_emit_state not in (3, 5) or len(pm.sseq) == 0:
        return None
    ns = pm.n_emit_state
    rng = np.random.default_rng(99)
    n = U * n_active
    hm = np.zeros(n, api.HMM_DTYPE)
    ssid = rng.integers(0, len(pm.sseq), n)
    hm["score"][:, :] = -0x20000000
    hm["score"][:, 0] = 0                                      # hmm_enter(score 0, history -1, frame 0)
    hm["history"][:, :] = -1
    hm["out_score"] = -0x20000000
    hm["out_history"] = -1
    hm["bestscore"] = -0x20000000
    hm["ssid"] = ssid
    hm["senid"][:, :ns] = pm.sseq[ssid]
    hm["tmatid"] = rng.integers(0, pm.tp.shape[0], n)
    hm["n_emit_state"] = ns
    hs = api.HmmSet(ctx, n + U * 512, U)                       # slack: segments start on storage-tile boundaries
    hs.upload(hm, np.arange(U + 1, dtype=np.int64) * n_active)
    F = min(n_frames, T)
    d_row0 = torch.from_numpy(np.asarray(off[:U], np.int64)).cuda()
    d_best = torch.empty((F, U), dtype=torch.int32, device="cuda")
    hs.eval_frames_device(batch.senscr_device_ptr(), 3, d_best.data_ptr(), d_row0=d_row0.data_ptr())   # warm-up
    ms = hs.eval_frames_device(batch.senscr_device_ptr(), F, d_best.data_ptr(), d_row0=d_row0.data_ptr())
    hs.close()
    # algorithmic bytes per instance and frame: state read + written (score, history per state,
    # exit score + history, best) + senone ids, transition id and the int16 score gathers
    alg = (2 * ns * 4) * 2 + 2 * 4 * 2 + 4 + 2 * ns + 2 + 2 * ns
    gbs = n * alg * F / (ms * 1e-3) / 1e9
    return {"kernel": "hmmset_eval_kernel", "active_hmms_per_utt": n_active, "utts": U, "frames_timed": F,
            "ms_per_frame_of_batch": ms / F, "hmm_updates_per_s": n * F / (ms * 1e-3),
            "frames_per_s": U * F / (ms * 1e-3),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         "algorithmic_bytes_per_hmm": alg},
            "note": "the per-frame kernel (state visible in HBM between frames), for comparison with search_viterbi: "
                    "`value` uses the fused sweep"}


def beam_stage(torch, hs, batch, total, T, U, d_row0, d_nrows, dev):
    """The same search-scale sweep with the beam applied between frames on the device (prune_channels' best score and
    -maxhmmpf histogram, prune_nonroot_chan's keep-or-hmm_clear; one thread-block cluster per utterance, DESIGN 4.19):
    not part of `value` -- the headline's 6 081 instances per frame ARE the reference's post-pruning count -- but timed on
    the scores the timed step just wrote.  -beam 1e-48 is -1080 in score units (logbase 1.0001, >> 10)."""
    d_best = torch.empty((T, U), dtype=torch.int32, device="cuda:%d" % dev)
    d_nact = torch.empty((T, U), dtype=torch.int32, device="cuda:%d" % dev)
    torch.cuda.synchronize()
    res = {"kernel": "hmmset_sweep_kernel<BEAM>", "instances_per_utt_at_frame_0": N_ACTIVE, "runs": {}}
    for name, beam, mh in (("beam_neutral", -0x1fffffff, -1), ("beam_1e-48", -1080, -1), ("beam_1e-48_maxhmmpf_3000", -1080, 3000)):
        hs.restore()
        ms = hs.sweep_beam_device(batch.senscr_device_ptr(), total, T, 0, beam, d_best.data_ptr(), maxhmmpf=mh,
                                  d_n_active=d_nact.data_ptr(), d_row0=d_row0.data_ptr(), d_n_rows=d_nrows.data_ptr(), timed=True)
        na = d_nact.float().mean(dim=1).cpu().numpy()
        res["runs"][name] = {"beam": beam, "maxhmmpf": mh, "ms": ms, "active_mean": float(na.mean()), "active_frame_1": float(na[1]) if T > 1 else None,
                             "active_last": float(na[-1])}
    hs.restore()
    return res


def align_stage(api, ctx, batch, pm, off, U, T, n_phones=100):
    """Batched forced alignment (state_align_search.c) over the scores the GMM stage left in HBM:
    every utterance is aligned to its own chain of n_phones phones (random senone sequences; a 10 s
    utterance has about that many).  Wall clock of the whole call: phone upload, the kernel (one CTA
    per utterance, token table in HBM), backtrace, state-level result download."""
    rng = np.random.default_rng(5)
    ph_off = np.arange(U + 1, dtype=np.int32) * n_phones
    ssid = rng.integers(0, len(pm.sseq), U * n_phones).astype(np.int32)
    tmat = rng.integers(0, pm.tp.shape[0], U * n_phones).astype(np.int32)
    ctx.align(None, off, ph_off, ssid, tmat, device_ptr=batch.senscr_device_ptr())       # warm-up
    t0 = time.perf_counter()
    status, st, du, sc = ctx.align(None, off, ph_off, ssid, tmat, device_ptr=batch.senscr_device_ptr())
    dt = time.perf_counter() - t0
    return {"kernel": "align_kernel", "utts": U, "phones_per_utt": n_phones, "ms": dt * 1e3,
            "kernel_ms": api.lib().psb_align_last_kernel_ms(ctx.h),
            "frames_per_s": U * T / dt, "aligned_ok": int((status == 0).sum()),
            "note": "not part of `value`; bit-exact vs the reference's state_align_search (tests)"}


def frontend_stage(api, torch, U, secs, budget_s=4.0):
    """Row f-2, reported beside the headline (not part of `value`): int16 PCM -> cepstra -> batch CMN
    -> 1s_c_d_dd features for the whole batch on the device (en-us feat.params: 25 mel filters,
    DCT-II, lifter 22, noise removal on), against the compiled reference's fe/ + feat/ on one core."""
    from pocketsphinx_b200.fe_tables import make_fe_desc
    desc = make_fe_desc()
    n = int(secs * 16000)
    rng = np.random.default_rng(7)
    base = np.clip(rng.normal(0, 2500, (16, n)), -32768, 32767).astype(np.int16)      # 16 distinct utterances, tiled
    pcm = np.ascontiguousarray(np.tile(base, ((U + 15) // 16, 1))[:U]).reshape(-1)
    off = np.arange(U + 1, dtype=np.int64) * n
    fe = api.FrontEnd(desc)
    T = fe.n_frames(n)
    d_pcm = torch.from_numpy(pcm).cuda()
    d_feats = torch.empty((U * T, 3 * desc["n_cep"]), dtype=torch.float32, device="cuda")
    fe.process_device(d_pcm.data_ptr(), off, d_feats.data_ptr())
    ms = min(fe.process_device(d_pcm.data_ptr(), off, d_feats.data_ptr())[1] for _ in range(3))
    fe.close()
    out = {"kernels": "fe_frame_kernel + fe_utt_kernel", "utts": U, "frames_per_utt": T, "ms": ms,
           "frames_per_s": U * T / (ms * 1e-3),
           "algorithmic_bytes": int(pcm.nbytes + U * T * 3 * desc["n_cep"] * 4),
           "note": "not part of `value`; parity with the reference at 1e-4 relative (tests/test_gpu_fe.py)"}
    try:
        from oracle import refdrv
        if refdrv.available():
            ref = refdrv.RefModel(os.path.join(os.path.dirname(refdrv.LIB_PATH), "model", "en-us"))
            t0, k = time.perf_counter(), 0
            while time.perf_counter() - t0 < budget_s:
                ref.featurize_fresh(base[k % 16])
                k += 1
            out["cpu_reference_frames_per_s_1core"] = k * T / (time.perf_counter() - t0)
            ref.close()
    except Exception as e:                                  # the CPU side is informational only
        out["cpu_reference_error"] = str(e)[:100]
    return out


def search_stage(api, torch, U=256):
    """Rows f-1 / f-4, reported beside the headline (not part of `value`): the three search kernels (fsg_search_kernel, ngs_fwdtree_kernel, ngs_fwdflat_kernel) over U copies
    of the reference's own utterance (goforward.raw: its golden senone scores, its flattened grammar /
    lextree / turtle LM from tests/golden/), wall clock of each call including table download, with the
    first utterance's tables compared against the reference's golden ones."""
    here = os.path.dirname(os.path.abspath(__file__))
    gd = os.path.join(here, "tests", "golden")
    m = np.load(os.path.join(gd, "en_us_ptm_model.npz"))
    gf = np.load(os.path.join(gd, "en_us_goforward.npz"))
    scr = gf["senscr"]
    T = len(scr)
    d_scr = torch.from_numpy(np.ascontiguousarray(np.tile(scr, (U, 1)))).cuda()
    off = (np.arange(U + 1, dtype=np.int64) * T).astype(np.int32)
    ctx = api.HmmContext(m["tp"], m["sseq"], int(m["n_sen"]))
    out = {"utts": U, "frames_per_utt": T, "note": "the searches over U copies of the reference utterance; not part of `value`"}

    def case(g, tag):
        return {k[len(tag) + 1:]: g[k] for k in g.files if k.startswith(tag + ".")}

    def timed(fn):
        fn()
        t0 = time.perf_counter()
        r = fn()
        return r, time.perf_counter() - t0
    c = case(np.load(os.path.join(gd, "en_us_fsg.npz")), "cmd")
    (hist, n), dt = timed(lambda: ctx.fsg(d_scr.data_ptr(), off, c, len(c["hist"]) + 64))
    out["fsg"] = {"kernel": "fsg_search_kernel", "pnodes": int(len(c["pnodes"])), "ms": dt * 1e3, "utts_per_s": U / dt,
                  "frames_per_s": U * T / dt, "matches_reference": bool(np.array_equal(hist[0], c["hist"]) and (n == n[0]).all())}
    c = case(np.load(os.path.join(gd, "en_us_fwdtree.npz")), "flat_default")
    first_ref = case(np.load(os.path.join(gd, "en_us_fwdtree.npz")), "lookahead")
    nci = int(c["info"][6])
    cit, cis = m["phone_tmat"][:nci], m["phone_ssid"][:nci]
    win = int(gf["pl_params"][4])
    d_pen = torch.from_numpy(np.ascontiguousarray(np.tile(gf["pl_pen"].astype(np.int32), (U, 1)))).cuda()
    first, dt1 = timed(lambda: ctx.ngram_fwdtree(d_scr.data_ptr(), off, c["info"], c["model"], cit, 2048, 1 << 15, d_pen.data_ptr(), win))
    out["fwdtree"] = {"kernel": "ngs_fwdtree_kernel", "channels": int(c["info"][2] + c["info"][3]), "ms": dt1 * 1e3,
                      "utts_per_s": U / dt1, "frames_per_s": U * T / dt1,
                      "matches_reference": bool(np.array_equal(first[0][0], first_ref["bp"]))}
    tabs = [f[0] for f in first]
    second, dt2 = timed(lambda: ctx.ngram_fwdflat(d_scr.data_ptr(), off, c["info"], c["model"], cit, cis, tabs, 2048, 1 << 15))
    out["fwdflat"] = {"kernel": "ngs_fwdflat_kernel", "ms": dt2 * 1e3, "utts_per_s": U / dt2, "frames_per_s": U * T / dt2,
                      "matches_reference": bool(np.array_equal(second[0][0], c["bp"]))}
    (both, n_first), dt3 = timed(lambda: ctx.ngram_two_pass(d_scr.data_ptr(), off, c["info"], c["model"], cit, cis, 2048, 1 << 15,
                                                             d_pen.data_ptr(), win, first_cap=2048, first_bss_cap=1 << 15))
    out["two_pass"] = {"call": "psb_ngram_two_pass_batch_device", "ms": dt3 * 1e3, "utts_per_s": U / dt3, "frames_per_s": U * T / dt3,
                       "matches_reference": bool(np.array_equal(both[0][0], c["bp"]) and np.array_equal(both[U - 1][0], c["bp"]))}
    try:                                               # the words, read from the tables alone (psb_result.cu)
        dflt = case(np.load(os.path.join(gd, "en_us_fwdtree.npz")), "default")
        vocab, words = str(dflt["vocab"]).split("\n"), dflt["words"]
        t0 = time.perf_counter()
        hyps = []
        for bp, bss, idx in both:
            entry, _, seg = api.ngram_hyp(bp, idx, T, int(c["info"][20]))
            hyps.append(" ".join(vocab[int(words[w][5])] for w in seg[:, 1]
                                 if not words[w][4] and int(words[w][5]) not in (int(c["info"][19]), int(c["info"][20]))))
        out["two_pass"]["hyp"] = hyps[0]
        out["two_pass"]["all_utts_same_hyp"] = bool(all(h == hyps[0] for h in hyps))
        out["two_pass"]["hyp_extraction_ms"] = (time.perf_counter() - t0) * 1e3
    except Exception as e:
        out["two_pass"]["hyp_error"] = str(e)[:100]
    ctx.close()
    try:
        from oracle import refdrv
        lm = os.path.join(os.path.dirname(refdrv.LIB_PATH), "data", "turtle.lm.bin")
        if refdrv.available() and os.path.exists(lm):
            rd = os.path.dirname(refdrv.LIB_PATH)
            pcm = np.fromfile(os.path.join(rd, "data", "goforward.raw"), np.int16)
            t0 = time.perf_counter()
            refdrv.decode(os.path.join(rd, "model", "en-us"), lm, os.path.join(rd, "data", "turtle.dic"), pcm, bestpath="no")
            out["cpu_reference_full_decode_ms_1core"] = (time.perf_counter() - t0) * 1e3      # init + GMM + both passes
    except Exception as e:
        out["cpu_reference_error"] = str(e)[:100]
    return out


def search_coupled_stage(api, torch, batch, pm, off, U, T, kind, gmm_ms_per_frame):
    """BASELINE configs 3 / 4 as written: the GMM stage of THIS model feeding a search kernel over the scores it just left in
    HBM -- `fwdtree` (config 3: n-gram first pass) or `fsg` (config 4: grammar search).  The search description is the
    reference's own flattened lextree / grammar for its test LM and grammar (tests/golden/, 5126 senones: any model with at
    least as many senone columns can drive it; the synthetic models' scores make it a load test, not a recognition test).
    Reported beside the headline: frames/s of the search call alone (tables downloaded) and of GMM + search in sequence."""
    here = os.path.dirname(os.path.abspath(__file__))
    gd = os.path.join(here, "tests", "golden")
    m = np.load(os.path.join(gd, "en_us_ptm_model.npz"))
    if pm.n_sen < int(m["n_sen"]):
        return {"error": "model has fewer senones than the search description uses"}
    Us = min(U, 256 if kind == "fsg" else 64)          # the first pass's tables: 128 entries per frame allowed on random scores
    offs = np.ascontiguousarray(off[:Us + 1], np.int32)
    ctx = api.HmmContext(m["tp"], m["sseq"], pm.n_sen)

    def case(g, tag):
        return {k[len(tag) + 1:]: g[k] for k in g.files if k.startswith(tag + ".")}
    out = {"search": kind, "utts": Us, "frames_per_utt": T}
    try:
        if kind == "fsg":
            c = case(np.load(os.path.join(gd, "en_us_fsg.npz")), "cmd")
            fn = lambda: ctx.fsg(batch.senscr_device_ptr(), offs, c, 64 * T)
        else:
            c = case(np.load(os.path.join(gd, "en_us_fwdtree.npz")), "default")
            nci = int(c["info"][6])
            fn = lambda: ctx.ngram_fwdtree(batch.senscr_device_ptr(), offs, c["info"], c["model"], m["phone_tmat"][:nci], 128 * T, 128 * T * 32)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        out.update({"search_ms": dt * 1e3, "search_frames_per_s": Us * T / dt,
                    "gmm_plus_search_frames_per_s": 1.0 / (gmm_ms_per_frame * 1e-3 + dt / (Us * T)),
                    "note": "not part of `value`; search call = kernel + table download, wall clock"})
    except Exception as e:
        out["error"] = str(e)[:200]
    ctx.close()
    return out


def cpu_baseline(args, pm, raw, feats, n_frames_per_utt, budget_s=15.0, threads=1):
    """The reference's CPU implementation of the path on host cores over a bounded sample of the
    same workload: senone evaluation through the COMPILED REFERENCE (oracle/_ref/libpsref.so:
    ptm_mgau_frame_eval itself, kind "reference") when it is present, else through the C port
    (oracle/ps_oracle.c, bit-exact vs the reference, kind "port"); the phone loop (<1 % of the
    time) always through the port."""
    import threading as th
    from oracle import oracle, refdrv
    ref_dir = reference_model_dir(args.model, pm, raw)
    kind = "reference" if ref_dir else "port"
    om = oracle.OracleModel(pm)
    local = th.local()
    tmpl = channel_template(pm, oracle.HMM_DTYPE)

    def sweeper():
        # the compiled reference's hmm_vit_eval (hmm.c:787) when it is there, else the port's
        if not hasattr(local, "hctx"):
            local.hctx = refdrv.RefHmmCtx(pm.tp, pm.sseq) if kind == "reference" else oracle.OracleHmmCtx(pm.tp, pm.sseq)
        return local.hctx

    def scorer():
        if kind == "port":
            return om.score_utt
        if not hasattr(local, "ref"):
            kv = {"senmgau": ".cont.", "topn": str(pm.topn)} if pm.kind == "ms" else {}
            local.ref = refdrv.RefModel(ref_dir, **kv)
        return local.ref.score

    # calibrate on one short slice, then size the sample to the budget
    sc = scorer()
    t0 = time.perf_counter()
    sc(feats[0][:64])
    per_frame = max(1e-6, (time.perf_counter() - t0) / 64)
    n_utt = int(max(1, min(len(feats), budget_s * threads / (per_frame * n_frames_per_utt))))
    if n_utt >= threads:
        n_utt -= n_utt % threads
    # a long stream (BASELINE config 5: one 60-minute utterance) does not fit the budget as a whole: a prefix of it
    t_cap = n_frames_per_utt
    if n_utt == 1 and per_frame * n_frames_per_utt > 1.5 * budget_s:
        t_cap = max(256, int(budget_s / per_frame))

    def work(u):
        s = scorer()(feats[u][:t_cap])
        oracle.phoneloop_run(pm.tp, pm.sseq, pm.phone_ssid[:pm.n_ciphone], pm.phone_tmat[:pm.n_ciphone], s,
                             PL["window"], PL["beam"], PL["pbeam"], PL["pip"], PL["weight"])
        if tmpl is not None:
            sweeper().sweep(tmpl.copy(), s)
        return len(s)

    if threads > 1:                       # load one reference model per worker before timing
        from concurrent.futures import ThreadPoolExecutor
        ex = ThreadPoolExecutor(threads)
        list(ex.map(lambda _: (scorer()(feats[0][:4]), sweeper()), range(threads * 2)))
    t0 = time.perf_counter()
    if threads == 1:
        done = sum(work(u) for u in range(n_utt))
    else:
        done = sum(ex.map(work, range(n_utt)))       # ctypes releases the GIL inside the C code
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "frames/s", "cores": threads, "kind": kind,
            "sample": "%d utterances x %d frames of the same batch: senone eval (%s) + phone loop (C port) + %s, %.1f s" % (
                n_utt, min(t_cap, n_frames_per_utt), "compiled reference" if kind == "reference" else "C port",
                ("hmm_vit_eval over %d active hmm_t per frame (%s)" % (N_ACTIVE, "compiled reference" if kind == "reference" else "C port"))
                if tmpl is not None else "no search-scale Viterbi for this topology", dt)}


def host_cores():
    """Usable host threads: nproc, capped by the cgroup CPU quota when there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def run_reference(args, pm, raw, desc, feats, T):
    """--impl reference: the reference algorithm's CPU implementation on all host cores."""
    cores = host_cores()
    steps = []
    base = None
    for i in range(args.warmup + args.steps):
        base = cpu_baseline(args, pm, raw, feats, T, budget_s=max(3.0, 60.0 / (args.warmup + args.steps)), threads=cores)
        if i >= args.warmup:
            steps.append(base["value"])
    v = float(np.mean(steps))
    base["value"] = v
    out = {"impl": "reference", "metric": "frames/sec senone-eval+Viterbi", "value": v, "unit": "frames/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": None,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32->i16/i32",
           "data": "synthetic", "config": {"workload": workload_name(args, pm), "model": desc},
           "cpu_baseline": base,
           "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def dump_outputs(out_dir, torch, batch, pm, total, H, d_best, d_pen, d_swbest):
    """Writes what the last timed step left on the device to out_dir/<name>.npy (integers as float64, int16 scores as
    float32, all exact; under 50 MB in all): the phone loop's best score per frame and the search-scale sweep's best
    score per (frame, utterance), whole up to 2^20 values; the phone-loop penalties and the senone scores (GBs at the
    default shape) on a fixed, seeded sample of frames.  A sampled array comes with <name>_rows.npy, the flat indices
    (rows) it holds.  The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda", torch.cuda.current_device())

    class DeviceArray:                      # a buffer the C API owns, seen by torch without a copy
        def __init__(self, ptr, shape, typestr):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "strides": None,
                                              "version": 3}

    def view(ptr, shape, typestr):
        return torch.as_tensor(DeviceArray(ptr, shape, typestr), device=dev)

    rng = np.random.default_rng(7)

    def save(name, x, cap, dtype):
        n = x.shape[0]
        if n > cap:
            rows = np.sort(rng.choice(n, cap, replace=False))
            x = x[torch.from_numpy(rows).to(dev)]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, name + ".npy"), x.cpu().numpy().astype(dtype))

    save("phoneloop_best", view(d_best, (total,), "<i4"), 1 << 20, np.float64)
    save("phoneloop_pen", view(d_pen, (total, H), "<i4"), 4096, np.float64)
    save("senscr", view(batch.senscr_device_ptr(), (total, pm.n_sen), "<i2"), max(1, (16 << 20) // (4 * pm.n_sen)), np.float32)
    if d_swbest is not None:
        sw = d_swbest if d_swbest.numel() <= 1 << 20 else d_swbest.reshape(-1)
        save("sweep_best", sw, 1 << 20, np.float64)


def workload_name(args, pm):
    n = ("%dutt_total" % args.batch_total) if getattr(args, "batch_total", 0) else ("%dutt" % args.utts)
    return "%s_%dx%dx%d_%dsen_%s_x_%ds" % (pm.kind, pm.n_mgau, pm.n_feat, pm.n_density, pm.n_sen, n, args.secs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="baseline", choices=["baseline", "en-us", "semi", "cont"])
    ap.add_argument("--utts", type=int, default=1000, help="utterances per GPU per step (weak scaling)")
    ap.add_argument("--batch-total", type=int, default=0,
                    help="fixed batch of this many utterances sharded over the GPUs (strong scaling, BASELINE config 3: 4096); "
                         "overrides --utts")
    ap.add_argument("--secs", type=int, default=10, help="seconds of 16 kHz audio per utterance")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--search", default="none", choices=["none", "fwdtree", "fsg"],
                    help="also couple a search kernel to the GMM stage's scores (BASELINE configs 3 / 4), reported as `search_coupled`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's shard) to DIR/<name>.npy, for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pm, desc, raw = load_model(args.model)
    T = frames_for(args.secs)

    if args.impl == "reference":
        if rank != 0:
            return
        feats = synth_feats(pm, min(args.utts, max(64, 2 * host_cores())), T, seed=1234)
        run_reference(args, pm, raw, desc, feats, T)
        return

    import torch
    import torch.distributed as dist
    from pocketsphinx_b200 import api

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # ---- acoustic model: rank 0 holds it, one NCCL broadcast per packed buffer at init ----
    from pocketsphinx_b200 import dist as pdist
    t_b = time.perf_counter()
    dev = pdist.broadcast_model(pm, src=0, device=torch.device("cuda", local))
    torch.cuda.synchronize()
    bcast_ms = (time.perf_counter() - t_b) * 1e3              # one-off at init: upload on rank 0 + NCCL broadcast
    model = api.Model(pm, device=local, device_ptrs=dev)

    # ---- this rank's shard of utterances (weak scaling: utts per GPU fixed) ----
    # weak scaling: --utts per GPU; strong scaling: --batch-total utterances dealt out over the ranks (equal lengths here, so
    # equal counts balance the frames; ragged batches would be dealt longest-first, pocketsphinx_b200/dist.py)
    strong = args.batch_total > 0
    U = args.utts if not strong else args.batch_total // world + (1 if rank < args.batch_total % world else 0)
    U_all = args.utts * world if not strong else args.batch_total
    feats_np = synth_feats(pm, U, T, seed=1234 + rank)
    total = U * T
    off = api.Batch.offsets([T] * U)
    feats_pinned = torch.from_numpy(feats_np.reshape(total, pm.sumlen)).pin_memory()
    d_feats = feats_pinned.cuda()
    batch = api.Batch(model, U, total)
    ctx = api.HmmContext(pm.tp, pm.sseq, pm.n_sen, device=local)
    H = pm.n_ciphone
    pl = api.PhoneLoop(ctx, pm.phone_ssid[:H], pm.phone_tmat[:H], PL["window"], PL["beam"], PL["pbeam"], PL["pip"],
                       PL["weight"])
    best_pinned = torch.empty(total, dtype=torch.int32).pin_memory()
    pen_pinned = torch.empty((total, H), dtype=torch.int32).pin_memory()

    # ---- search-scale Viterbi: N_ACTIVE entered hmm_t per utterance, resident on the device ----
    tmpl = channel_template(pm, api.HMM_DTYPE)
    hs = None
    if tmpl is not None:
        hs = api.HmmSet(ctx, U * N_ACTIVE + U * 512, U)       # slack: segments start on storage-tile boundaries
        hs.upload(np.tile(tmpl, U), np.arange(U + 1, dtype=np.int64) * N_ACTIVE)
        hs.use_batch_stream(batch)                            # behind the kernels that write the scores
        hs.snapshot()
        d_row0 = torch.from_numpy(np.asarray(off[:U], np.int64)).cuda(local)
        d_nrows = torch.from_numpy(np.diff(np.asarray(off, np.int64)).astype(np.int32)).cuda(local)
        d_swbest = torch.empty((T, U), dtype=torch.int32, device="cuda:%d" % local)
        swbest_pinned = torch.empty((T, U), dtype=torch.int32).pin_memory()
        batch.sync()

    def sweep():
        # every utterance's active set takes T hmm_vit_eval steps against the scores decode_* just left in HBM
        if hs is not None:
            hs.restore()
            hs.sweep_device(batch.senscr_device_ptr(), total, T, d_swbest.data_ptr(), d_row0=d_row0.data_ptr(),
                            d_n_rows=d_nrows.data_ptr(), timed=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        batch.sync()

    # ---- device-resident throughput: features already in HBM ----
    launches0 = api.lib().psb_kernel_launch_count()
    for _ in range(args.warmup):
        batch.decode_device(pl, d_feats.data_ptr(), off)
        sweep()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches1 = api.lib().psb_kernel_launch_count()
    batch.event_record(0)
    kern = {"transpose": 0.0, "topn": 0.0, "senone": 0.0}
    for _ in range(args.steps):
        d_best, d_pen = batch.decode_device(pl, d_feats.data_ptr(), off)
        sweep()
    batch.event_record(1)
    ms_total = batch.event_elapsed_ms()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, batch, pm, total, H, d_best, d_pen, d_swbest if hs is not None else None)
    launches = api.lib().psb_kernel_launch_count() - launches1
    # per-kernel durations for the roofline: two extra steps forced onto ONE stream (with
    # PSB_PIPELINE > 1 the timed region's kernels overlap and cannot be timed individually)
    batch.set_pipeline(1)
    for _ in range(2):
        batch.decode_device(pl, d_feats.data_ptr(), off)
    batch.sync()
    km = batch.last_kernel_ms()          # CUDA events around each kernel on the stream it runs on
    sweep_ms = None
    if hs is not None:                   # the sweep alone (its launch + the state restore), CUDA events on the same stream
        batch.sync()
        batch.event_record(0)
        sweep()
        batch.event_record(1)
        sweep_ms = batch.event_elapsed_ms()
    batch.set_pipeline(int(os.environ.get("PSB_PIPELINE", "0")))
    clocks = sampler.stop() if rank == 0 else None
    ms_step = ms_total / args.steps

    # ---- end to end through the public host-buffer call: H2D + kernels + D2H every step ----
    def e2e_step():
        batch.decode_host(pl, feats_pinned, off, best=best_pinned, pen=pen_pinned)
        if hs is not None:
            sweep()
            batch.sync()
            swbest_pinned.copy_(d_swbest)                     # the sweep's result: best path score per frame and utterance
            torch.cuda.synchronize()
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    # the same with the senone scores themselves copied back (what the larger-grain boundary hands to a host
    # search, SURVEY 8b): a bounded sample of the batch so that the pinned buffer stays small
    Us = min(U, 250)
    tot_s = int(off[Us])
    scr_pinned = torch.empty((tot_s, pm.n_sen), dtype=torch.int16).pin_memory()
    sub = api.Batch(model, Us, tot_s)
    def e2e_scr_step():
        sub.decode_host(pl, feats_pinned[:tot_s], off[:Us + 1], want_senscr=True, best=best_pinned[:tot_s], pen=pen_pinned[:tot_s],
                        senscr=scr_pinned)
    e2e_scr_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(2):
        e2e_scr_step()
    barrier()
    e2e_scr_ms = (time.perf_counter() - t0) * 1e3 / 2
    sub.close()
    del scr_pinned

    ms_step, e2e_ms, e2e_scr_ms = pdist.reduce_max_ms([ms_step, e2e_ms, e2e_scr_ms], device="cuda")

    if rank == 0:
        hbm_peak, peak_src, sm_max = peaks()
        frames_all = U_all * T
        value = frames_all / (ms_step * 1e-3)
        # roofline of the dominant kernel (the top-N kernel), algorithmic bytes per launch:
        # per frame 4*sumlen feature bytes read + 16*K top-N record bytes written, plus the
        # Gaussians once per launch (DESIGN.md "Kernels").
        K = pm.n_mgau * pm.n_feat
        # (ms models: the whole GMM stage is bracketed as "topn" by psb_launch_ms_batch)
        gau_bytes = (pm.mean.nbytes + pm.var.nbytes + pm.det.nbytes)
        topn_bytes = total * (4 * pm.sumlen + 16 * K) + gau_bytes
        topn_gbs = topn_bytes / (km["topn"] * 1e-3) / 1e9
        stage_bytes = total * (4 * pm.sumlen + 2 * pm.n_sen + 2 * 16 * K) + gau_bytes + pm.mixw.nbytes
        gmm_ms = km["transpose"] + km["topn"] + km["senone"]
        flop = 4.0 * pm.n_mgau * pm.n_density * pm.sumlen * total      # sub, mul, mul, sub per (codeword, dim)
        sm_mhz = (clocks or {}).get("sm_mhz") or sm_max
        fp32_peak = 148 * 128 * sm_mhz * 1e6 / 1e12                     # non-FMA FP32 lane-ops/s (TFLOP/s)
        tf32_peak = tensor_peak_bf16() / 2.0
        variant = int(os.environ.get("PSB_TOPN_VARIANT", "6"))
        tc_path = variant >= 6 and pm.kind == "ptm" and all(int(x) == 13 for x in pm.featlen) and pm.n_density in (64, 128, 256) \
            and int(getattr(pm, "ds_ratio", 1)) == 1
        topn_name = {"ms": "ms_dist_tile_kernel (distances + mixtures)", "s2_semi": "semi_dist_kernel+semi_scan_kernel"}.get(
            pm.kind, {0: "ptm_topn_kernel", 1: "ptm_topn2_kernel", 2: "ptm_topn2_kernel", 3: "ptm_topn_u2_kernel",
                      4: "ptm_topnq_kernel<NU=2>", 5: "ptm_topnq_kernel<NU=1>"}.get(variant, "ptm_topnq_kernel<NU=1>"))
        if tc_path:
            topn_name = "ptm_tc5_kernel" if os.environ.get("PSB_TC_IMPL") != "mma" else "ptm_tc_kernel"
        out = {
            "metric": "frames/sec senone-eval+Viterbi", "value": value, "unit": "frames/s",
            "xRT": FRAMES_PER_SEC_AUDIO / value,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32->i16/i32", "data": "synthetic",
            "config": {"workload": workload_name(args, pm), "model": desc,
                       "utts_per_gpu": U, "frames_per_utt": T, "frames_per_step_per_gpu": total,
                       "viterbi": ("phone loop (%d CI-phone HMMs x %d states, window %d) + search-scale hmm_vit_eval over %d active "
                                   "hmm_t per utterance and frame with a per-frame best-score reduction (evaluate_channels)"
                                   % (H, pm.n_emit_state, PL["window"], N_ACTIVE)) if hs is not None else
                                  "phone loop, %d CI-phone HMMs x %d states, window %d" % (H, pm.n_emit_state, PL["window"]),
                       "features": "synthetic dynamic features (AR(1) walk between model means), not PCM",
                       "parallelism": ("fixed batch of %d utterances dealt out over %d GPUs, no per-frame collective" % (U_all, world)) if strong
                                      else "utterances sharded, %d per GPU, no per-frame collective" % U,
                       "model_broadcast_ms": bcast_ms,
                       "l2": "per-step working set (%.1f GB of scores) exceeds L2; no explicit flush" % (total * pm.n_sen * 2 / 1e9)},
            "gpu_launches": int(launches),
            "kernel_ms_unpipelined": {**km, "note": "separate single-stream pass after the timed region"},
            "roofline": {"bound": "hbm", "kernel": topn_name, "achieved": topn_gbs, "peak": hbm_peak,
                         "unit": "GB/s", "frac": topn_gbs / hbm_peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this shape from an `ncu --set full`
                         # capture, when one is on file (profiles/ncu_traffic.json, written by profiles/ncu_traffic.py); else null
                         "traffic": ncu_traffic(topn_name, workload_name(args, pm)),
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": topn_bytes,
                         "note": "compute-bound by construction (SURVEY 8d): model is SMEM/L2 resident"},
            "roofline_fp32": {"bound": "fp32 non-FMA issue", "kernel": topn_name,
                              "achieved": flop / (km["topn"] * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                              "frac": flop / (km["topn"] * 1e-3) / 1e12 / fp32_peak,
                              "peak_source": "148 SMs x 128 lanes x sampled SM clock"},
            # the tensor-core filter of the top-N stage: 3 x TF32 GEMM [frames x 32] x [32 x n_density] per (codebook, stream) pair;
            # `achieved` counts those GEMM flops over the whole top-N stage (filter + exact rows + tie fix-up).  The stage's
            # algorithmic FP32 work (roofline_fp32) is what the scan kernels execute and this path mostly skips, so its
            # fraction there can exceed 1.
            "roofline_tensor": ({"bound": "tensor", "kernel": topn_name, "achieved": 3 * 2.0 * 32 * pm.n_density * K * total / (km["topn"] * 1e-3) / 1e12,
                                 "peak": tf32_peak, "unit": "TFLOP/s",
                                 "frac": 3 * 2.0 * 32 * pm.n_density * K * total / (km["topn"] * 1e-3) / 1e12 / tf32_peak,
                                 "peak_source": "half the measured dense bf16 rate of MEASURED_PEAKS.json (TF32 runs at half the bf16 rate)"}
                                if tc_path else None),
            "gmm_stage": {"ms": gmm_ms, "algorithmic_bytes": stage_bytes,
                          "achieved_gbs": stage_bytes / (gmm_ms * 1e-3) / 1e9},
            "e2e": {"value": frames_all / (e2e_ms * 1e-3), "unit": "frames/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(total * pm.sumlen * 4 + (U + 1) * 4),
                    "d2h_bytes_per_step": int(total * 4 + total * H * 4 + (total * 4 if hs is not None else 0)),
                    "call": "psb_decode_batch_host (pinned host features in, phone-loop best scores + penalties out) + "
                            "psb_hmmset_sweep_device (best path score per frame and utterance out)"},
            # the same boundary with the int16 senone scores themselves returned to the host (PCIe-bound)
            "e2e_with_senscr": {"value": tot_s * world / (e2e_scr_ms * 1e-3), "unit": "frames/s", "ms_per_step": e2e_scr_ms,
                                "sample": "%d utterances of the batch (pinned score buffer kept at %.1f GB)" % (Us, tot_s * pm.n_sen * 2 / 1e9),
                                "h2d_bytes_per_step": int(tot_s * pm.sumlen * 4), "d2h_bytes_per_step": int(tot_s * (pm.n_sen * 2 + 4 + 4 * H)),
                                "d2h_gbs": tot_s * (pm.n_sen * 2 + 4 + 4 * H) / (e2e_scr_ms * 1e-3) / 1e9,
                                "call": "psb_decode_batch_host with senscr != NULL (no search-scale Viterbi: the scores leave the device)"},
            "clocks": clocks,
        }
        if hs is not None:
            # registers hold the state, so the kernel's algorithmic traffic is the score rows (read once per CTA of a
            # segment; L2 serves the repeats) plus the state once: its bound is integer issue, not HBM
            n_inst = U * N_ACTIVE
            out["search_viterbi"] = {
                "kernel": "hmmset_sweep_kernel", "active_hmms_per_utt": N_ACTIVE, "ms": sweep_ms,
                "share_of_step": sweep_ms / ms_step, "hmm_updates_per_s": n_inst * T / (sweep_ms * 1e-3),
                "algorithmic_bytes": int(total * pm.n_sen * 2 + 2 * n_inst * (pm.n_emit_state * 10 + 14)),
                "hbm_streaming_equivalent_gbs": n_inst * T * ((2 * pm.n_emit_state * 4) * 2 + 2 * 4 * 2 + 4 + 2 * pm.n_emit_state + 2 + 2 * pm.n_emit_state)
                / (sweep_ms * 1e-3) / 1e9,
                "note": "part of `value`; state in registers for the whole utterance, score rows staged by TMA bulk copies "
                        "(cp.async.bulk + mbarrier); `hbm_streaming_equivalent_gbs` is what a per-frame kernel that moves the "
                        "state through HBM (viterbi_stage below) would have to sustain for the same time"}
        if world == 1:
            batch.set_pipeline(1)                           # leave the whole batch's scores in one buffer
            batch.decode_device(pl, d_feats.data_ptr(), off)
            batch.sync()
            if hs is not None:
                try:
                    out["search_viterbi_beam"] = beam_stage(torch, hs, batch, total, T, U, d_row0, d_nrows, local)
                except Exception as e:                          # an extra, never the reason for a missing bench line
                    out["search_viterbi_beam"] = {"error": str(e)[:300]}
            out["viterbi_stage"] = viterbi_stage(api, torch, ctx, batch, pm, off, U, T, hbm_peak)
            if pm.n_emit_state in (3, 5) and len(pm.sseq):
                out["align_stage"] = align_stage(api, ctx, batch, pm, off, U, T)
            out["frontend_stage"] = frontend_stage(api, torch, U, args.secs)
            out["search_stage"] = search_stage(api, torch)
            if args.search != "none":
                out["search_coupled"] = search_coupled_stage(api, torch, batch, pm, off, U, T, args.search, gmm_ms / total)
            out["cpu_baseline"] = cpu_baseline(args, pm, raw, feats_np, T, budget_s=args.cpu_budget, threads=1)
        print(json.dumps(out))
    if hs is not None:
        hs.close()
    batch.close(); pl.close(); ctx.close(); model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
