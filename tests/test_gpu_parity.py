"""GPU (-m gpu): the CUDA path through the C-ABI against the reference's golden vectors and
against the CPU oracle on seeded inputs.  Integer outputs must be bit-exact."""
import numpy as np
import pytest

from conftest import assert_hmm_equal, golden, hmm_view

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    from pocketsphinx_b200 import api
    assert api.device_count() > 0, "no CUDA device visible"
    return api


@pytest.fixture(scope="module")
def en_us_dev(api, en_us):
    m = api.Model(en_us)
    yield m
    m.close()


def test_ptm_batch_goforward_matches_reference(api, en_us_dev):
    g = golden("en_us_goforward.npz")
    b = api.Batch(en_us_dev, 4, 1024)
    scr = b.score_host(g["feats"], np.array([0, 278], np.int32))
    assert np.array_equal(scr, g["senscr"])
    b.close()


def test_ptm_batch_ragged_matches_oracle(api, en_us, en_us_dev):
    from oracle import oracle
    g = golden("en_us_goforward.npz")
    f = g["feats"]
    # 70 utterances of uneven length (0, 1, ... frames), cut from different places
    rng = np.random.default_rng(3)
    lens = [0, 1, 2, 33, 278] + [int(x) for x in rng.integers(1, 120, 65)]
    chunks = [f[s:s + n] for n, s in zip(lens, rng.integers(0, 278 - 120, len(lens)))]
    chunks[4] = f
    lens = [len(c) for c in chunks]
    feats = np.concatenate(chunks)
    off = api.Batch.offsets(lens)
    b = api.Batch(en_us_dev, 128, 8192)
    scr = b.score_host(feats, off)
    om = oracle.OracleModel(en_us)
    for u, c in enumerate(chunks):
        if len(c) == 0:
            continue
        want = om.score_utt(c)
        got = scr[off[u]:off[u + 1]]
        assert np.array_equal(got, want), "utterance %d (len %d)" % (u, len(c))
    # idempotent, and an empty batch is fine
    scr2 = b.score_host(feats, off)
    assert np.array_equal(scr, scr2)
    b.score_host(np.zeros((0, 39), np.float32), np.zeros(1, np.int32))
    b.close()


@pytest.mark.parametrize("n_density,n_sen", [(256, 5138), (128, 1000), (64, 300)])
def test_ptm_batch_synthetic_matches_oracle(api, n_density, n_sen):
    from oracle import oracle
    from pocketsphinx_b200.model import synth_feats, synth_ptm
    pm = synth_ptm(seed=5, n_density=n_density, n_sen=n_sen)
    feats = synth_feats(pm, 40, 24, seed=9)
    m = api.Model(pm)
    b = api.Batch(m, 64, 4096)
    off = api.Batch.offsets([24] * 40)
    scr = b.score_host(feats.reshape(-1, pm.sumlen), off)
    om = oracle.OracleModel(pm)
    for u in range(40):
        assert np.array_equal(scr[off[u]:off[u + 1]], om.score_utt(feats[u])), "utterance %d" % u
    b.close()
    m.close()


def test_scorer_frame_eval_compallsen(api, en_us_dev):
    g = golden("en_us_goforward.npz")
    s = api.Mgau(en_us_dev, pl_window=0)
    for t in range(60):
        scr = s.frame_eval(g["feats"][t], t)
        s.frame_idx = t + 1                      # acmod_advance
        assert np.array_equal(scr, g["senscr"][t]), "frame %d" % t
    # re-scoring the previous frame from the history ring gives the same scores
    again = s.frame_eval(g["feats"][59], 59)
    assert np.array_equal(again, g["senscr"][59])
    s.close()


def test_scorer_frame_eval_active_lists(api, en_us_dev):
    from oracle import oracle
    g = golden("en_us_active.npz")
    gf = golden("en_us_goforward.npz")
    n_sen = int(g["n_sen"])
    flags = np.unpackbits(g["flags"], axis=1)[:, :n_sen]
    s = api.Mgau(en_us_dev, pl_window=0)
    for t in range(flags.shape[0]):
        lst = oracle.flags2list(flags[t])
        scr = s.frame_eval(gf["feats"][t], t, lst, compallsen=False)
        s.frame_idx = t + 1
        assert np.array_equal(scr, g["senscr"][t]), "frame %d" % t
    s.close()


def test_scorer_lookahead_ring_matches_oracle(api, en_us, en_us_dev):
    """pl_window = 5: frame F scored for the phone loop with CI senones, then frame F-5 re-scored
    from the ring with a different active list (ps_search_forward, pocketsphinx.c:1173-1197)."""
    from oracle import oracle
    gf = golden("en_us_goforward.npz")
    rng = np.random.default_rng(1)
    om = oracle.OracleModel(en_us)
    dec = om.decoder(n_hist=7)
    s = api.Mgau(en_us_dev, pl_window=5)
    ci = np.zeros(en_us.n_sen, np.uint8)
    ci[:en_us.n_ci_sen] = 1
    ci_list = oracle.flags2list(ci)
    for F in range(40):
        a = s.frame_eval(gf["feats"][F], F, ci_list, compallsen=False)
        o = dec.frame_eval(gf["feats"][F], F, ci_list, compallsen=False)
        assert np.array_equal(a, o), "lookahead frame %d" % F
        if F >= 5:
            fl = (rng.random(en_us.n_sen) < 0.2).astype(np.uint8)
            lst = oracle.flags2list(fl)
            a = s.frame_eval(gf["feats"][F - 5], F - 5, lst, compallsen=False)
            o = dec.frame_eval(gf["feats"][F - 5], F - 5, lst, compallsen=False)
            assert np.array_equal(a, o), "search frame %d" % (F - 5)
        s.frame_idx = F + 1
        dec.set_frame_idx(F + 1)
    s.close()
    dec.close()


@pytest.mark.parametrize("n_emit", [3, 5, 4, 1])
def test_hmm_vit_eval_batch(api, n_emit):
    g = golden("hmm_vit_eval.npz")
    senscr = g["n%d_senscr" % n_emit]
    ctx = api.HmmContext(g["n%d_tp" % n_emit], g["n%d_sseq" % n_emit], len(senscr))
    hm = hmm_view(g["n%d_before" % n_emit]).copy()
    want = hmm_view(g["n%d_after" % n_emit])
    hm["ctx"] = 0x1234                      # caller's pointer must survive
    best = ctx.vit_eval(hm, senscr)
    assert best == int(g["n%d_best" % n_emit])
    assert (hm["ctx"] == 0x1234).all()
    assert_hmm_equal(hm, want, n_emit, "n_emit=%d" % n_emit)
    # active-list-of-pointers entry on a subset
    hm2 = hmm_view(g["n%d_before" % n_emit]).copy()
    idx = np.arange(0, len(hm2), 3)
    ctx.vit_eval_ptrs(hm2, idx, senscr)
    assert_hmm_equal(hm2[idx], want[idx], n_emit, "ptrs")
    untouched = np.setdiff1d(np.arange(len(hm2)), idx)
    assert_hmm_equal(hm2[untouched], hmm_view(g["n%d_before" % n_emit])[untouched], n_emit, "untouched")
    assert ctx.vit_eval(hm[:0], senscr) == -0x20000000
    ctx.close()


def test_phoneloop_matches_reference(api, en_us):
    g = golden("en_us_goforward.npz")
    n, beam, pbeam, pip, window = [int(x) for x in g["pl_params"]]
    ctx = api.HmmContext(en_us.tp, en_us.sseq, en_us.n_sen)
    pl = api.PhoneLoop(ctx, en_us.phone_ssid[:n], en_us.phone_tmat[:n], window, beam, pbeam, pip, float(g["pl_weight"]))
    # the same utterance three times in one batch, plus a truncated copy
    scr = np.concatenate([g["senscr"], g["senscr"][:100], g["senscr"]])
    off = api.Batch.offsets([278, 100, 278])
    r = pl.run_host(scr, off, trace=True)
    want = hmm_view(g["pl_hmm"])
    for u, (a, n_fr) in enumerate(zip(off[:-1], [278, 100, 278])):
        assert np.array_equal(r["best"][a:a + n_fr], g["pl_best"][:n_fr]), "utt %d best" % u
        assert np.array_equal(r["pen"][a:a + n_fr], g["pl_pen"][:n_fr]), "utt %d penalties" % u
        assert_hmm_equal(r["hmm"][a:a + n_fr], want[:n_fr], 3, "utt %d" % u)
    pl.close()
    ctx.close()


def test_decode_host_end_to_end(api, en_us, en_us_dev):
    g = golden("en_us_goforward.npz")
    n, beam, pbeam, pip, window = [int(x) for x in g["pl_params"]]
    ctx = api.HmmContext(en_us.tp, en_us.sseq, en_us.n_sen)
    pl = api.PhoneLoop(ctx, en_us.phone_ssid[:n], en_us.phone_tmat[:n], window, beam, pbeam, pip, float(g["pl_weight"]))
    b = api.Batch(en_us_dev, 8, 2048)
    feats = np.concatenate([g["feats"], g["feats"][:50], g["feats"]])
    off = api.Batch.offsets([278, 50, 278])
    best, pen, scr = b.decode_host(pl, feats, off, want_senscr=True)
    assert np.array_equal(scr[:278], g["senscr"]) and np.array_equal(scr[328:], g["senscr"])
    assert np.array_equal(best[:278], g["pl_best"]) and np.array_equal(best[328:], g["pl_best"])
    assert np.array_equal(pen[278:328], g["pl_pen"][:50])
    b.close(); pl.close(); ctx.close()


# ---------------------------------------------------------------------------------------
# semi-continuous (s2_semi_mgau) and generic multi-stream (ms_mgau) back-ends, batched

def _batch_vs_oracle(api, pm, feats_by_utt):
    from oracle import oracle
    m = api.Model(pm)
    lens = [len(f) for f in feats_by_utt]
    b = api.Batch(m, len(lens) + 1, sum(lens) + 8)
    off = api.Batch.offsets(lens)
    scr = b.score_host(np.concatenate(feats_by_utt), off)
    om = oracle.OracleModel(pm)
    for u, f in enumerate(feats_by_utt):
        want = om.score_utt(f)
        got = scr[off[u]:off[u + 1]]
        bad = np.argwhere(got != want)
        assert bad.size == 0, "utt %d: first mismatch (frame, senone) %s: got %s want %s" % (
            u, bad[0].tolist(), got[tuple(bad[0])], want[tuple(bad[0])])
    b.close()
    m.close()
    return scr, off


def test_semi_tidigits_matches_reference(api, tidigits):
    g = golden("tidigits_goforward.npz")
    scr, off = _batch_vs_oracle(api, tidigits, [g["feats"], g["feats"][:37]])
    assert np.array_equal(scr[:len(g["feats"])], g["senscr"])


@pytest.mark.parametrize("four_bit,beam,n_sen", [(False, None, 670), (True, None, 671), (False, [40, 0, 25, 96], 300)])
def test_semi_synthetic_matches_oracle(api, four_bit, beam, n_sen):
    from pocketsphinx_b200.model import synth_feats, synth_semi
    pm = synth_semi(seed=3, n_sen=n_sen, four_bit=four_bit, topn_beam=beam)
    feats = synth_feats(pm, 35, 30, seed=4)
    _batch_vs_oracle(api, pm, list(feats))


def test_ms_an4_matches_reference(api, an4):
    g = golden("an4_goforward.npz")
    scr, off = _batch_vs_oracle(api, an4, [g["feats"], g["feats"][:10]])
    assert np.array_equal(scr[:len(g["feats"])], g["senscr"])


@pytest.mark.parametrize("kw", [dict(n_sen=700, n_density=8, topn=4), dict(n_sen=300, n_density=4, topn=4),
                                dict(n_sen=500, n_density=16, topn=2, featlens=(13, 13, 13), n_mgau=42),
                                dict(n_sen=400, n_density=32, topn=8, featlens=(12, 24, 3, 12), n_mgau=1, aw=3)])
def test_ms_synthetic_matches_oracle(api, kw):
    from pocketsphinx_b200.model import synth_feats, synth_ms
    pm = synth_ms(seed=8, **kw)
    feats = synth_feats(pm, 9, 21, seed=5)
    _batch_vs_oracle(api, pm, list(feats))


def test_ptm_and_semi_tie_stress(api):
    """Integer-valued Gaussians and features: exact ties everywhere, so any deviation from the
    reference's insertion order / tie rules shows up."""
    from oracle import oracle
    from pocketsphinx_b200.model import quantize_for_ties, synth_ptm, synth_semi
    for base in (synth_ptm(seed=2, n_density=64, n_sen=400), synth_semi(seed=2, n_density=64, n_sen=200)):
        pm, gen = quantize_for_ties(base, seed=6)
        feats = gen(40, 25, s=9)
        om = oracle.OracleModel(pm)
        want0, topn = om.score_utt(feats[0], want_topn=True)
        # the stress is real: adjacent list entries tie at the int level in many frames
        sc = topn[..., 1]
        assert (sc[..., :-1] == sc[..., 1:]).mean() > 0.05
        _batch_vs_oracle(api, pm, list(feats))


# ---------------------------------------------------------------------------------------
# per-frame scorers (the ps_mgau_t drop-in) for the semi-continuous and ms back-ends

def _scorer_vs_oracle(api, pm, feats, n_hist_window, rng, p_active=0.3, lookback=0):
    """Drive Mgau.frame_eval and the oracle's frame_eval with identical call sequences."""
    from oracle import oracle
    m = api.Model(pm)
    s = api.Mgau(m, pl_window=n_hist_window)
    dec = oracle.OracleModel(pm).decoder(n_hist=n_hist_window + 2)
    host = np.zeros(pm.n_sen, np.int16)      # the caller-owned buffer (persists across calls)
    want = np.zeros(pm.n_sen, np.int16)
    for t in range(len(feats)):
        mode = t % 3
        if mode == 0:
            lst, compall = None, True
        else:
            fl = (rng.random(pm.n_sen) < p_active).astype(np.uint8)
            if mode == 2:
                fl[pm.n_sen // 3: pm.n_sen // 3 + 300] = 0          # a gap that needs bridging
            lst, compall = oracle.flags2list(fl), False
        got = s.frame_eval(feats[t], t, lst, compallsen=compall, out=host)
        dec.frame_eval_into(want, feats[t], t, lst, compallsen=compall)
        assert np.array_equal(got, want), "frame %d (mode %d)" % (t, mode)
        if lookback and t >= lookback:
            fl = (rng.random(pm.n_sen) < p_active).astype(np.uint8)
            lst = oracle.flags2list(fl)
            got = s.frame_eval(feats[t - lookback], t - lookback, lst, compallsen=False, out=host)
            dec.frame_eval_into(want, feats[t - lookback], t - lookback, lst, compallsen=False)
            assert np.array_equal(got, want), "re-scored frame %d" % (t - lookback)
        s.frame_idx = t + 1
        dec.set_frame_idx(t + 1)
    s.close(); dec.close(); m.close()


def test_scorer_semi_tidigits(api, tidigits):
    g = golden("tidigits_goforward.npz")
    m = api.Model(tidigits)
    s = api.Mgau(m, pl_window=0)
    for t in range(40):
        assert np.array_equal(s.frame_eval(g["feats"][t], t), g["senscr"][t]), "frame %d" % t
        s.frame_idx = t + 1
    s.close(); m.close()
    _scorer_vs_oracle(api, tidigits, g["feats"][:45], 3, np.random.default_rng(2), lookback=3)


@pytest.mark.parametrize("four_bit,beam", [(False, None), (True, [30, 0, 20, 96])])
def test_scorer_semi_synthetic(api, four_bit, beam):
    from pocketsphinx_b200.model import synth_feats, synth_semi
    pm = synth_semi(seed=11, n_sen=901, four_bit=four_bit, topn_beam=beam)
    feats = synth_feats(pm, 1, 36, seed=12)[0]
    _scorer_vs_oracle(api, pm, feats, 2, np.random.default_rng(3), lookback=2)


def test_scorer_ms(api, an4):
    from pocketsphinx_b200.model import synth_feats, synth_ms
    g = golden("an4_goforward.npz")
    m = api.Model(an4)
    s = api.Mgau(m, pl_window=0)
    for t in range(30):
        assert np.array_equal(s.frame_eval(g["feats"][t], t), g["senscr"][t]), "frame %d" % t
        s.frame_idx = t + 1
    s.close(); m.close()
    pm = synth_ms(seed=13, n_sen=800, n_density=8, topn=4)
    _scorer_vs_oracle(api, pm, synth_feats(pm, 1, 30, seed=14)[0], 0, np.random.default_rng(4))
    pm = synth_ms(seed=15, n_sen=500, n_density=16, topn=2, featlens=(13, 13, 13), n_mgau=42)
    _scorer_vs_oracle(api, pm, synth_feats(pm, 1, 24, seed=16)[0], 0, np.random.default_rng(5))


@pytest.mark.parametrize("n_emit,H,window,skip", [(3, 1500, 0, False), (5, 200, 3, True), (3, 64, 5, True)])
def test_phoneloop_large_and_5state_vs_oracle(api, n_emit, H, window, skip):
    """The device phone loop as a generic HMM-set Viterbi: thousands of HMMs per utterance in
    shared-memory SoA, 5-state topologies with skip arcs, ragged utterances -- against the oracle's
    restatement of phone_loop_search.c (itself pinned on the reference's trace)."""
    from oracle import oracle
    from pocketsphinx_b200.model import synth_tmat_float
    from pocketsphinx_b200 import s3io
    rng = np.random.default_rng(21)
    n_sen, n_tmat = 900, 12
    tp = s3io.quantize_tmat(synth_tmat_float(rng, n_tmat, n_emit, skip))
    sseq = rng.integers(0, n_sen, (H, n_emit)).astype(np.uint16)
    ssid = np.arange(H, dtype=np.int32)
    tmat = rng.integers(0, n_tmat, H).astype(np.int32)
    lens = [40, 1, 23]
    senscr = rng.integers(0, 400, (sum(lens), n_sen)).astype(np.int16)
    senscr[:, rng.integers(0, n_sen, 50)] = 0            # some very good senones every frame
    off = api.Batch.offsets(lens)
    ctx = api.HmmContext(tp, sseq, n_sen)
    pl = api.PhoneLoop(ctx, ssid, tmat, window, -300, -250, -7, 2.5)
    got = pl.run_host(senscr, off, trace=True)
    for u in range(len(lens)):
        a, b = off[u], off[u + 1]
        want = oracle.phoneloop_run(tp, sseq, ssid, tmat, senscr[a:b], max(window, 1) if window else 1,
                                    -300, -250, -7, 2.5) if window else None
        if window == 0:
            # the oracle's penalty ring needs window >= 1; penalties are not produced when window == 0
            want = oracle.phoneloop_run(tp, sseq, ssid, tmat, senscr[a:b], 1, -300, -250, -7, 2.5)
        assert np.array_equal(got["best"][a:b], want["best"]), "utt %d best" % u
        if window:
            assert np.array_equal(got["pen"][a:b], want["pen"]), "utt %d penalties" % u
        assert_hmm_equal(got["hmm"][a:b], want["hmm"], n_emit, "utt %d" % u)
    pl.close(); ctx.close()


# ---------------------------------------------------------------------------------------
# the scan kernels (PSB_TOPN_VARIANT=5, read at psb_batch_create) and the default selection by model shape (6) must
# give the same bits; the last four models reach the fallbacks that only a model's shape selects

@pytest.mark.parametrize("case", ["en_us", "ragged", "ties", "ds2", "ptm_logbase", "semi_logbase", "semi_nd32", "ptm_fl39"])
def test_topn_kernel_variants(api, en_us_dev, case, monkeypatch):
    from pocketsphinx_b200.model import make_logadd8, quantize_for_ties, synth_feats, synth_ptm, synth_semi
    if case == "ragged":
        # BASELINE shape, ragged batch of 70 utterances (3 lane groups: an odd group count, padding lanes,
        # zero-length utterances)
        pm = synth_ptm(seed=11, n_density=256, n_sen=600)
        lens = [0, 1, 40, 0, 17] + [int(x) for x in np.random.default_rng(4).integers(1, 40, 65)]
        feats = synth_feats(pm, len(lens), 40, seed=3)
        chunks = [feats[u][:n].reshape(n, pm.sumlen) for u, n in enumerate(lens)]
    elif case == "ties":
        # exact ties everywhere
        pm, gen = quantize_for_ties(synth_ptm(seed=2, n_density=64, n_sen=400), seed=6)
        chunks = list(gen(40, 25, s=9))
    elif case == "ds2":
        # frame down-sampling (-ds 2): odd frames only re-score the listed codewords
        pm = synth_ptm(seed=12, n_density=128, n_sen=300)
        pm.ds_ratio = 2
        chunks = list(synth_feats(pm, 33, 20, seed=5))
    elif case in ("ptm_logbase", "semi_logbase"):
        # -logbase 1.00003: the add table's largest entry is 23 and 3 * 23 >= SEN_BIAS, so the senone stage takes
        # ptm_senone_kernel<false> / semi_senone_kernel<false> instead of the 16x2 kernels
        pm = (synth_ptm if case == "ptm_logbase" else synth_semi)(seed=31, n_density=64, n_sen=400)
        pm.logadd8 = make_logadd8(base=1.00003)
        chunks = list(synth_feats(pm, 20, 25, seed=4))
    elif case == "semi_nd32":
        # semi-continuous with n_density 32, outside the split path: ptm_topn2_kernel for the 12- and 3-dimensional
        # streams, the float scalar ptm_topn_kernel<24, true, false> for the 24-dimensional one
        pm = synth_semi(seed=32, n_density=32, n_sen=300)
        chunks = list(synth_feats(pm, 20, 25, seed=4))
    elif case == "ptm_fl39":
        # PTM with one 39-dimensional stream (no tensor-core filter): the float scalar ptm_topn_kernel<39, false, false>
        pm = synth_ptm(seed=33, n_feat=1, featlen=39, n_density=64, n_sen=400)
        chunks = list(synth_feats(pm, 20, 25, seed=4))
    for variant in (5, 6):
        monkeypatch.setenv("PSB_TOPN_VARIANT", str(variant))
        if case == "en_us":
            # shipped model, real features
            g = golden("en_us_goforward.npz")
            b = api.Batch(en_us_dev, 4, 1024)
            assert np.array_equal(b.score_host(g["feats"], np.array([0, 278], np.int32)), g["senscr"]), variant
            b.close()
        else:
            _batch_vs_oracle(api, pm, chunks)


def test_topn_variant_outside_the_accepted_values_is_refused(api, en_us_dev, monkeypatch):
    """Values of PSB_TOPN_VARIANT that once selected other kernels are refused, not silently mapped to a path."""
    monkeypatch.setenv("PSB_TOPN_VARIANT", "2")
    with pytest.raises(api.PsbError, match="accepted: 5"):
        api.Batch(en_us_dev, 4, 1024)


TC_CHECK = r"""
import sys, json, numpy as np
sys.path.insert(0, %r)
sys.path.insert(0, %r)
from conftest import golden
from oracle import oracle
from pocketsphinx_b200 import api
from pocketsphinx_b200.model import PackedModel, quantize_for_ties, synth_feats, synth_ptm
out = {}
def run(name, pm, chunks):
    m = api.Model(pm); lens = [len(c) for c in chunks]; off = api.Batch.offsets(lens)
    b = api.Batch(m, len(chunks) + 1, int(off[-1]) + 1)
    scr = b.score_host(np.concatenate(chunks), off)
    om = oracle.OracleModel(pm)
    ok = all(np.array_equal(scr[off[u]:off[u + 1]], om.score_utt(c)) for u, c in enumerate(chunks) if len(c))
    r, n = b.tc_check()
    out[name] = {"identical": bool(ok), "ratio": float(r), "max_candidates": int(n), "stats": b.tc_stats}
    b.close(); m.close()
g = golden("en_us_goforward.npz")
run("en_us", PackedModel.load(%r), [g["feats"]])
pm = synth_ptm(seed=0); f = synth_feats(pm, 24, 60, seed=5)
run("baseline_shape", pm, [f[u] for u in range(24)])
run("baseline_shape_x100", pm, [f[u] * np.float32(100) for u in range(8)])      # features far outside the model
pmq, gen = quantize_for_ties(synth_ptm(seed=2, n_density=64, n_sen=400), seed=6)
run("ties", pmq, list(gen(20, 25, s=9)))
print(json.dumps(out))
"""


def test_tensor_core_filter_error_bound_holds_on_the_device():
    """PSB_TC_CHECK=1: the filter kernel compares every 3 x TF32 GEMM value it produced with the exact float
    distance and reports the worst |a - d| / eps (the bound the candidate selection relies on must hold
    with room to spare: the analysis in psb_ptm_tc.cu allows 0.8 of eps), on the shipped model with real
    features, the BASELINE shape, features scaled far outside the model's range and tie-stress data."""
    import json
    import os
    import subprocess
    import sys
    from conftest import GOLDEN, ROOT
    code = TC_CHECK % (ROOT, os.path.join(ROOT, "tests"), os.path.join(GOLDEN, "en_us_ptm_model.npz"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PSB_TC_CHECK="1", PSB_TOPN_VARIANT="6"),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    print(out)
    for name, v in out.items():
        assert v["identical"], name
        assert 0.0 <= v["ratio"] < 0.8, (name, v)
        assert v["max_candidates"] >= 5, (name, v)


def test_ptm_and_semi_mixw_extremes(api):
    """Mixture weights of 0 and 255 next to each other: |x - y| in fast_logmath_add exceeds the
    reference's 256-entry table (undefined there); both sides continue the table with zeros."""
    from pocketsphinx_b200.model import synth_feats, synth_ptm, synth_semi
    for pm in (synth_ptm(seed=21, n_density=64, n_sen=500), synth_semi(seed=21, n_density=64, n_sen=300)):
        rng = np.random.default_rng(8)
        mw = pm.mixw.copy()
        mask = rng.random(mw.shape) < 0.5
        mw[mask] = np.where(rng.random(mask.sum()) < 0.5, 0, 255).astype(mw.dtype)
        pm.mixw = np.ascontiguousarray(mw)
        feats = synth_feats(pm, 20, 12, seed=2)
        _batch_vs_oracle(api, pm, [feats[u].reshape(-1, pm.sumlen) for u in range(20)])


# ---------------------------------------------------------------------------------------
# device-resident HMM sets (segments = utterances), several frames, against hmm_vit_eval

@pytest.mark.parametrize("n_emit", [3, 5, 4])
def test_hmmset_frames_match_oracle(api, n_emit):
    import torch
    from oracle import oracle
    g = golden("hmm_vit_eval.npz")
    tp, sseq = g["n%d_tp" % n_emit], g["n%d_sseq" % n_emit]
    n_sen = len(g["n%d_senscr" % n_emit])
    hm0 = hmm_view(g["n%d_before" % n_emit]).copy()            # 4096 random records, mixed mpx
    # the golden's single step through the set (segment 0 of 1)
    ctx = api.HmmContext(tp, sseq, n_sen)
    hs = api.HmmSet(ctx, len(hm0) + 7, 16)
    hs.upload(hm0, [0, len(hm0)])
    best = hs.eval_host(g["n%d_senscr" % n_emit][None, :])
    assert best[0] == int(g["n%d_best" % n_emit])
    got = hs.download()
    assert_hmm_equal(got, hmm_view(g["n%d_after" % n_emit]), n_emit, "golden step")
    # ragged segments (one empty), own score rows, 6 frames, one segment finishing early
    rng = np.random.default_rng(12)
    seg_off = np.array([0, 1000, 1000, 1257, 4096], np.int64)
    n_seg, T = len(seg_off) - 1, 6
    n_rows = np.array([6, 6, 4, 6], np.int32)
    senscr = rng.integers(0, 900, (T, n_seg, n_sen)).astype(np.int16)
    hs.upload(hm0, seg_off)
    d_scr = torch.from_numpy(senscr).cuda()
    d_best = torch.zeros((T, n_seg), dtype=torch.int32, device="cuda")
    d_nrows = torch.from_numpy(n_rows).cuda()
    ms = hs.eval_frames_device(d_scr.data_ptr(), T, d_best.data_ptr(), d_n_rows=d_nrows.data_ptr())
    assert ms >= 0.0
    got = hs.download()
    gbest = d_best.cpu().numpy()
    octx = oracle.OracleHmmCtx(tp, sseq)
    want = hm0.copy()
    for s in range(n_seg):
        a, b = seg_off[s], seg_off[s + 1]
        for t in range(T):
            if t >= n_rows[s] or a == b:
                assert gbest[t, s] == -0x20000000
                continue
            seg = np.ascontiguousarray(want[a:b])
            wb = octx.vit_eval(seg, senscr[t, s])
            want[a:b] = seg
            assert gbest[t, s] == wb, "segment %d frame %d" % (s, t)
    assert_hmm_equal(got, want, n_emit, "after %d frames" % T)
    hs.close()
    ctx.close()


@pytest.mark.parametrize("n_emit,n_sen_odd", [(3, False), (5, False), (3, True)])
def test_hmmset_sweep_matches_per_frame_and_oracle(api, n_emit, n_sen_odd):
    """psb_hmmset_sweep_device (all frames in one launch, state in registers, score rows staged by TMA bulk
    copies) against the per-frame kernel and against hmm_vit_eval of the oracle: ragged segments (one empty,
    one of a single instance, one spanning several CTAs), segments finishing early, rows addressed through
    d_row0 up to the very last row of the matrix (the one that is not over-read), every row misaligned
    differently (n_sen * 2 is not a multiple of 16)."""
    import torch
    from oracle import oracle
    g = golden("hmm_vit_eval.npz")
    tp, sseq = g["n%d_tp" % n_emit], g["n%d_sseq" % n_emit]
    n_sen = len(g["n%d_senscr" % n_emit]) - (1 if n_sen_odd else 0)     # odd count: served by the per-frame launches
    if n_sen % 2 == 1 and not n_sen_odd:
        n_sen -= 1
    hm0 = hmm_view(g["n%d_before" % n_emit]).copy()
    hm0 = hm0[hm0["mpx"] == 0].copy()                                    # the fused kernel takes plain instances
    hm0 = hm0[(hm0["senid"][:, :n_emit] < n_sen).all(1)].copy()
    n = len(hm0)
    assert n > 1500
    rng = np.random.default_rng(5)
    seg_off = np.array([0, 1, 1, 260, 1300, n], np.int64)
    n_seg, T = len(seg_off) - 1, 9
    n_rows = np.array([9, 9, 5, 9, 7], np.int32)
    R = 40
    senscr = rng.integers(0, 900, (R, n_sen)).astype(np.int16)
    row0 = np.array([3, 0, 11, R - 9, 20], np.int64)                     # segment 3 ends on the matrix's last row
    ctx = api.HmmContext(tp, sseq, n_sen)
    d_scr = torch.from_numpy(senscr).cuda()
    d_row0, d_nrows = torch.from_numpy(row0).cuda(), torch.from_numpy(n_rows).cuda()
    res = []
    for fused in (False, True):
        hs = api.HmmSet(ctx, n + 8 * 512, 16)
        hs.upload(hm0, seg_off)
        d_best = torch.zeros((T, n_seg), dtype=torch.int32, device="cuda")
        if fused:
            hs.sweep_device(d_scr.data_ptr(), R, T, d_best.data_ptr(), d_row0=d_row0.data_ptr(), d_n_rows=d_nrows.data_ptr())
        else:
            hs.eval_frames_device(d_scr.data_ptr(), T, d_best.data_ptr(), d_row0=d_row0.data_ptr(), d_n_rows=d_nrows.data_ptr())
        res.append((hs.download(), d_best.cpu().numpy()))
        hs.close()
    assert np.array_equal(res[0][1], res[1][1])
    assert_hmm_equal(res[1][0], res[0][0], n_emit, "fused vs per-frame")
    octx = oracle.OracleHmmCtx(tp, sseq)
    want = hm0.copy()
    for s in range(n_seg):
        a, b = seg_off[s], seg_off[s + 1]
        for t in range(T):
            if t >= n_rows[s] or a == b:
                assert res[1][1][t, s] == -0x20000000
                continue
            seg = np.ascontiguousarray(want[a:b])
            wb = octx.vit_eval(seg, np.concatenate([senscr[row0[s] + t], np.zeros(len(g["n%d_senscr" % n_emit]) - n_sen, np.int16)]))
            want[a:b] = seg
            assert res[1][1][t, s] == wb, "segment %d frame %d" % (s, t)
    assert_hmm_equal(res[1][0], want, n_emit, "after %d frames" % T)
    ctx.close()


@pytest.mark.parametrize("n_emit,big,maxhmmpf", [(3, 6081, -1), (3, 6081, 2500), (5, 2300, 900), (3, 9100, 4000)])
def test_hmmset_sweep_beam_matches_oracle(api, n_emit, big, maxhmmpf):
    """psb_hmmset_sweep_beam_device -- the fused sweep with beam pruning between frames, one thread-block cluster per
    segment (maxima / counts / -maxhmmpf histograms exchanged through distributed shared memory) -- against
    oracle.sweep_beam (pinned on the reference's hmm_vit_eval and hmm_clear in tests/test_hmm_beam_oracle.py): ragged
    segments (empty, one instance, several CTAs; 9100 instances = a cluster of 9, beyond the portable 8), segments
    finishing early, instances that are not active and must stay untouched, the histogram walk with and without effect."""
    import torch
    from conftest import beam_case
    from oracle import oracle
    frame0, beam, T = 7, -3000, 11
    seg_len = [1, 0, 259, 1040, big]
    n = sum(seg_len)
    tp, sseq, hm0, n_sen = beam_case(n_emit, n, 40 + n_emit + big)
    n_sen -= n_sen & 1
    hm0 = hm0[(hm0["senid"][:, :n_emit] < n_sen).all(1)]
    seg_len[-1] -= n - len(hm0)
    n = len(hm0)
    seg_off = np.concatenate([[0], np.cumsum(seg_len)]).astype(np.int64)
    n_seg = len(seg_len)
    n_rows = np.array([11, 11, 5, 11, 9], np.int32)
    R = 40
    rng = np.random.default_rng(6)
    senscr = rng.integers(0, 900, (R, n_sen)).astype(np.int16)
    row0 = np.array([3, 0, 12, R - 11, 20], np.int64)                    # segment 3 ends on the matrix's last row
    ctx = api.HmmContext(tp, sseq, n_sen)
    d_scr = torch.from_numpy(senscr).cuda()
    d_row0, d_nrows = torch.from_numpy(row0).cuda(), torch.from_numpy(n_rows).cuda()
    hs = api.HmmSet(ctx, n + 8 * 512, 16)
    hs.upload(hm0, seg_off)
    d_best = torch.zeros((T, n_seg), dtype=torch.int32, device="cuda")
    d_nact = torch.full((T, n_seg), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()                                             # the set's stream does not wait for torch's
    hs.sweep_beam_device(d_scr.data_ptr(), R, T, frame0, beam, d_best.data_ptr(), maxhmmpf=maxhmmpf, d_n_active=d_nact.data_ptr(),
                         d_row0=d_row0.data_ptr(), d_n_rows=d_nrows.data_ptr())
    got, best, nact = hs.download(), d_best.cpu().numpy(), d_nact.cpu().numpy()
    hs.close()
    ctx.close()
    octx = oracle.OracleHmmCtx(tp, sseq)
    want = hm0.copy()
    for s in range(n_seg):
        a, b = seg_off[s], seg_off[s + 1]
        Ts = int(min(T, n_rows[s]))
        seg = np.ascontiguousarray(want[a:b])
        wb, wn = oracle.sweep_beam(octx, seg, senscr[row0[s]:row0[s] + Ts], frame0, beam, maxhmmpf)
        want[a:b] = seg
        assert np.array_equal(best[:Ts, s], wb), "segment %d best" % s
        assert np.array_equal(nact[:Ts, s], wn), "segment %d counts: %s vs %s" % (s, nact[:Ts, s], wn)
        assert (best[Ts:, s] == -0x20000000).all() and (nact[Ts:, s] == 0).all()
    assert_hmm_equal(got, want, n_emit, "beam sweep")
    big_n = nact[:9, n_seg - 1]
    assert big_n[0] > big_n[-1] > 0, "the beam must bite: %s" % big_n
    if maxhmmpf >= 0:
        assert big_n[0] > maxhmmpf, "the histogram walk must run: %s" % big_n


# ---------------------------------------------------------------------------------------
# BASELINE.json config 2 at FULL size (1000 utterances x 998 frames, 5138 senones): properties
# that do not need the oracle on every frame, plus the oracle on a sample of utterances.

def test_full_size_properties(api, monkeypatch):
    import torch
    import zlib
    from oracle import oracle
    from pocketsphinx_b200.model import synth_feats, synth_ptm
    pm = synth_ptm(seed=0)
    U, T = 1000, 998
    feats = synth_feats(pm, U, T, seed=77)
    flat = np.ascontiguousarray(feats.reshape(U * T, pm.sumlen))
    off = api.Batch.offsets([T] * U)
    m = api.Model(pm)
    ctx = api.HmmContext(pm.tp, pm.sseq, pm.n_sen)
    H = pm.n_ciphone
    pl = api.PhoneLoop(ctx, pm.phone_ssid[:H], pm.phone_tmat[:H], 5, -1080, -1080, 0, 3.0)
    d_feats = torch.from_numpy(flat).cuda()

    def run(variant, pipe):
        monkeypatch.setenv("PSB_TOPN_VARIANT", str(variant))
        b = api.Batch(m, U, U * T)
        b.set_pipeline(pipe)
        best, pen = b.decode_host(pl, flat, off)
        scr = torch.empty((U * T, pm.n_sen), dtype=torch.int16, device="cuda")
        b.score_device(d_feats.data_ptr(), off, scr.data_ptr())
        b.sync()
        # a checksum of per-row checksums of the 10 GB score matrix, computed on the device
        w = torch.arange(1, pm.n_sen + 1, device="cuda", dtype=torch.int64)
        rows = torch.zeros(U * T, dtype=torch.int64, device="cuda")
        for a in range(0, U * T, 65536):
            rows[a:a + 65536] = (scr[a:a + 65536].to(torch.int64) * w).sum(1)
        sample = {u: scr[off[u]:off[u + 1]].cpu().numpy() for u in (0, 499, 999)}
        mins = scr.view(U * T, pm.n_sen).min(1).values.cpu().numpy()
        b.close()
        return best, pen, rows.cpu().numpy(), sample, mins

    best5, pen5, rows5, sample5, mins5 = run(5, 1)
    # every frame's best senone scores 0 (ptm_mgau.c:398-400) and the phone loop saw every frame
    assert (mins5 == 0).all()
    assert best5.shape == (U * T,) and pen5.shape == (U * T, H)
    # oracle on three whole utterances
    om = oracle.OracleModel(pm)
    for u, got in sample5.items():
        assert np.array_equal(got, om.score_utt(feats[u])), "utterance %d" % u
    # same bits from two ranges in flight
    best2, pen2, rows2, _, _ = run(5, 2)
    assert np.array_equal(rows5, rows2)
    assert np.array_equal(best5, best2) and np.array_equal(pen5, pen2)
    # and from the path without the recurrence over time (tensor-core filter + exact rescoring + tie fix-up)
    best6, pen6, rows6, _, _ = run(6, 1)
    assert np.array_equal(rows5, rows6)
    assert np.array_equal(best5, best6) and np.array_equal(pen5, pen6)
    best6p, pen6p, rows6p, _, _ = run(6, 3)                 # ... and with three sub-batches of it in flight on their own streams
    assert np.array_equal(rows5, rows6p)
    assert np.array_equal(best5, best6p) and np.array_equal(pen5, pen6p)
    # utterance order does not matter: reversed batch gives the reversed result
    monkeypatch.setenv("PSB_TOPN_VARIANT", "5")
    b = api.Batch(m, U, U * T)
    rbest, rpen = b.decode_host(pl, np.ascontiguousarray(feats[::-1].reshape(U * T, pm.sumlen)), off)
    assert np.array_equal(rbest.reshape(U, T)[::-1], best5.reshape(U, T))
    assert np.array_equal(rpen.reshape(U, T, H)[::-1], pen5.reshape(U, T, H))
    b.close(); pl.close(); ctx.close(); m.close()
    assert zlib.crc32(rows5.tobytes()) == zlib.crc32(rows2.tobytes())


# ---------------------------------------------------------------------------------------
# forced alignment (state_align_search.c) for batches

def test_align_goforward_matches_reference(api, en_us, en_us_dev):
    g, ga = golden("en_us_goforward.npz"), golden("en_us_align.npz")
    b = api.Batch(en_us_dev, 4, 1024)
    scr = b.score_host(g["feats"], np.array([0, 278], np.int32))          # our scores (bit-exact, tested above)
    b.close()
    ctx = api.HmmContext(en_us.tp, en_us.sseq, en_us.n_sen)
    tags = ["a", "b", "c"]
    utt_off = np.arange(len(tags) + 1, dtype=np.int32) * 278
    ph_off = np.concatenate([[0], np.cumsum([len(ga[t + "_ssid"]) for t in tags])]).astype(np.int32)
    status, st, du, sc = ctx.align(np.concatenate([scr] * len(tags)), utt_off, ph_off,
                                   np.concatenate([ga[t + "_ssid"] for t in tags]),
                                   np.concatenate([ga[t + "_tmatid"] for t in tags]))
    assert (status == 0).all()
    for k, t in enumerate(tags):
        sl = slice(ph_off[k] * 3, ph_off[k + 1] * 3)
        assert np.array_equal(st[sl], ga[t + "_start"]), t
        assert np.array_equal(du[sl], ga[t + "_dur"]), t
        assert np.array_equal(sc[sl], ga[t + "_score"]), t
    ctx.close()


@pytest.mark.parametrize("n_emit", [3, 5])
def test_align_batch_matches_oracle(api, n_emit):
    import torch
    from oracle import oracle
    from pocketsphinx_b200.model import synth_ptm
    pm = synth_ptm(seed=31, n_density=32, n_sen=300, n_emit_state=n_emit, skip_arcs=(n_emit == 5))
    rng = np.random.default_rng(17)
    n_phones = [1, 2, 5, 40, 150, 3, 12, 60, 7, 0]
    frames = [30, 3, 4, 200, 700, 300, 36, 190, 500, 10]      # some too short to reach the end
    ssid = [rng.integers(0, len(pm.sseq), n).astype(np.int32) for n in n_phones]
    tmat = [rng.integers(0, pm.tp.shape[0], n).astype(np.int32) for n in n_phones]
    scr = [rng.integers(0, 400, (t, pm.n_sen)).astype(np.int16) for t in frames]
    # renormalisation: one utterance with huge negative scores so that best_score sinks below the bound
    scr[8] = rng.integers(20000, 32000, (frames[8], pm.n_sen)).astype(np.int16)
    sf = [np.zeros(n, np.int32) for n in n_phones]
    ef = [np.full(n, 2**31 - 1, np.int32) for n in n_phones]
    # alignment constraints on utterance 7: phones pinned to windows of ~3 frames per phone
    for i in range(n_phones[7]):
        sf[7][i] = max(0, 3 * i - 4)
        ef[7][i] = 3 * i + 12
    utt_off = np.concatenate([[0], np.cumsum(frames)]).astype(np.int32)
    ph_off = np.concatenate([[0], np.cumsum(n_phones)]).astype(np.int32)
    ctx = api.HmmContext(pm.tp, pm.sseq, pm.n_sen)
    d_scr = torch.from_numpy(np.concatenate(scr)).cuda()
    status, st, du, sc = ctx.align(None, utt_off, ph_off, np.concatenate(ssid), np.concatenate(tmat),
                                   sf=np.concatenate(sf), ef=np.concatenate(ef), device_ptr=d_scr.data_ptr())
    n_ok = 0
    for u in range(len(frames)):
        sl = slice(ph_off[u] * n_emit, ph_off[u + 1] * n_emit)
        if n_phones[u] == 0:
            assert status[u] == -1
            continue
        rc, wst, wdu, wsc = oracle.align_run(pm.tp, pm.sseq, ssid[u], tmat[u], scr[u], sf=sf[u], ef=ef[u])
        assert status[u] == rc, "utterance %d: status %d, oracle %d" % (u, status[u], rc)
        assert np.array_equal(st[sl], wst) and np.array_equal(du[sl], wdu) and np.array_equal(sc[sl], wsc), "utterance %d" % u
        n_ok += rc == 0
    assert n_ok >= 5                                           # the test exercises successes and failures
    ctx.close()


# ---------------------------------------------------------------------------------------
# keyword spotting (kws_search.c) for batches

def test_kws_goforward_matches_reference(api, en_us, en_us_dev):
    import torch
    from oracle import oracle
    g, gk = golden("en_us_goforward.npz"), golden("en_us_kws.npz")
    b = api.Batch(en_us_dev, 4, 1024)
    scr = b.score_host(g["feats"], np.array([0, 278], np.int32))
    b.close()
    ctx = api.HmmContext(en_us.tp, en_us.sseq, en_us.n_sen)
    d_scr = torch.from_numpy(np.concatenate([scr, scr[:150]])).cuda()
    utt_off = np.array([0, 278, 428], np.int32)
    for tag in ("a", "b"):
        cfg = [gk[tag + "_" + k] for k in ("pl_ssid", "pl_tmat", "kp_off", "kp_thresh", "kp_ssid", "kp_tmat")]
        hits, n = ctx.kws(d_scr.data_ptr(), utt_off, *cfg, int(gk[tag + "_beam"]), int(gk[tag + "_plp"]))
        assert np.array_equal(oracle.kws_detections(hits[0]), gk[tag + "_det"]), tag     # the reference's own detections
        for u, (a, e) in enumerate(((0, 278), (0, 150))):
            want = oracle.kws_run(en_us.tp, en_us.sseq, *cfg, int(gk[tag + "_beam"]), int(gk[tag + "_plp"]), scr[a:e])
            assert n[u] == len(want) and np.array_equal(hits[u], want), (tag, u)
    ctx.close()


@pytest.mark.parametrize("n_emit", [3, 5])
def test_kws_batch_matches_oracle(api, n_emit):
    import torch
    from oracle import oracle
    from pocketsphinx_b200.model import synth_ptm
    pm = synth_ptm(seed=41, n_density=32, n_sen=300, n_emit_state=n_emit, skip_arcs=(n_emit == 5))
    rng = np.random.default_rng(23)
    n_pl = 30
    pl_ssid = rng.integers(0, len(pm.sseq), n_pl).astype(np.int32)
    pl_tmat = rng.integers(0, pm.tp.shape[0], n_pl).astype(np.int32)
    chains = [4, 1, 9, 0, 17]                                   # one empty keyphrase (word missing from the dictionary)
    kp_off = np.concatenate([[0], np.cumsum(chains)]).astype(np.int32)
    kp_ssid = rng.integers(0, len(pm.sseq), kp_off[-1]).astype(np.int32)
    kp_tmat = rng.integers(0, pm.tp.shape[0], kp_off[-1]).astype(np.int32)
    kp_thresh = np.array([-200, -3000, -100, 0, -50000], np.int32)
    frames = [120, 1, 60, 300]
    scr = [rng.integers(0, 300, (t, pm.n_sen)).astype(np.int16) for t in frames]
    utt_off = np.concatenate([[0], np.cumsum(frames)]).astype(np.int32)
    ctx = api.HmmContext(pm.tp, pm.sseq, pm.n_sen)
    d_scr = torch.from_numpy(np.concatenate(scr)).cuda()
    total_hits = 0
    for beam, plp in ((-1080, -23), (-150, -400)):
        hits, n = ctx.kws(d_scr.data_ptr(), utt_off, pl_ssid, pl_tmat, kp_off, kp_thresh, kp_ssid, kp_tmat, beam, plp)
        for u in range(len(frames)):
            want = oracle.kws_run(pm.tp, pm.sseq, pl_ssid, pl_tmat, kp_off, kp_thresh, kp_ssid, kp_tmat, beam, plp, scr[u])
            assert n[u] == len(want) and np.array_equal(hits[u], want), "utterance %d beam %d" % (u, beam)
            total_hits += len(want)
        # truncation: the count is still the full number
        h2, n2 = ctx.kws(d_scr.data_ptr(), utt_off, pl_ssid, pl_tmat, kp_off, kp_thresh, kp_ssid, kp_tmat, beam, plp, cap=3)
        assert np.array_equal(n2, n) and all(np.array_equal(a, b[:3]) for a, b in zip(h2, hits))
    assert total_hits > 50
    ctx.close()


# ---------------------------------------------------------------------------------------
# phone decoding (allphone_search.c, no phone LM) for batches

def test_allphone_goforward_matches_reference(api, en_us, en_us_dev):
    import torch
    from oracle import oracle
    g, ga = golden("en_us_goforward.npz"), golden("en_us_allphone.npz")
    b = api.Batch(en_us_dev, 4, 1024)
    scr = b.score_host(g["feats"], np.array([0, 278], np.int32))
    b.close()
    ctx = api.HmmContext(en_us.tp, en_us.sseq, en_us.n_sen)
    d_scr = torch.from_numpy(np.concatenate([scr, scr[:100]])).cuda()
    args = (ga["ssid"], ga["tmatid"], ga["succ_off"], ga["succ"], int(ga["start"]), int(ga["beam"]), int(ga["pbeam"]),
            int(ga["inspen"]))
    hist, n = ctx.allphone(d_scr.data_ptr(), np.array([0, 278, 378], np.int32), *args)
    assert n[0] == int(ga["n_history"])
    segs = oracle.allphone_backtrace(hist[0], ga["ci"], 277, int(ga["inspen"]))
    assert np.array_equal(segs, ga["segs"])                                     # the reference's own segmentation
    want, wn = oracle.allphone_run(en_us.tp, en_us.sseq, *args, scr[:100])
    assert n[1] == wn and np.array_equal(hist[1], want)
    ctx.close()


@pytest.mark.parametrize("n_emit", [3, 5])
def test_allphone_batch_matches_oracle(api, n_emit):
    import torch
    from oracle import oracle
    from pocketsphinx_b200.model import synth_ptm
    pm = synth_ptm(seed=51, n_density=32, n_sen=300, n_emit_state=n_emit, skip_arcs=(n_emit == 5))
    rng = np.random.default_rng(29)
    H = 300                                                     # sparse random graph, some nodes without successors
    ssid = rng.integers(0, len(pm.sseq), H).astype(np.int32)
    tmat = rng.integers(0, pm.tp.shape[0], H).astype(np.int32)
    deg = rng.integers(0, 12, H)
    succ_off = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    succ = np.concatenate([rng.choice(H, d, replace=False) for d in deg]).astype(np.int32)
    frames = [90, 1, 40, 200]
    scr = [rng.integers(0, 300, (t, pm.n_sen)).astype(np.int16) for t in frames]
    utt_off = np.concatenate([[0], np.cumsum(frames)]).astype(np.int32)
    ctx = api.HmmContext(pm.tp, pm.sseq, pm.n_sen)
    d_scr = torch.from_numpy(np.concatenate(scr)).cuda()
    total = 0
    for beam, pbeam, inspen in ((-1080, -1080, 0), (-300, -120, -35)):
        hist, n = ctx.allphone(d_scr.data_ptr(), utt_off, ssid, tmat, succ_off, succ, 7, beam, pbeam, inspen)
        for u in range(len(frames)):
            want, wn = oracle.allphone_run(pm.tp, pm.sseq, ssid, tmat, succ_off, succ, 7, beam, pbeam, inspen, scr[u])
            assert n[u] == wn and np.array_equal(hist[u], want), "utterance %d beam %d" % (u, beam)
            total += wn
        h2, n2 = ctx.allphone(d_scr.data_ptr(), utt_off, ssid, tmat, succ_off, succ, 7, beam, pbeam, inspen, cap=5)
        assert np.array_equal(n2, n) and all(np.array_equal(a, b[:5]) for a, b in zip(h2, hist))
    assert total > 1000
    ctx.close()


def test_allphone_lm_goforward_matches_reference(api, en_us, en_us_dev):
    """With the shipped phone LM (dense score tables out of the reference's LM object)."""
    import torch
    from oracle import oracle
    g, ga = golden("en_us_goforward.npz"), golden("en_us_allphone.npz")
    b = api.Batch(en_us_dev, 4, 1024)
    scr = b.score_host(g["feats"], np.array([0, 278], np.int32))
    b.close()
    ctx = api.HmmContext(en_us.tp, en_us.sseq, en_us.n_sen)
    d_scr = torch.from_numpy(np.concatenate([scr, scr[40:160]])).cuda()
    args = (ga["ssid"], ga["tmatid"], ga["succ_off"], ga["succ"], int(ga["start"]), int(ga["beam"]), int(ga["pbeam"]),
            ga["ci"], ga["lm_bg"], ga["lm_tg"])
    hist, n = ctx.allphone_lm(d_scr.data_ptr(), np.array([0, 278, 398], np.int32), *args)
    assert n[0] == int(ga["lm_n_history"])
    assert np.array_equal(oracle.allphone_backtrace_lm(hist[0], ga["ci"], 277), ga["lm_segs"])   # the reference's segmentation
    want, wn = oracle.allphone_lm_run(en_us.tp, en_us.sseq, *args, scr[40:160])
    assert n[1] == wn and np.array_equal(hist[1], want)
    ctx.close()
