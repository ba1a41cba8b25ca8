"""Reference-keyframe matching against a device-resident keyframe set (sslpl_kfset + sslpl_match_ref_kf_batch_device): every frame
of a device batch matched against the keyframe slot it names, as Tracking::TrackReferenceKeyFrame does with
ORBmatcher(0.9, true).SearchByBoW(KF, F) and LSDmatcher().SearchByProjection(KF, F).  Checked against the reference itself, the
single-pair device calls and the consecutive-pair batch calls."""
import types
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

B, NL, LEVELSUP, KL, KD = 8, 40, 1, 3, 10
REF = [-1, 0, 0, 1, 2, -1, 3, 1]           # frame f -> slot; repeated slots and frames without a reference keyframe
KF_FRAMES = [0, 2, 3, 5]                    # slot -> batch frame it was stored from
THIN = 4                                    # frame whose line count the tests cut to 1


@pytest.fixture(scope="module")
def S(pkg, oracle, synth):
    frames = synth.batch(640, 480, B)
    ext = pkg.ORBextractor(1000, 1.2, 8, 20, 7, max_width=640, max_height=480, max_batch=B)
    kk, d, n = ext.extract_batch(frames)
    ls = pkg.LineSegment(NL, max_width=640, max_height=480, max_batch=B)
    _, ld, _, nl = ls.extract_batch(frames)
    dfr = torch.from_numpy(frames).cuda()
    ext.extract_batch_device(dfr.data_ptr(), B, 640, 480, 640, 640 * 480); ext.sync()
    ls.extract_batch_device(dfr.data_ptr(), B, 640, 480, 640, 640 * 480); ls.sync()
    kps, desc, dn, cap = ext.device_results()
    _, ldesc, _, _, capl = ls.device_results()
    nl = nl.copy(); nl[THIN] = 1                                      # fewer than 2 frame lines: no line match
    d_nl = torch.from_numpy(nl.astype(np.int32)).cuda()
    parent, ndesc, weight, is_leaf = pkg.Vocabulary.random_arrays(KD, KL, seed=4, stop_fraction=0.05)
    voc = pkg.Vocabulary(KD, KL, parent, ndesc, weight, is_leaf)
    fv = []
    for f in range(B):
        _, node, w = oracle.vocab_transform(KL, parent, ndesc, weight, is_leaf, d[f, :n[f]], LEVELSUP)
        fv.append(pkg.Vocabulary.feature_vector(node, w))
    mt = pkg.Matcher(max_features=cap, max_lines=NL, max_nodes=voc.level_nodes(LEVELSUP) + 1, max_batch=B)
    kfs = pkg.KeyframeSet(len(KF_FRAMES), cap, capl)
    rng = np.random.default_rng(7)
    state, has_ml = [], []
    for s, f in enumerate(KF_FRAMES):
        kfs.store_device(mt, s, desc, kps, dn, cap, ldesc, d_nl.data_ptr(), capl, f, voc, LEVELSUP)
        st = (rng.random(n[f]) < 0.7).astype(np.uint8)               # 1 = good MapPoint; some of the others are bad MapPoints (2)
        st[np.flatnonzero(st == 0)[::2]] = 2
        state.append(st); has_ml.append((rng.random(nl[f]) < 0.7).astype(np.uint8))
        kfs.set_masks(s, (st == 1).astype(np.uint8), has_ml[-1])
    return types.SimpleNamespace(kk=kk, d=d, n=n, ld=ld, nl=nl, kps=kps, desc=desc, dn=dn, cap=cap, ldesc=ldesc, d_nl=d_nl, capl=capl,
                                 voc=voc, fv=fv, mt=mt, kfs=kfs, state=state, has_ml=has_ml, ext=ext, ls=ls, dfr=dfr)


def run(S, kfs, ref, mt=None, ratio=0.9, ori=True):
    mt = mt or S.mt
    d_ref = torch.tensor(ref, dtype=torch.int32, device="cuda")
    nf = len(ref)
    m = torch.full((nf, S.cap), -7, dtype=torch.int32, device="cuda"); nm = torch.full((nf,), -7, dtype=torch.int32, device="cuda")
    lm = torch.full((nf, S.capl), -7, dtype=torch.int32, device="cuda"); nlm = torch.full((nf,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()                                          # the fills run on torch's stream, the matcher on its own
    mt.match_ref_kf_batch_device(kfs, d_ref.data_ptr(), nf, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, S.voc, LEVELSUP,
                                 ratio, ori, m.data_ptr(), nm.data_ptr(), lm.data_ptr(), nlm.data_ptr())
    mt.sync()
    return m.cpu().numpy(), nm.cpu().numpy(), lm.cpu().numpy(), nlm.cpu().numpy()


def single_pair(pkg, S, kf, f, valid, has_ml):
    """What sslpl_search_by_bow + sslpl_line_match mode 0 give for (KF = batch frame kf, frame f)."""
    ctx = pkg.Matcher(max_features=S.cap, max_lines=S.capl, max_nodes=S.voc.level_nodes(LEVELSUP) + 1)
    n_p, m_p = pkg.ORBmatcher(0.9, True, ctx).SearchByBoW(S.d[kf, :S.n[kf]], S.fv[kf], valid, S.kk[kf, :S.n[kf]]["angle"],
                                                          S.d[f, :S.n[f]], S.fv[f], S.kk[f, :S.n[f]]["angle"])
    n_l, m_l = 0, np.full(S.nl[f], -1, np.int32)
    if S.nl[f] >= 2:
        n_l, m_l = pkg.LSDmatcher(ctx).SearchByProjection(S.ld[kf, :S.nl[kf]], has_ml, S.ld[f, :S.nl[f]])
    return n_p, m_p, n_l, m_l


def check_frame(got, f, n_p, m_p, n_l, m_l, S):
    m, nm, lm, nlm = got
    assert nm[f] == n_p and np.array_equal(m[f, :S.n[f]], m_p) and (m[f, S.n[f]:] == -1).all(), f
    assert nlm[f] == n_l and np.array_equal(lm[f, :S.nl[f]], m_l) and (lm[f, S.nl[f]:] == -1).all(), f


def check_no_reference(got, f):
    m, nm, lm, nlm = got
    assert nm[f] == 0 and nlm[f] == 0 and (m[f] == -1).all() and (lm[f] == -1).all(), f


def test_equals_reference_search_by_bow_and_line_projection(S):
    from oracle import ref
    if not ref.available():
        pytest.skip("oracle/_ref/libref.so was not built")
    got = run(S, S.kfs, REF)
    for f, s in enumerate(REF):
        if s < 0:
            check_no_reference(got, f); continue
        kf = KF_FRAMES[s]
        n_r, m_r = ref.search_by_bow(S.d[kf, :S.n[kf]], S.kk[kf, :S.n[kf]], S.d[f, :S.n[f]], S.kk[f, :S.n[f]], S.fv[kf], S.fv[f],
                                     S.state[s], 0.9, True)
        n_l, m_l = 0, np.full(S.nl[f], -1, np.int32)
        if S.nl[f] >= 2:
            n_l, m_l, _ = ref.line_match(0, S.ld[kf, :S.nl[kf]], S.ld[f, :S.nl[f]], S.has_ml[s])
        check_frame(got, f, n_r, m_r, n_l, m_l, S)
    assert got[1].sum() > 0 and got[3].sum() > 0


def test_equals_single_pair_calls_and_host_store(pkg, S):
    got = run(S, S.kfs, REF)
    for f, s in enumerate(REF):
        if s >= 0:
            check_frame(got, f, *single_pair(pkg, S, KF_FRAMES[s], f, (S.state[s] == 1).astype(np.uint8), S.has_ml[s]), S)
    # the same keyframes stored from host buffers
    hk = pkg.KeyframeSet(len(KF_FRAMES), S.cap, S.capl)
    for s, kf in enumerate(KF_FRAMES):
        hk.store(S.mt, s, S.d[kf, :S.n[kf]], S.kk[kf, :S.n[kf]]["angle"], S.ld[kf, :S.nl[kf]], S.voc, LEVELSUP)
        hk.set_masks(s, (S.state[s] == 1).astype(np.uint8), S.has_ml[s])
    got_h = run(S, hk, REF)
    assert all(np.array_equal(a, b) for a, b in zip(got, got_h))


@pytest.mark.parametrize("ratio,ori", [(0.9, True), (0.7, False)])
def test_consecutive_keyframes_equal_the_pair_batch(pkg, S, ratio, ori):
    ks = pkg.KeyframeSet(B - 1, S.cap, S.capl)
    for s in range(B - 1):
        ks.store_device(S.mt, s, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, s, S.voc, LEVELSUP)
    got = run(S, ks, [-1] + list(range(B - 1)), ratio=ratio, ori=ori)
    pm = torch.empty((B - 1, S.cap), dtype=torch.int32, device="cuda"); pn = torch.empty((B - 1,), dtype=torch.int32, device="cuda")
    plm = torch.empty((B - 1, S.capl), dtype=torch.int32, device="cuda"); pln = torch.zeros((B - 1,), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    S.mt.match_bow_batch_device_vocab(S.desc, S.kps, S.dn, B, S.cap, S.voc, LEVELSUP, ratio, ori, pm.data_ptr(), pn.data_ptr())
    S.mt.match_lines_batch_device(S.ldesc, S.d_nl.data_ptr(), B, S.capl, plm.data_ptr(), pln.data_ptr())
    S.mt.sync()
    check_no_reference(got, 0)
    assert np.array_equal(got[0][1:], pm.cpu().numpy()) and np.array_equal(got[1][1:], pn.cpu().numpy())
    assert np.array_equal(got[2][1:], plm.cpu().numpy()) and np.array_equal(got[3][1:], pln.cpu().numpy())


def test_mask_and_slot_updates(pkg, S):
    ks = pkg.KeyframeSet(2, S.cap, S.capl)
    ref = [0, 1, 1, 0, 1, 1, 0, 1]
    for s, kf in enumerate((1, 4)):
        ks.store_device(S.mt, s, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, kf, S.voc, LEVELSUP)
    ones = lambda k: (np.ones(S.n[k], np.uint8), np.ones(S.nl[k], np.uint8))
    before = run(S, ks, ref)
    for f, s in enumerate(ref):
        check_frame(before, f, *single_pair(pkg, S, (1, 4)[s], f, *ones((1, 4)[s])), S)
    # masks of slot 1 only: slot 0's frames are untouched, slot 1's follow the new masks
    rng = np.random.default_rng(3)
    v = (rng.random(S.n[4]) < 0.5).astype(np.uint8); h = (rng.random(S.nl[4]) < 0.5).astype(np.uint8)
    ks.set_masks(1, v, h)
    after = run(S, ks, ref)
    changed = 0
    for f, s in enumerate(ref):
        if s == 0:
            assert all(np.array_equal(a[f], b[f]) for a, b in zip(before, after)), f
        else:
            check_frame(after, f, *single_pair(pkg, S, 4, f, v, h), S)
            changed += not all(np.array_equal(a[f], b[f]) for a, b in zip(before, after))
    assert changed > 0
    # storing again replaces the keyframe (and resets its masks)
    ks.store_device(S.mt, 1, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, 6, S.voc, LEVELSUP)
    again = run(S, ks, ref)
    for f, s in enumerate(ref):
        if s == 1:
            check_frame(again, f, *single_pair(pkg, S, 6, f, *ones(6)), S)
    # a cleared slot matches nothing; the other slot is untouched
    ks.clear(1)
    cleared = run(S, ks, ref)
    for f, s in enumerate(ref):
        if s == 1:
            check_no_reference(cleared, f)
        else:
            assert all(np.array_equal(a[f], b[f]) for a, b in zip(again, cleared)), f


def test_argument_errors_enqueue_nothing(pkg, S):
    def arg_error(fn, *a, **kw):
        with pytest.raises(pkg.SslplError, match=r"sslpl error -1:"):
            fn(*a, **kw)

    ks = pkg.KeyframeSet(2, S.cap, S.capl)
    ks.store_device(S.mt, 0, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, 2, S.voc, LEVELSUP)
    S.mt.sync()
    launches = S.mt.launch_count
    # slots out of range
    arg_error(ks.store_device, S.mt, 2, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, 0, S.voc, LEVELSUP)
    arg_error(ks.store_device, S.mt, -1, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, 0, S.voc, LEVELSUP)
    arg_error(ks.store, S.mt, 2, S.d[0, :S.n[0]], S.kk[0, :S.n[0]]["angle"], S.ld[0, :S.nl[0]], S.voc, LEVELSUP)
    arg_error(ks.set_masks, 2, None, None)
    arg_error(ks.clear, 2)
    arg_error(ks.set_masks, 0, np.ones(S.cap + 1, np.uint8), None)
    # store capacity
    small = pkg.KeyframeSet(1, S.cap - 1, S.capl)
    arg_error(small.store_device, S.mt, 0, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, 0, S.voc, LEVELSUP)
    assert S.mt.launch_count == launches

    other = pkg.Vocabulary.random(KD, KL, seed=9)
    d_ref = torch.zeros((B,), dtype=torch.int32, device="cuda")
    outs = [torch.full((B, S.cap), -7, dtype=torch.int32, device="cuda"), torch.full((B,), -7, dtype=torch.int32, device="cuda"),
            torch.full((B, S.capl), -7, dtype=torch.int32, device="cuda"), torch.full((B,), -7, dtype=torch.int32, device="cuda")]
    torch.cuda.synchronize()

    def call(mt=S.mt, kfs=ks, nf=B, cap=S.cap, capl=S.capl, voc=S.voc, levelsup=LEVELSUP):
        mt.match_ref_kf_batch_device(kfs, d_ref.data_ptr(), nf, S.desc, S.kps, S.dn, cap, S.ldesc, S.d_nl.data_ptr(), capl, voc, levelsup,
                                     0.9, True, *(o.data_ptr() for o in outs))

    arg_error(call, voc=other)                                         # slot 0 was built with another tree
    arg_error(call, levelsup=LEVELSUP + 1)                             # ... or levelsup
    arg_error(call, nf=B + 2)                                          # nframes over max_batch + 1
    arg_error(call, nf=0)
    arg_error(call, cap=S.mt.max_features + 65)
    arg_error(call, capl=S.mt.max_lines + 65)
    wide = pkg.KeyframeSet(1, S.cap, S.mt.max_lines + 65)
    arg_error(call, kfs=wide)                                          # the set's lines per keyframe over the matcher's knn table
    S.mt.sync()
    assert S.mt.launch_count == launches
    assert all((o.cpu() == -7).all() for o in outs)
    ks.clear(0)
    call(voc=other)                                                    # an empty set accepts any tree
    S.mt.sync()
    assert (outs[0].cpu() == -1).all() and (outs[1].cpu() == 0).all()


def test_sets_on_other_devices_are_refused(pkg, S):
    if pkg.device_count() < 2:
        pytest.skip("needs two GPUs")
    ks1 = pkg.KeyframeSet(1, S.cap, S.capl, device=1)
    voc1 = pkg.Vocabulary.random(KD, KL, seed=4, device=1)
    with pytest.raises(pkg.SslplError, match=r"sslpl error -1:"):
        ks1.store_device(S.mt, 0, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, 0, S.voc, LEVELSUP)
    d_ref = torch.zeros((B,), dtype=torch.int32, device="cuda")
    o = torch.empty((B, max(S.cap, S.capl)), dtype=torch.int32, device="cuda")
    for kfs, voc in ((ks1, S.voc), (S.kfs, voc1)):
        with pytest.raises(pkg.SslplError, match=r"sslpl error -1:"):
            S.mt.match_ref_kf_batch_device(kfs, d_ref.data_ptr(), B, S.desc, S.kps, S.dn, S.cap, S.ldesc, S.d_nl.data_ptr(), S.capl, voc,
                                           LEVELSUP, 0.9, True, o.data_ptr(), o.data_ptr(), o.data_ptr(), o.data_ptr())
