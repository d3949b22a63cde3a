"""Forced alignment (SURVEY 8f rank 4: the `return_logits` consumer, kraken/tasks/align.py:111-137).

CPU: oracle/align_oracle.py against the outputs of the reference's own get_trellis / backtrack / merge_repeats (bit for bit,
tests/golden/ref_align.npz) and against the committed goldens generated from the reference (tests/golden/align_cases.npz).
GPU: `kb_forced_align` through the C ABI against the oracle - token indices and frame ranges exact, scores within 1e-5."""
import hashlib
import os

import numpy as np
import pytest
import torch

import align_oracle as ao

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'align_cases.npz')


def random_case(rng, C, T, J, peaky=True):
    """(C, T) probabilities as the recogniser emits them and a label sequence; `peaky`: the transcription's labels win their frames"""
    z = rng.standard_normal((C, T)).astype(np.float32) * 2
    tokens = rng.integers(1, C, J)
    if peaky and J:
        cuts = np.sort(rng.choice(np.arange(1, T), size=min(2 * J, T - 1), replace=False))
        for k in range(min(J, len(cuts) // 2)):
            z[tokens[k], cuts[2 * k]:cuts[2 * k + 1]] += 6
        z[0] += 1
    p = torch.from_numpy(z).softmax(0)
    return p, [int(t) for t in tokens]


def test_oracle_is_the_reference_bit_for_bit():
    """120 random cases against the reference's get_trellis / backtrack / merge_repeats on them (tests/golden/ref_align.npz, generated
    by oracle/make_reference_checks.py).  Where this CPU's torch softmax reproduces the reference's probabilities bit for bit, the
    trellis (sha256 of its bytes), path and segments are compared exactly.  Elsewhere the probabilities and emissions differ in the
    last bits: token and frame indices stay exact, the trellis sum and the scores agree to float32 rounding."""
    g = np.load(os.path.join(os.path.dirname(GOLDEN), 'ref_align.npz'))
    rng = np.random.default_rng(0)
    n_failed, n_exact, pi, si = 0, 0, 0, 0
    for it in range(len(g['path_n'])):
        C = int(rng.integers(3, 60)); T = int(rng.integers(4, 160)); J = int(rng.integers(1, max(2, T // 2)))
        p, tokens = random_case(rng, C, T, J, peaky=bool(it % 3))
        exact = hashlib.sha256(p.numpy().tobytes()).digest() == g['probs_sha'][it].tobytes()
        n_exact += exact
        em = ao.emission_from_probs(p)
        tr = ao.trellis(em, tokens)
        assert tr.shape == tuple(g['trellis_shape'][it]), it
        if exact:
            assert hashlib.sha256(tr.tobytes()).digest() == g['trellis_sha'][it].tobytes(), it
        assert np.isclose(tr[np.isfinite(tr)].astype(np.float64).sum(), g['trellis_sum'][it], rtol=1e-6, atol=1e-4), it
        path = ao.backtrack(tr, em, tokens)
        npath, nsegs = int(g['path_n'][it]), int(g['segs_n'][it])
        if npath < 0:
            assert path is None
            n_failed += 1
            continue
        want = [(int(a), int(b), float(s)) for (a, b), s in zip(g['path_ij'][pi:pi + npath], g['path_score'][pi:pi + npath])]
        segs = ao.merge_repeats(path)
        want_segs = [(int(a), int(b), int(c), float(s)) for (a, b, c), s in zip(g['seg_lse'][si:si + nsegs], g['seg_score'][si:si + nsegs])]
        if exact:
            assert path == want, it
            assert segs == want_segs, it
        else:
            assert [q[:2] for q in path] == [q[:2] for q in want], it
            assert np.allclose([q[2] for q in path], [q[2] for q in want], rtol=1e-6, atol=0), it
            assert [s[:3] for s in segs] == [s[:3] for s in want_segs], it
            assert np.allclose([s[3] for s in segs], [s[3] for s in want_segs], rtol=1e-6, atol=0), it
        pi, si = pi + npath, si + nsegs
    assert it == 119 and n_failed < 120 and pi == len(g['path_ij']) and si == len(g['seg_lse'])
    print(f'{n_exact} of 120 cases with bit-identical probabilities')


def test_oracle_against_the_goldens():
    g = np.load(GOLDEN)
    for k in range(int(g['n_cases'])):
        p = torch.from_numpy(g[f'probs_{k}']); tokens = g[f'tokens_{k}'].tolist()
        status, segs = ao.align_line(p, tokens)
        assert status == int(g[f'status_{k}']), k
        if status > 0:
            assert [s[0] for s in segs] == g[f'seg_token_{k}'].tolist()
            assert [s[1] for s in segs] == g[f'seg_start_{k}'].tolist()
            assert [s[2] for s in segs] == g[f'seg_end_{k}'].tolist()
            assert np.array_equal(np.array([s[3] for s in segs], np.float64), g[f'seg_score_{k}'])


def test_oracle_edge_cases():
    rng = np.random.default_rng(2)
    p, tokens = random_case(rng, 12, 9, 5)
    assert ao.align_line(p, tokens) == (ao.TOO_SHORT, [])                   # T < 2 J
    with pytest.raises(IndexError):
        ao.align_line(p, [])
    p, tokens = random_case(rng, 12, 10, 5)                                 # T == 2 J is accepted
    assert ao.align_line(p, tokens)[0] != ao.TOO_SHORT
    # one token: one segment (where it lands is the reference's business: its emission is the log-softmax of PROBABILITIES, align.py:119)
    z = np.full((5, 30), -4, np.float32); z[0] = 2; z[3, 10:14] = 8
    st, segs = ao.align_line(torch.from_numpy(z).softmax(0), [3])
    assert st == 1 and segs[0][0] == 0 and 0 <= segs[0][1] < segs[0][2] <= 30


def test_wrapper_argument_errors():
    import kraken_b200 as kb
    from kraken_b200 import align
    m = kb.TorchVGSLModel(vgsl='[1,16,0,1 Cr3,3,8 Mp2,2 S1(1x0)1,3 Lbx16 O1c12]')
    m.init_weights()
    rec = kb.TorchSeqRecognizer(m, device=None)                         # argument checks come before any device work
    x = torch.rand(2, 1, 16, 64)
    with pytest.raises(ValueError):
        align.forced_align(rec, x, None)                                   # neither texts nor labels
    with pytest.raises(ValueError):
        align.forced_align(rec, x, None, texts=['a', 'b'])                 # no codec
    with pytest.raises(ValueError):
        align.forced_align_probs(torch.rand(2, 5, 9), [[1], [2]], lens=[9])          # one length per line
    with pytest.raises(IndexError):
        align.forced_align_probs(torch.rand(1, 5, 9), [[]])
    with pytest.raises(ValueError):
        align.forced_align_probs(torch.rand(2, 5, 9), [[1]])


CFG2 = '[1,48,0,1 Cr3,3,32 Mp2,2 Cr3,3,64 Mp2,2 S1(1x0)1,3 Lbx256 O1c200]'


def _oracle_batch(om, x, lens, labels, orig_widths=None, padding=0):
    """reference steps on the oracle network: probs = softmax(nn(x)) (rpred.py:225-227) -> per line align_line on [:, :olen] (:200)"""
    import vgsl_oracle as vo
    _, probs, ol, _ = vo.rec_predict(om, x, lens)                          # (N, C, T) probabilities = `self.outputs`
    res = []
    for i, lab in enumerate(labels):
        T = int(ol[i]) if ol is not None else probs.shape[-1]
        st, segs = ao.align_line(probs[i, :, :T], lab)
        if st > 0 and orig_widths is not None:
            wi = int(lens[i]); ns = wi / T; isc = orig_widths[i] / (wi - 2 * padding)
            segs = [(s[0], ao.scale_val(s[1], ns, isc, padding, orig_widths[i]), ao.scale_val(s[2], ns, isc, padding, orig_widths[i]), s[3]) for s in segs]
        res.append((st, segs))
    return res


@pytest.mark.gpu
@pytest.mark.parametrize('spec,n,h,w', [(CFG2, 24, 48, 400), ('[1,16,0,1 Cr3,3,32 Mp2,2 S1(1x0)1,3 Lbx64 O1c40]', 9, 16, 120)])
def test_gpu_forced_align_equals_oracle(spec, n, h, w):
    import kraken_b200 as kb
    import vgsl_oracle as vo
    from kraken_b200 import align
    om = vo.OracleModel(spec)
    wts = om.init_like_reference(21)
    g = torch.Generator().manual_seed(21)
    lens = torch.randint(w // 3, w + 1, (n,), generator=g)
    lens[0] = w
    x = torch.rand(n, 1, h, w, generator=g)
    for i, l in enumerate(lens.tolist()):
        x[i, ..., l:] = 0
    m = kb.TorchVGSLModel(vgsl=spec)
    m.load_state_dict(wts)
    rec = kb.TorchSeqRecognizer(m, device='cuda:0')
    C = m.infer_dims(n, h, w)[1]
    rng = np.random.default_rng(21)
    _, _, ol, _ = vo.rec_predict(om, x, lens)
    labels = []
    for i in range(n):
        T = int(ol[i])
        J = int(rng.integers(1, max(2, T // 2 + 1)))
        if i == 1:
            J = T // 2 + 3                                                  # too short for its transcription
        if i == 2:
            J = T // 2                                                      # exactly 2 J frames
        labels.append(rng.integers(1, C, J).tolist())
    ref = _oracle_batch(om, x, lens, labels)
    try:
        got = align.forced_align(rec, x.cuda(), lens, labels=labels)
        failed = False
    except ValueError:
        failed = True
    assert failed == any(st == ao.FAILED for st, _ in ref)
    if not failed:
        for i, (st, segs) in enumerate(ref):
            if st == ao.TOO_SHORT:
                assert got[i] == []
                continue
            assert [(s[0], s[1], s[2]) for s in got[i]] == [(s[0], s[1], s[2]) for s in segs], i
            assert np.allclose([s[3] for s in got[i]], [s[3] for s in segs], rtol=1e-5, atol=1e-7), i
        assert got[1] == []
    # pixel positions in the original line images (`_scale_val`), host lines this time
    ow = [int(v) for v in (lens * 3 + 5).tolist()]
    pad = 4
    ref = _oracle_batch(om, x, lens, labels, ow, pad)
    if not any(st == ao.FAILED for st, _ in ref):
        got = align.forced_align(rec, x, lens, labels=labels, orig_widths=ow, padding=pad)
        for i, (st, segs) in enumerate(ref):
            if st > 0:
                assert [(s[0], s[1], s[2]) for s in got[i]] == [(s[0], s[1], s[2]) for s in segs], i


@pytest.mark.gpu
def test_gpu_forced_align_texts_and_errors():
    import kraken_b200 as kb
    from kraken_b200 import align
    spec = '[1,16,0,1 Cr3,3,16 Mp2,2 S1(1x0)1,3 Lbx32 O1c12]'
    m = kb.TorchVGSLModel(vgsl=spec)
    m.init_weights()
    codec = kb.PytorchCodec('abcdefghijk')
    rec = kb.TorchSeqRecognizer(m, device='cuda:0')
    rec.codec = codec
    x = torch.rand(3, 1, 16, 96)
    texts = ['abc', 'kja?b', 'hhhh']                                       # '?' is not in the codec: skipped by encode (codec.py:140-144)
    by_text = align.forced_align(rec, x, None, texts=texts)
    by_lab = align.forced_align(rec, x, None, labels=[codec.encode(t).tolist() for t in texts])
    for t, a, b in zip(texts, by_text, by_lab):
        assert [(t[s[0]], s[1], s[2]) for s in b] == [(s[0], s[1], s[2]) for s in a]
    with pytest.raises(IndexError):
        align.forced_align(rec, x, None, labels=[[1], [], [2]])
    with pytest.raises(Exception):
        align.forced_align(rec, x, None, labels=[[1], [99], [2]])         # label outside the model's classes


@pytest.mark.gpu
def test_gpu_forced_align_probs_equals_the_reference_goldens():
    """tests/golden/align_cases.npz was produced by the reference's own get_trellis / backtrack / merge_repeats (oracle/make_align_golden.py):
    probabilities in, segments out, one case per call and all cases of one shape in one ragged batch."""
    from kraken_b200 import align
    g = np.load(GOLDEN)
    for k in range(int(g['n_cases'])):
        p = torch.from_numpy(g[f'probs_{k}']); tokens = g[f'tokens_{k}'].tolist()
        st = int(g[f'status_{k}'])
        for src in (p, p.cuda()):
            got = align.forced_align_probs(src, [tokens])[0]
            if st == ao.TOO_SHORT:
                assert got == []
                continue
            assert st > 0
            assert [s[0] for s in got] == g[f'seg_token_{k}'].tolist(), k
            assert [s[1] for s in got] == g[f'seg_start_{k}'].tolist(), k
            assert [s[2] for s in got] == g[f'seg_end_{k}'].tolist(), k
            assert np.allclose([s[3] for s in got], g[f'seg_score_{k}'], rtol=1e-5, atol=1e-7), k
    # a ragged batch: the first 40 / 25 / 64 frames of one probability tensor, different label sequences
    rng = np.random.default_rng(8)
    p, _ = random_case(rng, 50, 64, 4)
    lens = [40, 25, 64]
    labels = [rng.integers(1, 50, j).tolist() for j in (7, 12, 30)]
    got = align.forced_align_probs(torch.stack([p, p, p]).cuda(), labels, lens=lens)
    for i in range(3):
        st, segs = ao.align_line(p[:, :lens[i]], labels[i])
        assert st > 0 and [(s[0], s[1], s[2]) for s in got[i]] == [(s[0], s[1], s[2]) for s in segs]
        assert np.allclose([s[3] for s in got[i]], [s[3] for s in segs], rtol=1e-5, atol=1e-7)
    # the per-record form: every record its own length
    recs = [p[:, :l] for l in lens]
    assert align.align_records(recs, labels) == got
    assert align.align_records([r[:, None, :].cuda() for r in recs], labels) == got
