"""Generates the fixtures with which the CPU tests compare the oracle and the host-side mirrors against the UNMODIFIED reference
(imported through oracle/refshim.py), so that those comparisons run wherever the tests run.  TEST INFRASTRUCTURE ONLY.
Usage: python oracle/make_reference_checks.py

  tests/golden/ref_oracle_specs.npz    seven VGSL specs (recognition, segmentation, nesting, legacy clstm / ocropy cells): named spec,
                                       output shape, `nn(x, lens)` of the reference model loaded with the oracle's seeded weights
                                       (output lengths and a fixed sample of at most 256 logits), greedy_decoder on the softmax of
                                       all of them, or the fact that the reference raised
  tests/golden/ref_align.npz           get_trellis / backtrack / merge_repeats on the 120 cases tests/test_align.py generates:
                                       sha256 of the inputs and of the trellis bytes, the sum of the finite trellis entries, the path
                                       and the merged segments
  tests/golden/ref_codec.json          PytorchCodec.encode / decode on seeded random streams over three charsets
  tests/golden/ref_scale_val.npz       VGSLRecognitionInference._scale_val on seeded random positions and scales
  tests/golden/{overfit.mlmodel, model_small.mlmodel, model_small.safetensors, model_small_fp16.safetensors}
                                       the reference's own model files (data fixtures, copied unchanged)
"""
import hashlib
import json
import os
import random
import shutil
import sys
import types
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, 'tests', 'golden')
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import refshim  # noqa: E402

refshim.install()
warnings.simplefilter('ignore')

import vgsl_oracle as vo  # noqa: E402

from test_oracle import ORACLE_LENS, ORACLE_SPECS, logit_sample, oracle_case_input  # noqa: E402  (the cases the tests use)

N_ALIGN = 120


def oracle_specs():
    from kraken.lib.ctc_decoder import greedy_decoder
    from kraken.lib.vgsl.model import TorchVGSLModel
    d = {'specs': np.array(ORACLE_SPECS)}
    for k, sp in enumerate(ORACLE_SPECS):
        om = vo.OracleModel(sp)
        w = om.init_like_reference(k)
        ref = TorchVGSLModel(vgsl=sp)
        ref.load_state_dict({n: v.float() for n, v in w.items()})
        ref.eval()
        d[f'named_spec_{k}'] = np.array(ref.user_metadata['vgsl'])
        d[f'output_{k}'] = np.asarray(ref.output, np.int64)
        x = oracle_case_input(k, om)
        for li, lens in enumerate(ORACLE_LENS):
            key = f'{k}_{li}'
            try:
                with torch.inference_mode():
                    ro, rl = ref.nn(x, None if lens is None else torch.tensor(lens))
            except Exception:
                d[f'raises_{key}'] = np.bool_(True)
                continue
            d[f'raises_{key}'] = np.bool_(False)
            d[f'logits_{key}'] = ro.numpy().reshape(-1)[logit_sample(ro.numel(), k)]
            if rl is not None:
                d[f'olens_{key}'] = rl.numpy().astype(np.int64)
            oo, _ = om.forward(x, None if lens is None else torch.tensor(lens))
            assert torch.equal(oo, ro), (sp, lens)                  # same machine, same ATen build: bit for bit
            if ro.shape[2] == 1:
                p = ro.softmax(1).squeeze(2)
                ll = rl if rl is not None else torch.tensor([p.shape[-1]] * 3)
                dec = greedy_decoder(p, ll)
                d[f'dec_{key}'] = np.array([(i, l, s, e, c) for i, line in enumerate(dec) for (l, s, e, c) in line], np.float64).reshape(-1, 5)
    np.savez_compressed(os.path.join(OUT, 'ref_oracle_specs.npz'), **d)


def align_cases():
    from kraken.tasks import align as ra
    from test_align import random_case
    rng = np.random.default_rng(0)
    sha_p, sha_tr, tr_shape, tr_sum, paths, segs_all, path_n, segs_n = [], [], [], [], [], [], [], []
    for it in range(N_ALIGN):
        C = int(rng.integers(3, 60)); T = int(rng.integers(4, 160)); J = int(rng.integers(1, max(2, T // 2)))
        p, tokens = random_case(rng, C, T, J, peaky=bool(it % 3))
        labels = torch.tensor(tokens, dtype=torch.int32).long()
        em = p.squeeze().log_softmax(0).T
        tr = ra.get_trellis(em, labels)
        sha_p.append(np.frombuffer(hashlib.sha256(p.numpy().tobytes()).digest(), np.uint8))
        sha_tr.append(np.frombuffer(hashlib.sha256(tr.contiguous().numpy().tobytes()).digest(), np.uint8))
        tr_shape.append(tr.shape)
        tr_sum.append(float(tr[torch.isfinite(tr)].double().sum()))
        try:
            path = ra.backtrack(tr, em, labels)
        except ValueError:                                      # no path: -1 in the counts
            path_n.append(-1); segs_n.append(-1)
            continue
        segs = ra.merge_repeats(path, list(range(len(tokens))))
        paths += [(q.token_index, q.time_index, q.score) for q in path]
        segs_all += [(s.label, s.start, s.end, s.score) for s in segs]
        path_n.append(len(path)); segs_n.append(len(segs))
    paths, segs_all = np.array(paths, np.float64), np.array(segs_all, np.float64)
    assert np.array_equal(paths[:, 2].astype(np.float32), paths[:, 2])      # path scores are float32 values (`.exp().item()`)
    np.savez_compressed(os.path.join(OUT, 'ref_align.npz'), probs_sha=np.stack(sha_p), trellis_sha=np.stack(sha_tr),
                        trellis_shape=np.asarray(tr_shape, np.int16),
                        trellis_sum=np.asarray(tr_sum, np.float64), path_n=np.asarray(path_n, np.int16), segs_n=np.asarray(segs_n, np.int16),
                        path_ij=paths[:, :2].astype(np.int16), path_score=paths[:, 2].astype(np.float32),
                        seg_lse=segs_all[:, :3].astype(np.int16), seg_score=segs_all[:, 3])


def codec_streams():
    from kraken.lib.codec import PytorchCodec as RefCodec
    rnd = random.Random(5)
    charsets = [{'a': [1], 'b': [2], 'c': [3]},
                {'a': [1], 'ab': [2, 3], 'b': [4], 'cde': [5, 6, 7]},
                {chr(0x710 + i): [i + 1] for i in range(15)}]                 # cfg1's Syriac alphabet shape
    out = []
    for cs in charsets:
        ref = RefCodec(cs)
        case = {'charset': cs, 'len': len(ref), 'max_label': ref.max_label, 'streams': []}
        alphabet = ''.join(cs.keys()) + '?'
        for _ in range(50):
            s = ''.join(rnd.choice(alphabet) for _ in range(rnd.randint(0, 12)))
            labs = [(rnd.randint(1, ref.max_label + 1), 3 * i, 3 * i + rnd.randint(0, 2), rnd.random()) for i in range(rnd.randint(0, 10))]
            case['streams'].append({'text': s, 'encoded': ref.encode(s).tolist(), 'labels': labs,
                                    'decoded': [[y[0], int(y[1]), int(y[2]), float(y[3])] for y in ref.decode(labs)]})
        out.append(case)
    with open(os.path.join(OUT, 'ref_codec.json'), 'w', encoding='utf-8') as fh:
        json.dump(out, fh, ensure_ascii=False, separators=(',', ':'))


def scale_val():
    from kraken.lib.vgsl.rpred import VGSLRecognitionInference as Ref
    obj = Ref.__new__(Ref)
    obj._inf_config = types.SimpleNamespace(padding=16)
    rng = np.random.default_rng(1)
    rows = []
    for _ in range(3000):
        w = int(rng.integers(40, 3000)); olen = int(rng.integers(1, 800)); ow = int(rng.integers(5, 5000))
        obj.net_scale, obj.in_scale = w / olen, ow / (w - 32)
        v = int(rng.integers(0, olen + 1))
        rows.append((w, olen, ow, v, obj._scale_val(v, 0, ow)))
    # net_scale = width / olen and in_scale = max_val / (width - 2 padding), as the tests recompute them
    np.savez_compressed(os.path.join(OUT, 'ref_scale_val.npz'), padding=np.int16(16),
                        **dict(zip(('width', 'olen', 'max_val', 'val', 'scaled'), np.array(rows, np.int16).T)))


def model_files():
    res = os.path.join(refshim.REFERENCE_ROOT, 'tests', 'resources')
    for f in ('overfit.mlmodel', 'model_small.mlmodel', 'model_small.safetensors', 'model_small_fp16.safetensors'):
        shutil.copyfile(os.path.join(res, f), os.path.join(OUT, f))


if __name__ == '__main__':
    oracle_specs()
    align_cases()
    codec_streams()
    scale_val()
    model_files()
    for f in ('ref_oracle_specs.npz', 'ref_align.npz', 'ref_codec.json', 'ref_scale_val.npz'):
        print(f, os.path.getsize(os.path.join(OUT, f)), 'bytes')
