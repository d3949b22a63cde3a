"""Native readers of kraken's on-disk formats (kraken_b200/weights.py; replaces kraken/models/loaders.py:46-254 and
kraken/models/_coreml.py for the engine): synthetic files, and the reference's own model files (copies in tests/golden)."""
import json
import os
import struct

import numpy as np
import pytest

from kraken_b200.weights import load_coreml, load_model_file, load_safetensors

RES = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def write_safetensors(path, tensors, metadata):
    header, blob = {}, b''
    for name, (dtype, arr) in tensors.items():
        raw = arr.tobytes()
        header[name] = {'dtype': dtype, 'shape': list(arr.shape), 'data_offsets': [len(blob), len(blob) + len(raw)]}
        blob += raw
    if metadata is not None:
        header['__metadata__'] = metadata
    hj = json.dumps(header).encode()
    with open(path, 'wb') as fh:
        fh.write(struct.pack('<Q', len(hj)) + hj + blob)


def test_safetensors_roundtrip_prefix_dtypes_and_metadata(tmp_path):
    rng = np.random.default_rng(0)
    w32 = rng.standard_normal((4, 1, 3, 3)).astype(np.float32)
    w16 = rng.standard_normal((7,)).astype(np.float16)
    wbf = rng.standard_normal((5, 2)).astype(np.float32)
    bf_raw = (wbf.view(np.uint32) >> 16).astype(np.uint16)                 # truncated bf16 payload
    meta = {'kraken_meta': json.dumps({
        'abc-uuid': {'_model': 'TorchVGSLModel', '_tasks': ['recognition'], '_kraken_min_version': '7.0', 'vgsl': '[1,8,0,1 Cr3,3,4 O1c3]',
                     'codec': json.dumps({'a': [1], 'b': [2]}), 'hyper_params': json.dumps({'lrate': 0.1}), 'one_channel_mode': '1'},
        'other': {'_model': 'SomethingElse', '_tasks': ['segmentation'], 'vgsl': 'x'}})}
    p = str(tmp_path / 'm.safetensors')
    write_safetensors(p, {'abc-uuid.nn.C_0.co.weight': ('F32', w32), 'abc-uuid.nn.C_0.co.bias': ('F16', w16),
                          'abc-uuid.nn.O_1.lin.weight': ('BF16', bf_raw), 'other.w': ('F32', w32)}, meta)
    files = load_safetensors(p)
    assert len(files) == 1                                               # foreign model classes are skipped
    mf = files[0]
    assert mf.vgsl == '[1,8,0,1 Cr3,3,4 O1c3]' and mf.codec == {'a': [1], 'b': [2]}
    assert mf.metadata['model_type'] == ['recognition'] and mf.metadata['hyper_params'] == {'lrate': 0.1}
    assert set(mf.weights) == {'nn.C_0.co.weight', 'nn.C_0.co.bias', 'nn.O_1.lin.weight'}     # uuid prefix stripped
    assert all(v.dtype == np.float32 for v in mf.weights.values())       # fp16 / bf16 storage widened (test_loaders.py:117-149)
    assert np.array_equal(mf.weights['nn.C_0.co.weight'], w32)
    assert np.array_equal(mf.weights['nn.C_0.co.bias'], w16.astype(np.float32))
    assert np.array_equal(mf.weights['nn.O_1.lin.weight'].view(np.uint32), wbf.view(np.uint32) & 0xFFFF0000)
    assert load_safetensors(p, tasks=['segmentation']) == []             # task filter
    assert load_model_file(p)[0].vgsl == mf.vgsl                         # dispatch on the file type


def test_safetensors_error_paths(tmp_path):
    p = str(tmp_path / 'bad.safetensors')
    with open(p, 'wb') as fh:
        fh.write(b'\x01\x02')
    with pytest.raises(ValueError):
        load_safetensors(p)                                              # truncated header
    write_safetensors(p, {'x': ('F32', np.zeros(1, np.float32))}, None)
    with pytest.raises(ValueError):
        load_safetensors(p)                                              # no metadata (loaders.py: "No model metadata found")
    write_safetensors(p, {'x': ('F32', np.zeros(1, np.float32))}, {'kraken_meta': '{not json'})
    with pytest.raises(ValueError):
        load_safetensors(p)
    write_safetensors(p, {'u.x': ('F32', np.zeros(1, np.float32))}, {'kraken_meta': json.dumps({'u': {'_model': 'TorchVGSLModel', '_tasks': ['recognition']}})})
    with pytest.raises(ValueError):
        load_safetensors(p)                                              # no VGSL spec


def test_reference_fixtures_fp16_and_coreml():
    a = load_safetensors(os.path.join(RES, 'model_small.safetensors'))[0]
    c = load_safetensors(os.path.join(RES, 'model_small_fp16.safetensors'))[0]
    assert a.vgsl == c.vgsl == '[1,48,0,1 Cr{C_0}4,2,1,4,2 O{O_1}1c4]'
    assert {k: v.shape for k, v in a.weights.items()} == {'nn.C_0.co.bias': (1,), 'nn.C_0.co.weight': (1, 1, 4, 2), 'nn.O_1.lin.bias': (4,),
                                                          'nn.O_1.lin.weight': (4, 1)}
    for k in a.weights:
        assert c.weights[k].dtype == np.float32 and np.allclose(a.weights[k], c.weights[k], atol=1e-3)
    o = load_coreml(os.path.join(RES, 'overfit.mlmodel'))[0]             # the cfg1 model: its goldens reproduce the reference's strings
    assert o.vgsl.startswith('[1,30,0,1 Cr{C_0}3,3,32,2,2 Gn{Gn_1}32') and o.metadata['model_type'] == ['recognition']
    assert len(o.weights) == 10 and o.weights['nn.C_0.co.weight'].shape == (32, 1, 3, 3) and o.codec[' '] == [1]
    with pytest.raises(ValueError):                                       # `model_type: null` under kraken_meta: the reference refuses it too
        load_coreml(os.path.join(RES, 'model_small.mlmodel'))             # (kraken/models/loaders.py:195-200)


def test_model_object_from_file_matches_reference_surface():
    import kraken_b200 as kb
    m = kb.TorchVGSLModel.load_model(os.path.join(RES, 'overfit.mlmodel'))
    assert m.input == (1, 1, 30, 0) and m.one_channel_mode == '1' and m.seg_type == 'bbox'
    assert '[' + ' '.join(m.named_spec) + ']' == '[1,30,0,1 Cr{C_0}3,3,32,2,2 Gn{Gn_1}32 Cr{C_2}3,3,64,2,2 Gn{Gn_3}32 S{S_4}1(1x0)1,3 O{O_5}1c16]'   # model.py:198-199
    assert sorted(m.state_dict()) == sorted('nn.' + k for k in ('C_0.co.weight', 'C_0.co.bias', 'Gn_1.layer.weight', 'Gn_1.layer.bias', 'C_2.co.weight',
                                                                'C_2.co.bias', 'Gn_3.layer.weight', 'Gn_3.layer.bias', 'O_5.lin.weight', 'O_5.lin.bias'))
    assert m.codec is not None and m.codec.max_label == 15
