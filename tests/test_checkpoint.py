"""CPU: TensorFlow V2 checkpoint (tensor bundle) reader / writer and the eval result writers.
The file format is restated from its specification (TensorFlow cannot be installed here), so these
tests pin the pieces that have known answers — CRC-32C test vector, LevelDB mask, block / footer
layout byte by byte on a tiny table — and the round trip, including a Snappy-compressed block."""
import os
import struct

import numpy as np
import pytest

from n2nmn_b200 import checkpoint as ck


def test_crc32c_known_answers():
    assert ck.crc32c(b'123456789') == 0xE3069283            # RFC 3720 / iSCSI check value
    assert ck.crc32c(b'\x00' * 32) == 0x8A9136AA             # RFC 3720 B.4 test patterns
    assert ck.crc32c(b'\xff' * 32) == 0x62A8AB43
    assert ck.crc32c(b'6789', ck.crc32c(b'12345')) == 0xE3069283   # incremental
    for v in (0, 1, 0xE3069283, 0xFFFFFFFF):
        assert ck._unmask(ck._mask(v)) == v and ck._mask(v) != v


def test_round_trip_and_layout(tmp_path):
    rng = np.random.RandomState(0)
    tensors = {ck.MODULE_SCOPE + 'FindModule/conv_image/weights': rng.randn(7, 5).astype(np.float32),
               ck.MODULE_SCOPE + 'FindModule/conv_image/biases': rng.randn(5).astype(np.float32),
               'global_step': np.array(50000, np.int64),
               'beta1_power': np.array(0.5, np.float32)}
    for i in range(150):                                     # several data blocks in the index
        tensors['filler/var_%03d/Adam' % i] = rng.randn(3).astype(np.float32)
    prefix = str(tmp_path / 'snap' / '00050000')
    ck.write_checkpoint(prefix, tensors)
    got = ck.read_checkpoint(prefix)
    assert set(got) == set(tensors)
    for k, v in tensors.items():
        assert got[k].dtype == v.dtype and got[k].shape == v.shape
        np.testing.assert_array_equal(got[k], v)
    # file anatomy: 48-byte footer ending in the table magic; data = tensors back to back in key order
    idx = open(prefix + '.index', 'rb').read()
    assert struct.unpack('<Q', idx[-8:])[0] == 0xdb4775248b80fb57
    data = open(prefix + '.data-00000-of-00001', 'rb').read()
    assert len(data) == sum(v.nbytes for v in tensors.values())
    first = sorted(tensors, key=lambda s: s.encode())[0]
    assert data[:tensors[first].nbytes] == tensors[first].tobytes()
    # a flipped data byte is caught by the per-tensor checksum
    bad = bytearray(data)
    bad[5] ^= 1
    open(prefix + '.data-00000-of-00001', 'wb').write(bytes(bad))
    with pytest.raises(ValueError):
        ck.read_checkpoint(prefix)


def test_snappy_blocks_and_prefix_compression():
    raw = b'FindModule/conv_image/weights' * 4 + b'xyz'
    # hand-built snappy stream: literal(29 bytes) + copy(offset 29, len 64) + copy(29, 23) + literal
    lit = b'FindModule/conv_image/weights'
    comp = ck._put_varint(len(raw)) + bytes([(len(lit) - 1) << 2]) + lit
    comp += bytes([((64 - 1) << 2) | 2]) + struct.pack('<H', 29)
    comp += bytes([((23 - 1) << 2) | 2]) + struct.pack('<H', 29)
    comp += bytes([(3 - 1) << 2]) + b'xyz'
    assert ck._snappy_decompress(comp) == raw
    items = [(b'a/b/weights', b'1'), (b'a/b/weights/Adam', b'22'), (b'a/c', b'333')]
    blk = ck._build_block(items, 16)
    assert list(ck._block_entries(blk)) == items
    assert blk[0:3] == bytes([0, 11, 1]) and blk[15:18] == bytes([11, 5, 2])   # shared prefix 11


def snappy_cases():
    """Inputs of the Snappy streams in tests/golden/golden_snappy.npz (make_golden_snappy.py)."""
    rng = np.random.RandomState(0)
    names = [('neural_module_network/layout_execution/module_variables/%s/%s/%s%s' % (m, l, k, a))
             .encode() for m in ('FindModule', 'TransformModule', 'DescribeModule')
             for l in ('conv_image', 'fc_text', 'fc_att') for k in ('weights', 'biases')
             for a in ('', '/Adam', '/Adam_1')]
    return [b'', b'a', b'ab' * 5000, b''.join(names), bytes(rng.randint(0, 256, 70000, dtype=np.uint8)),
            b'\x00' * 100000, b''.join(names) * 40 + bytes(rng.randint(0, 4, 3000, dtype=np.uint8))]


def test_snappy_decoder_against_an_independent_encoder():
    """TensorFlow compresses index blocks with Snappy: the decoder here against streams written by
    the Snappy library itself (through pyarrow's codec, stored in tests/golden/golden_snappy.npz) —
    variable-name-like text with long runs (overlapping copies), > 60-byte literals (multi-byte
    literal lengths), random bytes, empty."""
    z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'golden_snappy.npz'))
    cases = snappy_cases()
    assert len(z.files) == len(cases)
    for i, raw in enumerate(cases):
        assert ck._snappy_decompress(z['case_%d' % i].tobytes()) == raw
    assert len(z['case_2']) < 600                                  # it really compressed


def test_import_export_module_weights(tmp_path):
    from n2nmn_b200 import weights as wts
    W = wts.init_weights('clevr', 10, 15, 512, 28, seed=3, bias_std=0.1)
    prefix = str(tmp_path / 'tfmodel' / '00000010')
    extra = {'neural_module_network/layout_generation/encoder_decoder/embedding_mat':
             np.zeros((4, 3), np.float32),
             ck.MODULE_SCOPE + 'FindModule/conv_image/weights/Adam': np.zeros((512, 250), np.float32)}
    ck.export_module_weights(prefix, W, extra=extra)
    got, ignored = ck.import_module_weights(prefix)
    assert set(got) == set(W) and sorted(ignored) == sorted(extra)
    for k in W:
        np.testing.assert_array_equal(got[k], np.asarray(W[k], np.float32))
    with pytest.raises((KeyError, ValueError)):             # a snapshot of another family
        ck.import_module_weights(prefix, family='vqa', H=14, W=14, D=2048, num_choices=3001)


def test_eval_writers(tmp_path):
    from n2nmn_b200 import evaluate as ev
    res = dict(split='val', num_questions=8, answer_correct=6, layout_correct=8, layout_valid=7,
               answer_accuracy=0.75, layout_accuracy=1.0, layout_validity=0.875)
    f = tmp_path / 'acc.txt'
    ev.write_accuracy_file(str(f), res)
    assert f.read_text() == ('On split: val\n\tanswer accuracy = 0.750000 (6 / 8)\n'
                             '\tlayout accuracy = 1.000000 (8 / 8)\n'
                             '\tlayout validity = 0.875000 (7 / 8)\n')
    p = tmp_path / 'pred.txt'
    ev.write_prediction_file(str(p), ['yes', '2', 'red'])
    assert p.read_text() == 'yes\n2\nred\n'
    j = tmp_path / 'vqa.json'
    ev.write_vqa_prediction_file(str(j), [11, 12], ['cat', 'no'])
    assert j.read_text() == '[{"question_id":\n11,\n"answer":\n"cat"},\n{"question_id":\n12,\n"answer":\n"no"}]'


def test_merge_rank_results_restores_split_order():
    """Data-parallel evaluation: per-rank results (round-robin deal of the split) merge into the
    single-process result, prediction lines back in split order."""
    from n2nmn_b200 import evaluate as ev
    answers = ['a%d' % i for i in range(7)]
    world = 3
    parts = []
    for r in range(world):
        mine = answers[r::world]
        parts.append(dict(split='val', num_questions=len(mine), answer_correct=r + 1,
                          layout_correct=len(mine), layout_valid=len(mine) - (r == 0),
                          answer_accuracy=0.0, layout_accuracy=0.0, layout_validity=0.0,
                          output_answers=mine))
    res = ev.merge_rank_results(parts)
    assert res['output_answers'] == answers and res['num_questions'] == 7
    assert (res['answer_correct'], res['layout_correct'], res['layout_valid']) == (6, 7, 6)
    assert abs(res['answer_accuracy'] - 6 / 7) < 1e-12 and res['split'] == 'val'
    parts[1]['output_answers'] = parts[1]['output_answers'][:-1]
    parts[1]['num_questions'] -= 1
    with pytest.raises(ValueError):          # not a round-robin deal of one split
        ev.merge_rank_results(parts)
