"""The pure-Python HDF5 reader and the converted weight artefact (SURVEY.md section 8a / 8c)."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLD, SNAP


def test_npz_inventory():
    z = np.load(SNAP)
    names = [k for k in z.files if not k.startswith("__")]
    assert len(names) == 315
    assert sum(z[k].size for k in names) == 4_372_376
    assert all(z[k].dtype == np.float32 for k in names)
    layer_names = [str(s) for s in z["__layer_names__"]]
    assert len(layer_names) == 250
    assert layer_names[0] == "input_1" and layer_names[-3:] == ["yaw_new", "pitch_new", "roll_new"]
    assert str(z["__keras_version__"]) == "2.1.6" and str(z["__backend__"]) == "tensorflow"
    for prefix, count in (("conv2d_", 65), ("depthwise_conv2d_", 16), ("batch_normalization_", 49), ("swish_", 49),
                          ("lambda_", 16), ("activation_", 16), ("multiply_", 16), ("add_", 9), ("drop_connect_", 9)):
        assert sum(1 for n in layer_names if n.startswith(prefix) and n[len(prefix):].isdigit()) == count, prefix


def test_assign_weights_shapes():
    from whenet_b200 import arch, weights
    _names, w = weights.load_snapshot(SNAP)
    stem, blks, head = arch.assign_weights(w)
    assert len(blks) == 16
    assert [(b.hin, b.hout, b.cin, b.cexp, b.cout, b.k, b.s, b.cse, b.skip) for b in blks][:4] == [
        (112, 112, 32, 32, 16, 3, 1, 8, False), (112, 56, 16, 96, 24, 3, 2, 4, False),
        (56, 56, 24, 144, 24, 3, 1, 6, True), (56, 28, 24, 144, 40, 5, 2, 6, False)]
    assert blks[1].w == {"expand": "conv2d_5", "expand_bn": "batch_normalization_4", "dw": "depthwise_conv2d_2",
                         "dw_bn": "batch_normalization_5", "se_reduce": "conv2d_6", "se_expand": "conv2d_7",
                         "project": "conv2d_8", "project_bn": "batch_normalization_6"}
    assert head == {"conv": "conv2d_65", "bn": "batch_normalization_49"}
    assert sum(b.skip for b in blks) == 9


def test_macs_match_survey():
    from whenet_b200 import arch
    m = arch.macs_per_crop()
    assert m["total"] == 389_533_088
    assert m["stem"] == 10_838_016


def test_same_padding_rule():
    from whenet_b200 import arch
    assert arch.same_pad(224, 3, 2) == (112, 0, 1)
    assert arch.same_pad(112, 3, 2) == (56, 0, 1)
    assert arch.same_pad(56, 5, 2) == (28, 1, 2)
    assert arch.same_pad(14, 5, 1) == (14, 2, 2)
    assert [b.pad_before for b in arch.blocks()][:6] == [1, 0, 1, 1, 2, 0]


def test_bad_weights_rejected():
    from whenet_b200 import arch, weights
    _n, w = weights.load_snapshot(SNAP)
    w = dict(w)
    w["conv2d_5/kernel:0"] = w["conv2d_5/kernel:0"][:, :, :, :90]
    with pytest.raises(ValueError):
        arch.assign_weights(w)
    with pytest.raises(OSError):
        weights.load_snapshot("/nonexistent.h5")


def test_random_weights_cover_everything():
    from whenet_b200 import arch
    w = arch.random_weights(0)
    arch.assign_weights(w)
    assert len(w) == 315


def test_h5_reader_matches_npz_bit_for_bit(tmp_path):
    """The reader walks the original WHENet.h5 structure (stored with most tensor data zeroed, tools/make_h5_fixture.py);
    the values it keeps and the SHA-256 of every full tensor of the original file match the converted npz bit for bit."""
    from whenet_b200 import h5lite
    with open(os.path.join(GOLD, "whenet_h5_digests.json")) as f:
        gold = json.load(f)
    path = tmp_path / "WHENet.h5"
    with gzip.open(os.path.join(GOLD, "whenet_h5_skeleton.h5.gz")) as f:
        path.write_bytes(f.read())
    names, w, meta = h5lite.read_keras_weights(str(path))
    z = np.load(SNAP)
    assert names == [str(s) for s in z["__layer_names__"]] == gold["layer_names"]
    assert meta == gold["meta"] == {"backend": "tensorflow", "keras_version": "2.1.6"}
    assert len(w) == 315 and sorted(w) == sorted(gold["sha256"])
    keep = gold["keep"]
    for k, v in w.items():
        ref = z[k]
        assert v.dtype == np.float32 and v.shape == ref.shape, k
        a, b = v.reshape(-1), ref.reshape(-1)
        assert np.array_equal(a[:keep].view(np.uint32), b[:keep].view(np.uint32)), k
        assert np.array_equal(a[-keep:].view(np.uint32), b[-keep:].view(np.uint32)), k
        assert hashlib.sha256(np.ascontiguousarray(ref, dtype="<f4").tobytes()).hexdigest() == gold["sha256"][k], k


def test_h5_reader_rejects_garbage(tmp_path):
    from whenet_b200 import h5lite
    p = tmp_path / "x.h5"
    p.write_bytes(b"not an hdf5 file at all")
    with pytest.raises(h5lite.H5FormatError):
        h5lite.H5File(str(p))


def test_safetensors_artefact_round_trip(tmp_path):
    """The persisted artefact (SURVEY.md 8f rank 2): same tensors bit for bit, layer order kept, loadable as a snapshot."""
    from whenet_b200 import stlite, weights
    names, w = weights.load_snapshot(SNAP)
    path = os.path.join(tmp_path, "whenet.safetensors")
    weights.save_safetensors(path, names, w)
    names2, w2 = weights.load_snapshot(path)
    assert names2 == names and sorted(w2) == sorted(w)
    for k in w:
        assert w2[k].dtype == np.float32 and w2[k].shape == w[k].shape and np.array_equal(w2[k].view(np.uint32), w[k].view(np.uint32)), k
    raw, meta = stlite.load(path)
    assert meta["format"] == "whenet-keras-raw-f32" and len(raw) == 315
    # container checks: truncated data, bad header length, non-JSON header
    blob = open(path, "rb").read()
    bad = os.path.join(tmp_path, "bad.safetensors")
    for mutated in (blob[:len(blob) - 4096], b"\xff" * 8 + blob[8:], blob[:8] + b"{" * 64 + blob[72:]):
        with open(bad, "wb") as f:
            f.write(mutated)
        with pytest.raises(ValueError):
            stlite.load(bad)
    with pytest.raises(ValueError):
        stlite.save(bad, {"x": np.zeros(3, dtype=np.complex64)})
