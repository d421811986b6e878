"""N1 (SURVEY §8f): Piper ONNX initialiser import.  No real voice exists offline, so the importer is exercised on ONNX
files written here with the same wire format: state-dict names, weight-normalised WaveNet convs, raw / float_data
payloads, fp16 tensors, packed and unpacked dims, and the failure modes it must report."""
import json
import os
import struct
import zlib

import numpy as np
import pytest

from sonata_b200 import onnx_import, voicegen
from sonata_b200.svw import read_svw


def _varint(v: int) -> bytes:
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _ld(fno: int, payload: bytes) -> bytes:
    return _varint((fno << 3) | 2) + _varint(len(payload)) + payload


def _tensor(name: str, arr: np.ndarray, mode: str) -> bytes:
    arr = np.asarray(arr)
    msg = b""
    if mode == "packed_dims":
        msg += _ld(1, b"".join(_varint(int(d)) for d in arr.shape))
    else:
        msg += b"".join(_varint((1 << 3) | 0) + _varint(int(d)) for d in arr.shape)
    if arr.dtype == np.float16:
        msg += _varint((2 << 3) | 0) + _varint(10) + _ld(9, arr.astype("<f2").tobytes())
    elif mode == "float_data":
        msg += _varint((2 << 3) | 0) + _varint(1) + _ld(4, arr.astype("<f4").tobytes())
    else:
        msg += _varint((2 << 3) | 0) + _varint(1) + _ld(9, arr.astype("<f4").tobytes())
    msg += _ld(8, name.encode())
    return msg


def _model(tensors) -> bytes:
    graph = _ld(1, b"torch_jit")                           # GraphProto.name is field 2; a stray field must be skipped
    graph += b"".join(_ld(5, t) for t in tensors)
    return _varint((1 << 3) | 0) + _varint(8) + _ld(2, b"pytorch") + _ld(7, graph)   # ir_version, producer, graph


def _write_voice(tmp_path, quality, decompose=True, drop=None, extra=None, n_speakers=1):
    tensors = voicegen.make_tensors(quality, 77, n_speakers=n_speakers)
    blobs = []
    for i, (name, arr) in enumerate(tensors.items()):
        if (drop and name == drop) or name.startswith("hp."):
            continue
        mode = ("raw", "float_data", "packed_dims")[i % 3]
        if decompose and (".enc.in_layers." in name or ".enc.cond_layer." in name) and name.endswith(".weight"):
            # weight_norm(dim=0): g = ||w|| per output channel, v = any rescaling of w
            w = arr.astype(np.float64)
            g = np.sqrt((w * w).sum(axis=(1, 2), keepdims=True))
            v = w * 3.0
            stem = name[:-len(".weight")]
            if i % 2:
                blobs.append(_tensor(stem + ".weight_g", g.astype(np.float32), mode))
                blobs.append(_tensor(stem + ".weight_v", v.astype(np.float32), mode))
            else:
                blobs.append(_tensor(stem + ".parametrizations.weight.original0", g.astype(np.float32), mode))
                blobs.append(_tensor(stem + ".parametrizations.weight.original1", v.astype(np.float32), mode))
        else:
            blobs.append(_tensor(name, arr, mode))
    for name, arr in (extra or {}).items():
        blobs.append(_tensor(name, arr, "raw"))
    onnx = tmp_path / f"voice-{quality}.onnx"
    onnx.write_bytes(_model(blobs))
    cfg = tmp_path / f"voice-{quality}.onnx.json"
    cfg.write_text(json.dumps(voicegen.make_config(quality, n_speakers=n_speakers)))
    return str(onnx), str(cfg), tensors


@pytest.mark.parametrize("quality", ["medium", "high"])
def test_import_roundtrip(tmp_path, quality):
    onnx, cfg, ref = _write_voice(tmp_path, quality)
    out_cfg = onnx_import.import_voice(onnx, cfg, str(tmp_path / "out"))
    assert os.path.exists(out_cfg) and out_cfg.endswith(".onnx.json")
    got = read_svw(out_cfg[:-len(".onnx.json")] + ".svw")
    assert [k for k in got if not k.startswith("hp.")] == list(voicegen.tensor_specs(voicegen.ARCH[quality]))
    for name, a in ref.items():
        if name.startswith("hp."):
            assert np.array_equal(got[name], a), name
            continue
        tol = 2e-6 if ".enc.in_layers." in name else 0.0       # folded weight norm: fp64 fold of fp32 factors
        assert got[name].dtype == np.float32 and got[name].shape == a.shape
        assert np.abs(got[name] - a).max() <= tol * max(1.0, float(np.abs(a).max())), name
    assert onnx_import.detect_quality(onnx_import.read_initializers(onnx)) == quality


def test_fp16_payload_and_scalar(tmp_path):
    blobs = [_tensor("a.weight", np.arange(6, dtype=np.float16).reshape(2, 3), "raw"),
             _tensor("s", np.float32(2.5), "raw")]
    p = tmp_path / "m.onnx"
    p.write_bytes(_model(blobs))
    t = onnx_import.read_initializers(str(p))
    assert t["a.weight"].dtype == np.float16 and t["a.weight"].tolist() == [[0, 1, 2], [3, 4, 5]]
    assert t["s"].shape == () and float(t["s"]) == 2.5


def test_reports_missing_and_anonymous(tmp_path):
    onnx, cfg, _ = _write_voice(tmp_path, "medium", decompose=False, drop="dec.ups.1.weight",
                                extra={"onnx::ConvTranspose_4711": np.zeros((128, 64, 16), np.float32)})
    with pytest.raises(ValueError) as e:
        onnx_import.import_voice(onnx, cfg, str(tmp_path / "out"))
    assert "dec.ups.1.weight" in str(e.value) and "anonymous" in str(e.value)


def test_multi_speaker_import_and_garbage(tmp_path):
    """multi-speaker voices: `emb_g` + the conditioning convs (the weight-normed `cond_layer` folded like the in_layers)"""
    onnx, cfg, ref = _write_voice(tmp_path, "medium", n_speakers=3)
    out_cfg = onnx_import.import_voice(onnx, cfg, str(tmp_path / "out"))
    got = read_svw(out_cfg[:-len(".onnx.json")] + ".svw")
    spk = voicegen.speaker_specs(voicegen.ARCH["medium"], 3)
    assert all(k in got for k in spk) and got["emb_g.weight"].shape == (3, 512)
    for name in spk:
        tol = 2e-6 if ".cond_layer.weight" in name else 0.0
        assert np.abs(got[name] - ref[name]).max() <= tol * max(1.0, float(np.abs(ref[name]).max())), name
    # an embedding without its conditioning layers is reported, not half-loaded
    onnx2, cfg2, _ = _write_voice(tmp_path, "medium", decompose=False, extra={"emb_g.weight": np.zeros((4, 512), np.float32)})
    with pytest.raises(ValueError, match="dp.cond.weight"):
        onnx_import.import_voice(onnx2, cfg2, str(tmp_path / "out2"))
    bad = tmp_path / "bad.onnx"
    bad.write_bytes(_ld(2, b"not a model"))
    with pytest.raises(ValueError, match="GraphProto"):
        onnx_import.read_initializers(str(bad))


GOLDEN_ONNX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "onnx")
REAL_ONNX = os.path.join(GOLDEN_ONNX, "libtashkeel_sample.onnx")


def test_reader_parses_a_real_exported_onnx_file():
    """Every other test here reads files written by this suite's own writer.  This one reads what a real exporter
    produced: libtashkeel's model (a torch.onnx export, not a Piper voice), shrunk to a sample that keeps the exporter's
    encoding of every initialiser (tests/golden/onnx/make_onnx_golden.py).  The hand-rolled protobuf reader must get the
    initialisers out -- names, dims, dtypes, raw payloads, as the manifest written alongside the sample lists them --
    and account for nearly all of the file's bytes."""
    with open(os.path.join(GOLDEN_ONNX, "libtashkeel_sample.json")) as f:
        manifest = json.load(f)["initializers"]
    t = onnx_import.read_initializers(REAL_ONNX)
    assert list(t) == [e["name"] for e in manifest]
    for e in manifest:
        a = t[e["name"]]
        assert e["data_type"] == 1 and a.dtype == np.float32 and list(a.shape) == e["dims"], e["name"]
        assert zlib.crc32(np.ascontiguousarray(a).astype("<f4").tobytes()) == e["crc32"], e["name"]
    assert len(t) == 127
    assert t["char_emb.weight"].shape == (54, 56) and t["char_emb.weight"].dtype == np.float32
    assert t["attn_layers.0.ccm.batchnorm.running_var"].shape == (112,)
    assert all(np.isfinite(v).all() for v in t.values() if v.dtype.kind == "f")
    assert all(v.size > 0 for v in t.values())
    payload = sum(v.nbytes for v in t.values())
    assert 0.95 * os.path.getsize(REAL_ONNX) < payload < os.path.getsize(REAL_ONNX)
    # spot values: an embedding table of a trained model is O(1), LayerNorm gains sit around 1
    assert 0.5 < float(np.abs(t["char_emb.weight"]).max()) < 10 and 0.2 < float(t["attn_layers.0.attn.layernorm.weight"].mean()) < 2
