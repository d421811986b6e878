"""Writes tests/golden/onnx/libtashkeel_sample.onnx and its manifest from libtashkeel's exported model
(`crates/core/data/ort/model.onnx` of libtashkeel, MIT licence; a torch.onnx export, 4.8 MB):

    python tests/golden/onnx/make_onnx_golden.py <path to libtashkeel's model.onnx>

The sample keeps the exporter's bytes except where it has to shrink them: every model field and every graph field
other than the nodes is copied as is, one node in NODE_STRIDE is kept, and every initialiser keeps its name, data
type, field order and encoding; an initialiser whose payload exceeds CAP bytes keeps only the leading entries of its
largest axis (its dims are rewritten to match), except the character embedding table, which the test checks whole.
The manifest lists name, dims, data type and the CRC-32 of the raw payload of every initialiser, worked out here with
a protobuf walker of its own, not with sonata_b200.onnx_import."""
import json
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CAP = 3072              # bytes of payload an initialiser may keep
KEEP_WHOLE = {"char_emb.weight"}
NODE_STRIDE = 30


def varint(b, i):
    v = s = 0
    while True:
        c = b[i]
        i += 1
        v |= (c & 0x7F) << s
        if not c & 0x80:
            return v, i
        s += 7


def enc_varint(v):
    out = bytearray()
    while True:
        c = v & 0x7F
        v >>= 7
        out.append(c | (0x80 if v else 0))
        if not v:
            return bytes(out)


def fields(b):
    """(field number, wire type, value, the field's bytes as written)"""
    i = 0
    while i < len(b):
        s = i
        key, i = varint(b, i)
        wt = key & 7
        if wt == 0:
            v, i = varint(b, i)
        elif wt == 2:
            n, i = varint(b, i)
            v = b[i:i + n]
            i += n
        elif wt in (1, 5):
            n = 8 if wt == 1 else 4
            v = b[i:i + n]
            i += n
        else:
            raise ValueError(wt)
        yield key >> 3, wt, v, b[s:i]


def ld(fno, payload):
    return enc_varint(fno << 3 | 2) + enc_varint(len(payload)) + payload


def shrink_tensor(b):
    """TensorProto -> (bytes written, manifest entry).  Expects what torch.onnx writes: unpacked dims, float32 raw_data."""
    fs = list(fields(b))
    dims = [v for f, wt, v, _ in fs if f == 1]
    assert all(wt == 0 for f, wt, _, _ in fs if f == 1), "packed dims"
    dtype = next(v for f, _, v, _ in fs if f == 2)
    name = next(v for f, _, v, _ in fs if f == 8).decode()
    raw = next(v for f, _, v, _ in fs if f == 9)
    assert dtype == 1, (name, dtype)
    a = np.frombuffer(raw, dtype="<f4").reshape(dims)
    if a.nbytes > CAP and name not in KEEP_WHOLE:
        ax = int(np.argmax(a.shape))
        keep = max(1, CAP // (a.nbytes // a.shape[ax]))
        a = np.ascontiguousarray(np.take(a, np.arange(keep), axis=ax))
    out, dims_done = b"", False
    for f, wt, v, whole in fs:
        if f == 1:
            if not dims_done:
                out += b"".join(enc_varint(1 << 3) + enc_varint(d) for d in a.shape)
                dims_done = True
        elif f == 9:
            out += ld(9, a.tobytes())
        else:
            out += whole
    return out, {"name": name, "dims": list(a.shape), "data_type": dtype, "crc32": zlib.crc32(a.tobytes())}


def main(src):
    model = open(src, "rb").read()
    manifest, out = [], b""
    for f, wt, v, whole in fields(model):
        if f != 7:
            out += whole
            continue
        graph, node = b"", 0
        for gf, gwt, gv, gwhole in fields(v):
            if gf == 1:
                if node % NODE_STRIDE == 0:
                    graph += gwhole
                node += 1
            elif gf == 5:
                t, entry = shrink_tensor(gv)
                graph += ld(5, t)
                manifest.append(entry)
            else:
                graph += gwhole
        out += ld(7, graph)
    dst = os.path.join(HERE, "libtashkeel_sample.onnx")
    with open(dst, "wb") as fh:
        fh.write(out)
    with open(os.path.join(HERE, "libtashkeel_sample.json"), "w") as fh:
        fh.write('{"source_bytes": %d, "initializers": [\n' % len(model))
        fh.write(",\n".join(json.dumps(e) for e in manifest))
        fh.write("\n]}\n")
    payload = sum(4 * int(np.prod(e["dims"])) for e in manifest)
    print(dst, len(out), "bytes,", len(manifest), "initialisers,", payload, "payload bytes")


if __name__ == "__main__":
    main(sys.argv[1])
