#!/usr/bin/env python
"""The reference's shipped whole-object snapshot, stored small enough to keep: writes tests/golden/snapshot_chaconne_pickle.npz.

    python tests/golden/make_golden_pickle.py <checkout of the original pytorch-wavenet>

The snapshot (snapshots/chaconne_model_2017-12-28_16-44-12, 7.8 MB) is a torch 0.3 legacy-format ``torch.save`` of the
whole WaveNetModel: a header (magic number, protocol, system info, the object pickle, the storage keys) followed by every
storage as an int64 element count and its float32 bytes.  Each storage is either a parameter or an all-zero
DilatedQueue buffer, so the fixture keeps the header, its SHA-256, the element counts and the state_dict key each storage
holds ('' for zeros).  tests/test_host_logic.py reassembles a file from them, filling the parameters from
snapshot_chaconne_state.npz, and unpickles it into this package's classes.

The object pickle embeds the source text of the pickled module classes (WaveNetModel, ModuleList, Conv1d) for torch's
source-change warning.  Those strings are replaced by empty ones: torch.load only compares them and warns.
"""
import hashlib
import io
import os
import pickle
import pickletools
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(os.path.dirname(os.path.dirname(HERE)), "pytorch-wavenet_b200")
SNAPSHOT = os.path.join("snapshots", "chaconne_model_2017-12-28_16-44-12")


def split_legacy(data):
    """(header bytes, [(element count, storage bytes)]) of a legacy-format torch.save file of float32 storages."""
    f = io.BytesIO(data)
    for _ in range(3):                                     # magic number, protocol version, system info
        pickle.load(f)
    for _ in pickletools.genops(f):                        # the object pickle (its classes need not be importable)
        pass
    keys = pickle.load(f)
    pos, storages = f.tell(), []
    head = data[:pos]
    for _ in keys:
        n, = struct.unpack("<q", data[pos:pos + 8])
        storages.append((n, data[pos + 8:pos + 8 + 4 * n]))
        pos += 8 + 4 * n
    assert pos == len(data), "trailing bytes: not a file of float32 storages"
    return head, storages


def blank_class_sources(head):
    """torch 0.3 pickles each nn.Module class, at its first instance, with the persistent id tuple
    ('module', class, source file, source text): MARK, 'module', GLOBAL, file, BINUNICODE text, TUPLE, BINPERSID, where
    the strings other than the text may be memo references (BINGET) and memo BINPUTs are interleaved.  Replace the text
    of each such tuple by an empty string (protocol 2 has no frames or offsets, so the rest of the stream is unaffected)."""
    f = io.BytesIO(head)
    for _ in range(3):
        pickle.load(f)
    start = f.tell()
    memo, ops, prev = {}, [], None
    for op, arg, pos in pickletools.genops(head[start:]):
        if op.name == "BINPUT":
            memo[arg] = prev
            continue
        prev = arg if op.name == "BINUNICODE" else None
        if op.name == "BINGET":                            # a memo reference: (kind, value) of what it refers to
            ops.append(("STR", memo.get(arg), None))
        else:
            ops.append(("STR" if op.name == "BINUNICODE" else op.name, arg, start + pos))
    shape = [{"MARK"}, {"STR"}, {"GLOBAL", "STR"}, {"STR"}, {"STR"}, {"TUPLE"}, {"BINPERSID"}]
    out, last = [], 0
    for i in range(len(ops) - len(shape) + 1):
        win = ops[i:i + len(shape)]
        if all(o[0] in k for o, k in zip(win, shape)) and win[1][1] == "module" and win[4][2] is not None:
            _, text, at = win[4]
            out += [head[last:at], b"X" + struct.pack("<I", 0)]
            last = at + 5 + len(text.encode("utf-8"))
    return b"".join(out + [head[last:]])


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    path = os.path.join(sys.argv[1], SNAPSHOT)
    data = open(path, "rb").read()
    head, storages = split_legacy(data)
    head = blank_class_sources(head)
    sys.path.insert(0, PKG)                                # the pickle's classes resolve to this package's
    import torch
    model = torch.load(path, map_location="cpu", weights_only=False)
    by_bytes = {v.numpy().astype("<f4").tobytes(): k for k, v in model.state_dict().items()}
    sources = []
    for n, raw in storages:
        if raw in by_bytes:
            sources.append(by_bytes[raw])
        else:
            assert raw == bytes(4 * n), "a storage is neither a parameter nor all zeros"
            sources.append("")
    np.savez_compressed(os.path.join(HERE, "snapshot_chaconne_pickle.npz"),
                        head=np.frombuffer(head, dtype=np.uint8), head_sha256=np.array(hashlib.sha256(head).hexdigest()),
                        sources=np.array(sources), counts=np.array([n for n, _ in storages], dtype=np.int64))
    print(f"{len(storages)} storages ({sources.count('')} zero), header {len(head)} bytes")


if __name__ == "__main__":
    main()
