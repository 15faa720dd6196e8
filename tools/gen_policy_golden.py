#!/usr/bin/env python3
"""Commit what the tests read from the policies the reference ships (rex_gym/policies/<task>/<signal>/) as golden fixtures.

  python tools/gen_policy_golden.py <reference checkout>/rex_gym/policies

1. tests/golden/policies/<task>/<signal>/model.ckpt-N.{index,data-00000-of-00001}: each shipped TensorFlow checkpoint cut
   down to the variables the project restores (policy and value networks, both streaming normalisers, global_step) plus the
   memory variables cut to their first control step.  Tensor bytes are copied unchanged; the index is rewritten in the same
   checkpoint-V2 format (one data block, crc32c on every block and tensor), so the project's reader and TensorFlow's
   both load it.  Adam slots and the bulk of the episode memory are left out: they are what makes the originals 1-6 MB.
2. tests/golden/tf_memory_golden.npz: what TensorFlow recorded in the PPO EpisodeMemory over the first STEPS control steps of
   all 25 episodes (memory/Variable_1..5 = observation, action, action mean, log-stddev, reward):
     <t>_<s>_rows [R]            flat indices (episode * STEPS + step) of a fixed, seeded sample of R rows
     <t>_<s>_observ/_action/_mean [R][.], _reward [R]   float32 as stored, at those rows
     <t>_<s>_logstd [25][STEPS][A]   float32, the whole window (a handful of distinct vectors: it compresses to nothing)
     <t>_<s>_noise  [25][STEPS][A]   action - mean over the whole window, float16 (the sampling-law statistics need every row)
"""
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
from rex_gym_b200.agents import tf_checkpoint as tfc  # noqa: E402
from rex_gym_b200.agents.networks import _TF, _TF_NAMES  # noqa: E402

GOLDEN = os.path.join(HERE, "..", "tests", "golden")
POLICIES = ["walk/ik", "walk/ol", "gallop/ik", "gallop/ol", "turn/ik", "turn/ol", "standup/ol", "poses"]
RECORDED = ["gallop/ik", "gallop/ol", "standup/ol", "turn/ik", "turn/ol", "walk/ik", "walk/ol"]
KEEP = ([_TF + n for _, n in _TF_NAMES] + ["global_step"]
        + ["normalize_%s/Variable%s" % (k, s) for k in ("observ", "reward") for s in ("", "_1", "_2")])
MEMORY = ["memory/Variable", "memory/Variable_1", "memory/Variable_2", "memory/Variable_3", "memory/Variable_4", "memory/Variable_5"]
STEPS, ROWS, SEED = 400, 1200, 0

_CRC_TABLE = []
for _i in range(256):
    _c = _i
    for _ in range(8):
        _c = (_c >> 1) ^ 0x82F63B78 if _c & 1 else _c >> 1
    _CRC_TABLE.append(_c)


def crc32c(data):
    c = 0xFFFFFFFF
    for b in data:
        c = _CRC_TABLE[(c ^ b) & 0xFF] ^ (c >> 8)
    return c ^ 0xFFFFFFFF


def masked_crc(data):
    c = crc32c(data)
    return (((c >> 15) | (c << 17)) + 0xA282EAD8) & 0xFFFFFFFF


def varint(n):
    out = bytearray()
    while True:
        b = n & 0x7F
        n >>= 7
        out.append(b | (0x80 if n else 0))
        if not n:
            return bytes(out)


def _entry_proto(dtype, shape_proto, offset, size, crc):
    """BundleEntryProto {1: dtype, 2: shape, 4: offset, 5: size, 6: crc32c (masked, fixed32)}; shard 0 is the default."""
    out = varint(1 << 3) + varint(dtype) + varint(2 << 3 | 2) + varint(len(shape_proto)) + shape_proto
    if offset:
        out += varint(4 << 3) + varint(offset)
    return out + varint(5 << 3) + varint(size) + varint(6 << 3 | 5) + struct.pack("<I", crc)


def _shape_proto(shape):
    dims = b"".join(varint(2 << 3 | 2) + varint(len(d)) + d for d in (varint(1 << 3) + varint(n) for n in shape))
    return dims


def _table_block(entries):
    """Uncompressed table block, every entry a restart point, followed by its type byte and masked crc32c."""
    body, restarts = bytearray(), []
    for k, v in entries:
        restarts.append(len(body))
        body += varint(0) + varint(len(k)) + varint(len(v)) + k + v
    if not restarts:
        restarts = [0]
    body += b"".join(struct.pack("<I", r) for r in restarts) + struct.pack("<I", len(restarts))
    return bytes(body), bytes(body) + b"\x00" + struct.pack("<I", masked_crc(bytes(body) + b"\x00"))


def write_checkpoint(prefix, header, tensors):
    """tensors: sorted list of (name, dtype enum, shape, raw bytes)."""
    data, entries = bytearray(), [(b"", header)]
    for name, dtype, shape, raw in tensors:
        entries.append((name.encode(), _entry_proto(dtype, _shape_proto(shape), len(data), len(raw), masked_crc(raw))))
        data += raw
    entries.sort(key=lambda e: e[0])
    out = bytearray()
    body, blk = _table_block(entries)
    data_handle = varint(0) + varint(len(body))
    out += blk
    body, blk = _table_block([])
    meta_handle = varint(len(out)) + varint(len(body))
    out += blk
    body, blk = _table_block([(entries[-1][0], data_handle)])
    index_handle = varint(len(out)) + varint(len(body))
    out += blk
    footer = meta_handle + index_handle
    out += footer + b"\x00" * (40 - len(footer)) + struct.pack("<Q", tfc._MAGIC)
    with open(prefix + ".index", "wb") as f:
        f.write(out)
    with open(prefix + ".data-00000-of-00001", "wb") as f:
        f.write(data)


def _header(prefix):
    """The BundleHeaderProto: value of key "", the first entry of the first data block."""
    data = open(prefix + ".index", "rb").read()
    pos = 0
    for _ in range(2):                                     # skip the metaindex handle
        _, pos = tfc._varint(data[-48:], pos)
    ioff, pos = tfc._varint(data[-48:], pos)
    isize, pos = tfc._varint(data[-48:], pos)
    handle = tfc._block(data, ioff, isize)[0][1]
    boff, p = tfc._varint(handle, 0)
    bsize, _ = tfc._varint(handle, p)
    key, value = tfc._block(data, boff, bsize)[0]
    assert key == b"", prefix
    return bytes(value)


def pruned_checkpoint(ref, rel):
    src = tfc.latest_checkpoint(os.path.join(ref, rel))
    ents = tfc.list_variables(src)
    raw = np.memmap(src + ".data-00000-of-00001", dtype=np.uint8, mode="r")
    tensors = []
    for name in sorted(KEEP + MEMORY):
        dtype, shape, _, offset, size = ents[name]
        b = bytes(raw[offset:offset + size])
        if name in MEMORY and len(shape) >= 2:             # [episodes][capacity][...] -> first control step only
            a = np.frombuffer(b, tfc._DTYPES[dtype]).reshape(shape)[:, :1]
            shape, b = a.shape, a.tobytes()
        tensors.append((name, dtype, shape, b))
    os.makedirs(os.path.join(GOLDEN, "policies", rel), exist_ok=True)
    dst = os.path.join(GOLDEN, "policies", rel, os.path.basename(src))
    write_checkpoint(dst, _header(src), tensors)
    back = tfc.load_variables(dst)
    orig = tfc.load_variables(src, KEEP)
    assert all(np.array_equal(back[k], orig[k]) for k in KEEP), rel
    print(dst, os.path.getsize(dst + ".data-00000-of-00001") + os.path.getsize(dst + ".index"), "bytes")


def recorded_memory(ref):
    out = {}
    for rel in RECORDED:
        v = tfc.load_variables(tfc.latest_checkpoint(os.path.join(ref, rel)), MEMORY[1:])
        ob, ac, mean, logstd = (v["memory/Variable_%d" % k][:, :STEPS] for k in (1, 2, 3, 4))
        rw = v["memory/Variable_5"][:, :STEPS]
        name = rel.replace("/", "_")
        rows = np.sort(np.random.default_rng(SEED).choice(ob.shape[0] * STEPS, ROWS, replace=False)).astype(np.int32)
        out[name + "_rows"] = rows
        out[name + "_observ"] = ob.reshape(-1, ob.shape[-1])[rows]
        out[name + "_action"] = ac.reshape(-1, ac.shape[-1])[rows]
        out[name + "_mean"] = mean.reshape(-1, mean.shape[-1])[rows]
        out[name + "_reward"] = rw.reshape(-1)[rows]
        out[name + "_logstd"] = logstd
        out[name + "_noise"] = (ac - mean).astype(np.float16)
    path = os.path.join(GOLDEN, "tf_memory_golden.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    for rel in POLICIES:
        pruned_checkpoint(sys.argv[1], rel)
    recorded_memory(sys.argv[1])
