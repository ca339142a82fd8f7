"""BGZF inflate on the device (B200 only: `pytest -m gpu`): msnv_inflate gives the bytes zlib gives for every member of
seeded and hand-made BAM sets and of zlib's own streams, in batches small and large, a malformed member gets its status
without touching the others, and inflaters run from several threads next to a context."""
import json
import os
import subprocess
import sys
import threading
import zlib

import numpy as np
import pytest

from conftest import GOLDEN
from metasnv_b200 import abi
from metasnv_b200.paths import bin_path

sys.path.insert(0, GOLDEN)
import span_set  # noqa: E402

pytestmark = pytest.mark.gpu


def zlib_members(comp, m):
    return b"".join(zlib.decompress(comp[int(x["coff"]):int(x["coff"]) + int(x["clen"])].tobytes(), -15) for x in m)


def check_file(inf, path):
    """Every member of the file through msnv_inflate, in batches of the inflater's size, against zlib."""
    n = 0
    for comp, m in abi.bgzf_batches(*abi.bgzf_members(path), inf.max_batch_bytes):
        out, st = inf.inflate(comp, m)
        assert (st == abi.INFLATE_OK).all(), (path, np.flatnonzero(st != abi.INFLATE_OK)[:5], st[st != 0][:5])
        assert out.tobytes() == zlib_members(comp, m), path
        n += len(m)
    return n


def bams_of(data):
    return [l.strip() for l in open(os.path.join(data, "all_samples")) if l.strip()]


@pytest.mark.parametrize("name,batch", [("c1_tiny", 8 << 20), ("c4_tiny_deep", 8 << 20), ("c5_tiny_annotated", 8 << 20),
                                        ("c4_tiny_deep", 256 << 10), ("c4_tiny_deep", 64 << 20)])
def test_presets_equal_zlib(name, batch, datasets):
    recipe = json.load(open(os.path.join(GOLDEN, name, "recipe.json")))
    data = datasets(recipe["preset"], recipe["scale"], recipe["samples"], **recipe["extra"])
    with abi.Inflater(0, batch) as inf:
        n = sum(check_file(inf, b) for b in bams_of(data))
    assert n > 0


def test_span_set_and_hand_sams_equal_zlib(built, tmp_path):
    data = span_set.write_span_set(str(tmp_path / "span"))
    bams = bams_of(data)
    for s in ("s1", "s2"):
        out = str(tmp_path / (s + ".bam"))
        subprocess.run([bin_path("msnv_synth"), "--sam", os.path.join(GOLDEN, "hand", s + ".sam"), "--bam", out], check=True)
        bams.append(out)
    with abi.Inflater(0, 8 << 20) as inf:
        for b in bams:
            check_file(inf, b)


def zlib_streams():
    rng = np.random.default_rng(7)
    datas = [b"", b"A", rng.integers(0, 256, 65536, dtype=np.uint8).tobytes(), b"\0" * 65536,
             bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), 50000)), bytes(rng.choice(np.frombuffer(b"IIIIFF<7", np.uint8), 65280))]
    out = []
    for d in datas:
        for level in (0, 1, 6, 9):
            for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE):
                c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
                out.append((c.compress(d) + c.flush(), d))
    out.append((b"\x03\x00", b""))                                     # the BGZF EOF member
    return out


def batch(streams):
    comp = b"".join(c for c, _ in streams)
    rows, coff, ooff = [], 0, 0
    for c, d in streams:
        rows.append((coff, len(c), len(d), zlib.crc32(d), 0, ooff))
        coff += len(c)
        ooff += len(d)
    return np.frombuffer(comp, np.uint8), np.array(rows, dtype=abi.MEMBER_DTYPE)


def test_zlib_streams_and_one_malformed_member(built):
    streams = zlib_streams()
    comp, m = batch(streams)
    want = b"".join(d for _, d in streams)
    with abi.Inflater(0, 16 << 20) as inf:
        out, st = inf.inflate(comp, m)
        assert (st == abi.INFLATE_OK).all() and out.tobytes() == want
        # one member of each kind of damage in an otherwise good batch: it gets its status, the others are right
        bad = m.copy()
        k = [i for i, (c, d) in enumerate(streams) if len(d) > 1000 and len(c) > 100]
        bad[k[0]]["crc"] ^= 1
        bad[k[1]]["isize"] -= 1
        bad[k[2]]["clen"] //= 2
        out, st = inf.inflate(comp, bad)
        assert st[k[0]] == abi.INFLATE_BAD_CRC and st[k[1]] == abi.INFLATE_TOO_LONG and st[k[2]] == abi.INFLATE_TRUNCATED
        for i, (c, d) in enumerate(streams):
            if i not in k[:3]:
                assert st[i] == abi.INFLATE_OK and out[int(bad[i]["ooff"]):int(bad[i]["ooff"]) + len(d)].tobytes() == d
        # a member outside the compressed bytes is refused before anything runs
        oob = m.copy()
        oob[0]["coff"] = comp.size
        oob[0]["clen"] = 1
        with pytest.raises(abi.MsnvError):
            inf.inflate(comp, oob)
        assert inf.kernel_ms() >= 0
    # more members than the inflater takes is refused, not grown into
    with abi.Inflater(0, 64 << 10) as small:
        cap = small.lib.msnv_inflater_max_members(64 << 10)
        many = np.array([(0, 2, 0, 0, 0, 0)] * (cap + 1), dtype=abi.MEMBER_DTYPE)
        with pytest.raises(abi.MsnvError):
            small.inflate(np.frombuffer(b"\x03\x00", np.uint8), many)
        out, st = small.inflate(np.frombuffer(b"\x03\x00", np.uint8), many[:cap])
        assert (st == abi.INFLATE_OK).all()


def test_four_inflaters_next_to_a_context(datasets):
    data = datasets("c1", 0.05, 8)
    files = bams_of(data)
    errors = []

    def work(i):
        try:
            with abi.Inflater(0, 8 << 20) as inf:
                for _ in range(3):
                    for b in files[i::4]:
                        check_file(inf, b)
        except Exception as e:          # reported by the main thread
            errors.append(repr(e))
    threads = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    with abi.Context(0) as ctx:
        rng = np.random.default_rng(3)
        for _ in range(20):
            beg = np.sort(rng.integers(0, 90000, 20000)).astype(np.uint32)
            end = (beg + rng.integers(1, 150, beg.size)).astype(np.uint32)
            ctx.cov_run(np.array([100000], np.uint32), np.array([0, beg.size], np.uint64), beg, end, 10)
    for t in threads:
        t.join()
    assert not errors, errors
