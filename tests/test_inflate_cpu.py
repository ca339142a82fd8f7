"""csrc/gpu/inflate_member.h without a device: the DEFLATE member decoder and the CRC pieces that inflate_kernel runs,
compiled for the host under AddressSanitizer and UBSan and compared with zlib (tests/inflate_member_check.cc)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_inflate_member_agrees_with_zlib_under_sanitizers(tmp_path):
    """Every block type from zlib's levels 0/1/6/9 and its Z_FIXED / Z_HUFFMAN_ONLY / Z_RLE strategies, sizes 0..65536,
    matches at distance 1 and 32768, the BGZF EOF member; truncated members, over-subscribed code lengths, a distance
    past the start, wrong isize and wrong CRC each give their status; the 32-piece CRC equals zlib's crc32."""
    exe = str(tmp_path / "inflate_member_check")
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-I", os.path.join(ROOT, "metasnv_b200", "csrc", "gpu"), os.path.join(ROOT, "tests", "inflate_member_check.cc"),
                    "-lz", "-o", exe], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0 and "mismatches: 0" in r.stdout and "runtime error" not in r.stderr, r.stdout + r.stderr[-2000:]


def test_member_parser_matches_the_bgzf_layout(tmp_path):
    """abi.bgzf_members (what the GPU tests feed msnv_inflate) on a file of two members and the EOF member."""
    import zlib
    import numpy as np
    import sys
    sys.path.insert(0, ROOT)
    from metasnv_b200 import abi

    def member(d):
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = c.compress(d) + c.flush()
        hdr = bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 66, 67, 2, 0]) + (len(body) + 25).to_bytes(2, "little")
        return hdr + body + zlib.crc32(d).to_bytes(4, "little") + len(d).to_bytes(4, "little")
    ds = [b"abc" * 1000, bytes(range(256)) * 10, b""]
    comp, m = abi.bgzf_members(b"".join(member(d) for d in ds))
    assert list(m["isize"]) == [len(d) for d in ds] and list(m["ooff"]) == [0, 3000, 5560]
    for x, d in zip(m, ds):
        assert zlib.decompress(comp[int(x["coff"]):int(x["coff"]) + int(x["clen"])].tobytes(), -15) == d
        assert int(x["crc"]) == zlib.crc32(d)
    assert np.dtype(abi.MEMBER_DTYPE).itemsize == 32
