"""Test helpers: per-position A,C,G,T,N counts from two independent sources.

oracle_counts()   parses `samtools mpileup` text (the oracle's or the pinned golden files)
numpy_counts()    recounts one sample from the structure-of-arrays batch of include/msnv.h (position-aligned
                  segments) with numpy: a third statement of the counting rules, independent of both the C oracle
                  and the CUDA kernels. Rules restated: a base counts when (q & 127) >= 13 (mpileup -Q 13 default,
                  SURVEY.md Annex A.4); bit 7 marks a non-ACGT base; before counting, the qualities of positions that
                  both mates of a pair cover are corrected by htslib's tweak_overlap_quality (Annex A.2): equal bases ->
                  the earlier read gets min(qa+qb, 127... htslib: 200) and the later one 0; different bases -> the better one keeps
                  int(0.8*q), the other 0, ties go to the earlier read.
decode_dump()     runs bin/msnv_decode_dump and loads the batches it writes: the decoder's BAM-shaped records expanded
                  on the host into that layout, and with raw=True the records themselves (expand_raw() restates the
                  expansion in Python).
"""
import json
import os
import subprocess

import numpy as np

ARRAYS = (("pos", np.int32), ("seg_off", np.uint32), ("q4_off", np.uint32), ("mate", np.int32),
          ("seg_pos", np.int32), ("seg_len", np.uint16), ("seq2", np.uint8), ("qual", np.uint8))


def oracle_counts(pile_path, n_samples, layout, P):
    """Parse mpileup text into [S][P][5] counts: a column's letters go to their base, '.'/',' to the reference's."""
    off = {name: o for name, o, _ in layout}
    cnt = np.zeros((n_samples, P, 5), np.uint16)
    chan = {"A": 0, "C": 1, "G": 2, "T": 3, "a": 0, "c": 1, "g": 2, "t": 3}
    for line in open(pile_path):
        f = line.rstrip("\n").split("\t")
        p = off[f[0]] + int(f[1]) - 1
        r = f[2].upper()
        rch = chan.get(r, 4)
        for s in range(n_samples):
            b = f[4 + 3 * s]
            i = 0
            while i < len(b):
                ch = b[i]
                if ch == "^":
                    i += 2
                    continue
                if ch in "+-":
                    j = i + 1
                    while b[j].isdigit():
                        j += 1
                    i = j + int(b[i + 1:j])
                    continue
                if ch in ".,":
                    cnt[s, p, rch] += 1
                elif ch in chan:
                    cnt[s, p, chan[ch]] += 1
                elif ch in "Nn":
                    cnt[s, p, 4] += 1
                i += 1
    return cnt


def check_layout(e):
    """Structural invariants of one sample's batch (include/msnv.h)."""
    n = e["pos"].size
    seg_off, q4_off = e["seg_off"].astype(np.int64), e["q4_off"].astype(np.int64)
    assert seg_off.size == n + 1 and q4_off.size == n + 1 and seg_off[0] == 0 and q4_off[0] == 0
    assert np.all(np.diff(seg_off) >= 1) and e["seg_pos"].size == seg_off[-1] == e["seg_len"].size
    assert e["seq2"].size == q4_off[-1] and e["qual"].size == 4 * q4_off[-1]
    assert np.all(np.diff(e["pos"].astype(np.int64)) >= 0), "reads are in coordinate order"
    sp, sl = e["seg_pos"].astype(np.int64), e["seg_len"].astype(np.int64)
    assert np.all(sl >= 1)
    nq = ((sp & 3) + sl + 3) >> 2
    per_read = np.add.reduceat(nq, seg_off[:-1]) if n else np.zeros(0, np.int64)
    assert np.array_equal(per_read, np.diff(q4_off)), "a read owns exactly the quads of its segments"
    # pos is the first reference base the read covers: the first segment's start unless the CIGAR opens with a deletion / skip
    assert np.all(sp[seg_off[:-1]] >= e["pos"].astype(np.int64)), "no segment starts in front of the read"
    span = np.maximum.reduceat(sp + sl, seg_off[:-1]) - e["pos"].astype(np.int64) if n else np.zeros(0, np.int64)
    assert n == 0 or span.max() <= int(e["max_span"])
    m = e["mate"].astype(np.int64)
    has = np.nonzero(m >= 0)[0]
    assert np.array_equal(m[m[has]], has), "mate links are symmetric"
    # padding in front of and behind every segment: quality 0, base bits 0
    q0 = np.concatenate([[0], np.cumsum(nq)[:-1]]) if sp.size else np.zeros(0, np.int64)
    real = np.zeros(e["qual"].size + 1, np.int32)
    np.add.at(real, q0 * 4 + (sp & 3), 1)
    np.add.at(real, q0 * 4 + (sp & 3) + sl, -1)
    real = np.cumsum(real[:-1]) > 0
    assert not e["qual"][~real].any(), "padding bytes carry quality 0"
    codes = (e["seq2"][np.arange(e["qual"].size) >> 2] >> ((np.arange(e["qual"].size) & 3) * 2)) & 3
    assert not codes[~real].any(), "padding positions carry base bits 0"
    assert not codes[real & ((e["qual"] & 0x80) != 0)].any(), "non-ACGT bases carry base bits 0"
    return q0, nq


def numpy_counts(e, P):
    """[P][5] uint16 counts of one sample from its batch `e` (dict of the arrays of msnv_sample_reads)."""
    n = e["pos"].size
    out = np.zeros((P, 5), np.int64)
    if n == 0:
        return out.astype(np.uint16)
    sp, sl = e["seg_pos"].astype(np.int64), e["seg_len"].astype(np.int64)
    seg_off = e["seg_off"].astype(np.int64)
    nq = ((sp & 3) + sl + 3) >> 2
    q0 = np.concatenate([[0], np.cumsum(nq)[:-1]])
    total = int(sl.sum())
    seg_of = np.repeat(np.arange(sp.size, dtype=np.int64), sl)
    off = np.arange(total, dtype=np.int64) - np.repeat(np.cumsum(sl) - sl, sl)
    pos = sp[seg_of] + off
    byte = q0[seg_of] * 4 + (sp[seg_of] & 3) + off
    qual = e["qual"][byte].astype(np.int64)
    code = ((e["seq2"][byte >> 2] >> ((byte & 3) * 2)) & 3).astype(np.int64)
    read = np.repeat(np.arange(n, dtype=np.int64), np.diff(seg_off))[seg_of]
    del seg_of, off, byte

    mate = e["mate"].astype(np.int64)[read]
    idx = np.nonzero(mate >= 0)[0]
    if idx.size:
        pair = np.minimum(read[idx], mate[idx])
        later = (read[idx] > mate[idx]).astype(np.int64)
        order = np.lexsort((later, pos[idx], pair))          # by pair, then position, earlier read first
        k = idx[order]
        same_key = (pair[order][1:] == pair[order][:-1]) & (pos[k][1:] == pos[k][:-1])
        ia, ib = k[:-1][same_key], k[1:][same_key]            # records of the earlier (a) and later (b) read
        va, vb = qual[ia], qual[ib]
        fa, fb, qa, qb = va & 0x80, vb & 0x80, va & 0x7F, vb & 0x7F
        same = np.where(((va | vb) & 0x80) != 0, (va & vb & 0x80) != 0, code[ia] == code[ib])
        a_wins = qa >= qb
        na = np.where(same, fa | np.minimum(qa + qb, 127), np.where(a_wins, fa | (0.8 * qa).astype(np.int64), fa))
        nb = np.where(same, fb, np.where(a_wins, fb, fb | (0.8 * qb).astype(np.int64)))
        qual[ia], qual[ib] = na, nb
    ok = (qual & 0x7F) >= 13
    ch = np.where((qual & 0x80) != 0, 4, code)
    flat = np.bincount((pos * 5 + ch)[ok], minlength=P * 5)
    assert flat.size == P * 5, "a base lies outside the shard"
    return flat.reshape(P, 5).astype(np.uint16)


def first_difference(want, got, layout):
    """Description of where [S][P][5] counts `got` first differ from `want` ('' if equal); layout: [(name, offset, len)]."""
    bad = np.argwhere(want != got)
    if not bad.size:
        return ""
    s, p, c = bad[0]
    ctg = max((o, n) for n, o, _ in layout if o <= p)
    return ("%d differing counts; first: sample %d, %s:%d (shard position %d), channel %s: oracle %d, GPU %d"
            % (len(bad), s, ctg[1], p - ctg[0] + 1, p, "ACGTN"[c], want[s, p, c], got[s, p, c]))


RAW_ARRAYS = (("raw_pos", np.int32), ("raw_mate", np.int32), ("raw_seg_off", np.uint32), ("raw_q4_off", np.uint32),
              ("raw_off", np.uint32), ("raw_n_cigar", np.uint16), ("raw_l_seq", np.uint16), ("raw", np.uint32))


def expand_raw(r):
    """Plain-Python restatement of expand_kernel (csrc/gpu/kernels.cuh): reads as BAM stores them (msnv_raw_reads) -> the
    position-aligned arrays of msnv_sample_reads. Slow on purpose (one base at a time); for small batches only."""
    n = r["raw_pos"].size
    raw8 = r["raw"].view(np.uint8)
    n_seg, n_q4 = int(r["raw_seg_off"][-1]), int(r["raw_q4_off"][-1])
    seg_pos = np.zeros(n_seg, np.int32); seg_len = np.zeros(n_seg, np.uint16)
    seq2 = np.zeros(n_q4, np.uint8); qual = np.zeros(4 * n_q4, np.uint8)
    code = {1: 0, 2: 1, 4: 2, 8: 3}                       # "=ACMGRSVTWYHKDBN": the one-hot codes are A, C, G, T
    for i in range(n):
        b0 = 4 * int(r["raw_off"][i])
        nc, ls = int(r["raw_n_cigar"][i]), int(r["raw_l_seq"][i])
        cig = r["raw"][int(r["raw_off"][i]):int(r["raw_off"][i]) + nc]
        seq4 = raw8[b0 + 4 * nc:b0 + 4 * nc + (ls + 1) // 2]
        ql = raw8[b0 + 4 * nc + (ls + 1) // 2:b0 + 4 * nc + (ls + 1) // 2 + ls]
        rx, qy, k, Q = int(r["raw_pos"][i]), 0, int(r["raw_seg_off"][i]), int(r["raw_q4_off"][i])
        for w in cig:
            op, ln = int(w) & 15, int(w) >> 4
            if op in (0, 7, 8):
                if ln:
                    a = rx & 3
                    seg_pos[k], seg_len[k] = rx, ln
                    for o in range(ln):
                        q = qy + o
                        b4 = (int(seq4[q >> 1]) >> (4 if q % 2 == 0 else 0)) & 15
                        other = b4 not in code
                        at = 4 * Q + a + o
                        qual[at] = min(int(ql[q]), 127) | (0x80 if other else 0)
                        if not other:
                            seq2[at >> 2] |= code[b4] << (2 * (at & 3))
                    k += 1; Q += (a + ln + 3) >> 2
                rx += ln; qy += ln
            elif op in (2, 3):
                rx += ln
            elif op in (1, 4):
                qy += ln
        assert k == int(r["raw_seg_off"][i + 1]) and Q == int(r["raw_q4_off"][i + 1]) and qy <= ls
    return {"pos": r["raw_pos"], "mate": r["raw_mate"], "seg_off": r["raw_seg_off"], "q4_off": r["raw_q4_off"],
            "seg_pos": seg_pos, "seg_len": seg_len, "seq2": seq2, "qual": qual}


def _load_batch(out, prefix, meta, raw):
    e = {k: np.fromfile(os.path.join(out, "%s%s.bin" % (prefix, k)), dt) for k, dt in ARRAYS}
    e["max_span"] = meta["max_span"]
    if raw:
        for k, dt in RAW_ARRAYS:
            e[k] = np.fromfile(os.path.join(out, "%s%s.bin" % (prefix, k)), dt)
    assert e["pos"].size == meta["n_reads"] and e["seg_pos"].size == meta["n_segs"] and e["seq2"].size == meta["n_q4"]
    return e


def decode_dump(ref, lst, out, raw=False, windows=0):
    """Run msnv_decode_dump: (layout.json, [the whole shard's batch per sample]); with windows=N also
    [per window: [its batch per sample]] (the decoder's windows, carried reads included)."""
    from metasnv_b200.paths import bin_path
    os.makedirs(out, exist_ok=True)
    env = dict(os.environ)
    if raw:
        env["MSNV_DUMP_RAW"] = "1"
    if windows:
        env["MSNV_DUMP_WINDOWS"] = str(windows)
    r = subprocess.run([bin_path("msnv_decode_dump"), ref, lst, out], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    lay = json.load(open(os.path.join(out, "layout.json")))
    samples = [_load_batch(out, "s%d." % s, meta, raw) for s, meta in enumerate(lay["samples"])]
    if not windows:
        return lay, samples
    wins = []
    for k, w in enumerate(lay["windows"]):
        batches = []
        for s, meta in enumerate(w["samples"]):
            e = _load_batch(out, "w%d.s%d." % (k, s), meta, raw)
            if raw:
                assert e["raw_pos"].size == meta["raw_n_reads"]
                e["raw_max_span"] = meta["raw_max_span"]
            batches.append(e)
        wins.append(batches)
    return lay, samples, wins
