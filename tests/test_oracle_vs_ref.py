"""Checks the restatement (oracle/cimbar_oracle.c) against the reference's own OpenCV-free code compiled
unmodified into oracle/_ref/libcimbar_ref.so (oracle/Makefile `ref`, oracle/ref_shim.cpp):
libcorrect RS incl. its failure/miscorrection behaviour, the flood walk on the real std::priority_queue,
cell geometry, interleave, the RS->aligned_stream->escrow stack, FountainMetadata, wirehair.

Each check runs one fixed input sequence through a "side" -- OracleSide here, RefSide (tests/golden/make_ref_goldens.py)
for the reference -- and compares the digest of what came out with the reference's, stored in tests/golden/ref_outputs.json."""
import ctypes as C

import numpy as np
import pytest

from oracle_lib import Oracle, _ptr, digest, ref_outputs

ORA = Oracle()

MODES = [68, 4, 8, 67, 66]
INTERLEAVE_ARGS = [(12400, 155, 2), (12400, 155, 1), (12400, 0, 2), (8592, 179, 2), (5376, 168, 2)]
WALK_MODES, WALK_NOISE = [68, 67, 66], [0, 3, 30, 100]
RS_CODES = [(30, 155), (33, 168), (36, 179), (40, 216), (15, 155)]
STREAM_MODES = [68, 4, 67, 66]


class OracleSide:
    """the restatement, behind the calls the reference side makes"""

    def cell_positions(self, m, xs, ys):
        return ORA.lib.cbo_cell_positions(C.byref(m), 0, _ptr(xs, C.c_int), _ptr(ys, C.c_int))

    def adjacent(self, m, xs, idx, out):
        ORA.lib.cbo_adjacent(C.byref(m), _ptr(xs, C.c_int), m.total_cells, idx, _ptr(out, C.c_int))

    def interleave_reverse(self, args, out):
        ORA.lib.cbo_interleave_reverse(*args, _ptr(out, C.c_uint))

    def flood_walk(self, m, seed, noise, o, d, c):
        return ORA.lib.cbo_flood_walk_synthetic(C.byref(m), seed, noise, _ptr(o, C.c_uint16), _ptr(d, C.c_int8), _ptr(c))

    def fuzzy_ahash(self, bits, w, wx, wy, all_, out):
        ORA.lib.cbo_fuzzy_ahash(_ptr(bits), w, wx, wy, all_, out)

    def rs_create(self, parity):
        return ORA.lib.cbo_rs_create(parity)

    def rs_destroy(self, h):
        ORA.lib.cbo_rs_destroy(h)

    def rs_encode(self, h, msg, out):
        return ORA.lib.cbo_rs_encode(h, _ptr(msg), msg.size, _ptr(out))

    def rs_decoder(self, encoder, parity):
        return encoder          # the restatement decodes with the object that encoded the blocks

    def rs_decode(self, h, blk, out):
        return ORA.lib.cbo_rs_decode(h, _ptr(blk), blk.size, _ptr(out))

    def rs_stream(self, parity, block, raw, sym_len):
        """Decoder::decode: the corrected bytes of the symbol stream"""
        return ORA.rs_stream(parity, block, raw[:sym_len])[0]

    def rs_align(self, m, raw, sym_len, col_len):
        """Decoder::decode_fountain: (bytes written, chunks written, the chunks) -- rs_stream + align_chunks"""
        parity, block = m.ecc_bytes, m.ecc_block_size
        msg, nblocks = block - parity, ORA.capacity(m) // block
        data = np.zeros(nblocks * msg, np.uint8)
        okall = np.zeros(nblocks, np.uint8)
        o1, k1 = ORA.rs_stream(parity, block, raw[:sym_len])
        data[:o1.size], okall[:k1.size] = o1, k1
        if col_len:
            o2, k2 = ORA.rs_stream(parity, block, raw[sym_len:])
            data[o1.size:], okall[k1.size:] = o2, k2
        chunks = np.zeros((m.chunks_per_frame, m.chunk_size), np.uint8)
        mask = C.c_uint32(0)
        good = ORA.lib.cbo_align_chunks(_ptr(data), _ptr(okall), nblocks, msg, m.chunk_size, _ptr(chunks), C.byref(mask))
        used = bin(mask.value).count("1")
        assert good == used * m.chunk_size
        return good, used, chunks

    def md_pack(self, eid, size, bid, out):
        ORA.lib.cbo_md_pack(eid, size, bid, _ptr(out))

    def md_fields(self, a):
        return ORA.lib.cbo_md_file_size(_ptr(a)), ORA.lib.cbo_md_block_id(_ptr(a)), ORA.lib.cbo_md_encode_id(_ptr(a))


def cell_positions_and_adjacency(side, mode):
    m = ORA.mode(mode)
    n = m.total_cells
    xs, ys = np.zeros(n, np.int32), np.zeros(n, np.int32)
    assert side.cell_positions(m, xs, ys) == n
    out = [xs, ys]
    rng = np.random.default_rng(1)
    for idx in list(rng.integers(0, n, 300)) + [0, n - 1, 99, 100, 599, 600, 711, 712, n - 600, n - 601]:
        a = np.zeros(4, np.int32)
        side.adjacent(m, xs, int(idx), a)
        out.append(a)
    return out


def interleave_reverse(side, args):
    a = np.zeros(args[0], np.uint32)
    side.interleave_reverse(args, a)
    return a


def flood_walks(side, mode, noise):
    m = ORA.mode(mode)
    n = m.total_cells
    out = []
    for seed in range(4):
        o, d, c = np.zeros(n, np.uint16), np.zeros(2 * n, np.int8), np.zeros(n, np.uint8)
        assert side.flood_walk(m, seed, noise, o, d, c) == n
        out += [o, d, c]
    return out


def fuzzy_ahashes(side):
    rng = np.random.default_rng(7)
    w, h = 64, 40
    bits = rng.integers(0, 256, w * h // 8, dtype=np.uint8)
    out = []
    for _ in range(200):
        wx, wy, all_ = int(rng.integers(0, w - 10)), int(rng.integers(0, h - 10)), int(rng.integers(0, 2))
        r = (C.c_uint64 * 9)()
        side.fuzzy_ahash(bits, w, wx, wy, all_, r)
        out.append(list(r))
    return out


def rs_known_answer(side):
    # reed_solomon_streamTest.cpp:23: RS(155,140) parity of the ASCII digits message
    msg = np.frombuffer((b"0123456789" * 14), dtype=np.uint8).copy()
    h = side.rs_create(15)
    enc = np.zeros(255, np.uint8)
    assert side.rs_encode(h, msg, enc) == 255
    side.rs_destroy(h)
    return enc[:155]


def rs_decode_trials(side, parity, block):
    """1500 blocks with 0 .. parity + 8 symbol errors (and some pure noise), encoded by the restatement, decoded by `side` with
    one persistent decoder object (libcorrect keeps state across calls): [(trial, errors, message, returned, decoded)]"""
    rng = np.random.default_rng(parity * 1000 + block)
    o = ORA.lib.cbo_rs_create(parity)
    h = side.rs_decoder(o, parity)
    msg_len = block - parity
    trials = []
    for trial in range(1500):
        msg = rng.integers(0, 256, msg_len, dtype=np.uint8)
        enc = np.zeros(255, np.uint8)
        ORA.lib.cbo_rs_encode(o, _ptr(msg), msg_len, _ptr(enc))
        blk = enc[:block].copy()
        kind = trial % 6
        t = parity // 2
        nerr = [0, 1, t, t + 1, int(rng.integers(1, parity + 8)), int(rng.integers(t - 2, t + 3))][kind]
        nerr = max(0, min(nerr, block))
        pos = rng.choice(block, nerr, replace=False)
        blk[pos] ^= rng.integers(1, 256, nerr, dtype=np.uint8)
        if trial % 97 == 0:
            blk = rng.integers(0, 256, block, dtype=np.uint8)  # pure noise
        a = np.zeros(256, np.uint8)
        n = side.rs_decode(h, blk, a)
        trials.append((trial, nerr, msg, n, a[:msg_len].copy()))
    if h != o:
        side.rs_destroy(h)
    ORA.lib.cbo_rs_destroy(o)
    return trials


def rs_decode_outputs(trials):
    """what the comparison covers: the return value of every decode, and the message wherever one came back"""
    return [np.array([n for _, _, _, n, _ in trials], np.int64)] + [a for _, _, _, n, a in trials if n > 0]


def rs_stream_and_aligned_chunks(side, mode):
    m = ORA.mode(mode)
    rng = np.random.default_rng(mode)
    cap = ORA.capacity(m)
    block, parity = m.ecc_block_size, m.ecc_bytes
    msg = block - parity
    nblocks = cap // block
    if m.legacy_mode:
        sym_len, col_len = cap, 0
    else:
        sym_len, col_len = ORA.capacity(m, m.symbol_bits), ORA.capacity(m, m.color_bits)
    rs = ORA.lib.cbo_rs_create(parity)
    out = []
    for trial in range(40):
        payload = rng.integers(0, 256, nblocks * msg, dtype=np.uint8)
        raw = np.zeros(cap, np.uint8)
        enc = np.zeros(255, np.uint8)
        for b in range(nblocks):
            ORA.lib.cbo_rs_encode(rs, _ptr(payload[b * msg:(b + 1) * msg].copy()), msg, _ptr(enc))
            raw[b * block:(b + 1) * block] = enc[:block]
        # break some blocks beyond repair; always include the last block of a chunk / of the symbol stream
        bad = set(rng.choice(nblocks, int(rng.integers(0, 6)), replace=False).tolist())
        per_chunk = m.chunk_size // msg
        if trial % 4 == 1:
            bad.add(per_chunk - 1)
        if trial % 4 == 2 and not m.legacy_mode:
            bad.add(sym_len // block - 1)
        if trial % 4 == 3:
            bad.add(nblocks - 1)
        for b in bad:
            raw[b * block:b * block + parity] = rng.integers(0, 256, parity, dtype=np.uint8)
        # (a) Decoder::decode semantics; (b) Decoder::decode_fountain semantics
        stream = side.rs_stream(parity, block, raw, sym_len)
        good, used, chunks = side.rs_align(m, raw, sym_len, col_len)
        out += [stream.size, stream, good, used, chunks]
    ORA.lib.cbo_rs_destroy(rs)
    return out


def fountain_metadata(side):
    rng = np.random.default_rng(3)
    out = []
    for _ in range(200):
        eid, size, bid = int(rng.integers(0, 256)), int(rng.integers(0, 1 << 25)), int(rng.integers(0, 65536))
        a = np.zeros(6, np.uint8)
        side.md_pack(eid, size, bid, a)
        fields = side.md_fields(a)
        assert fields == (size, bid, eid & 0x7F)
        out += [a, fields]
    return out


@pytest.mark.parametrize("mode", MODES)
def test_cell_positions_and_adjacency(mode):
    out = cell_positions_and_adjacency(OracleSide(), mode)
    if mode == 68:  # CellPositionsTest.cpp:11-27
        assert (out[0][0], out[1][0]) == (62, 8) and out[0].size == 12400
    assert digest(*out) == ref_outputs()["cell_positions_and_adjacency"][str(mode)]


@pytest.mark.parametrize("args", INTERLEAVE_ARGS)
def test_interleave_reverse(args):
    a = interleave_reverse(OracleSide(), args)
    if args == (12400, 155, 1):  # InterleaveTest.cpp:14-58
        assert a[1] == 80
    assert digest(a) == ref_outputs()["interleave_reverse"][repr(args)]


@pytest.mark.parametrize("mode", WALK_MODES)
@pytest.mark.parametrize("noise", WALK_NOISE)
def test_flood_walk_matches_std_priority_queue(mode, noise):
    out = flood_walks(OracleSide(), mode, noise)
    n = ORA.mode(mode).total_cells
    for o in out[0::3]:
        assert sorted(o.tolist()) == list(range(n))
    if mode == 68 and noise == 0:  # FloodDecodePositionsTest.cpp:11-129 seeds; SURVEY appendix A.6 clean walk order
        assert out[0][:4].tolist() == [0, 12399, 99, 12300]
    assert digest(*out) == ref_outputs()["flood_walk"]["%d/%d" % (mode, noise)]


def test_fuzzy_ahash_vs_reference_extractors():
    assert digest(fuzzy_ahashes(OracleSide())) == ref_outputs()["fuzzy_ahash"]


def test_rs_known_answer():
    enc = rs_known_answer(OracleSide())
    assert enc[140:155].tobytes().hex() == "a4740203 72c3adf2 60c5b69e 267873".replace(" ", "")
    assert digest(enc) == ref_outputs()["rs_known_answer"]


@pytest.mark.parametrize("parity,block", RS_CODES)
def test_rs_decode_matches_libcorrect_including_failures(parity, block):
    trials = rs_decode_trials(OracleSide(), parity, block)
    n_fail = 0
    for trial, nerr, msg, n, a in trials:
        if n > 0:
            if nerr <= parity // 2:
                assert np.array_equal(a, msg), (trial, nerr)
        else:
            n_fail += 1
    assert n_fail > 0  # the sweep really exercised libcorrect's failure path
    assert digest(*rs_decode_outputs(trials)) == ref_outputs()["rs_decode"]["%d/%d" % (parity, block)]


@pytest.mark.parametrize("mode", STREAM_MODES)
def test_rs_stream_and_aligned_chunks_match_reference_stack(mode):
    assert digest(*rs_stream_and_aligned_chunks(OracleSide(), mode)) == ref_outputs()["rs_stream_and_aligned_chunks"][str(mode)]


def test_fountain_metadata():
    assert digest(*fountain_metadata(OracleSide())) == ref_outputs()["fountain_metadata"]


def test_sample_stream_reassembles_with_reference_wirehair():
    # samples/b/tr_0..3.png are a complete 4-frame fountain stream (.github/workflows/wasm.yml:48-49):
    # oracle decode_fountain -> chunk headers -> the reference's wirehair -> recovered (zstd) file
    from oracle_lib import Ref, load_sample
    try:
        REF = Ref()
    except (FileNotFoundError, OSError) as e:  # pragma: no cover
        pytest.skip(f"oracle/_ref not available: {e}")
    m = ORA.mode(68)
    codec, size = None, None
    seen = set()
    done = False
    for k in range(4):
        good, chunks, mask = ORA.decode_fountain(m, load_sample(f"b/tr_{k}.png"))
        assert good == 7500 and mask == 0xFFF
        for ch in chunks:
            fsize = ORA.lib.cbo_md_file_size(_ptr(ch))
            bid = ORA.lib.cbo_md_block_id(_ptr(ch))
            assert ORA.lib.cbo_md_encode_id(_ptr(ch)) == 0
            if codec is None:
                size = fsize
                codec = REF.lib.wirehair_decoder_create(None, size, m.chunk_size - 6)
            assert fsize == size == 23586
            if bid in seen or done:
                continue
            seen.add(bid)
            payload = ch[6:].copy()
            res = REF.lib.wirehair_decode(codec, bid, _ptr(payload, C.c_uint8), payload.size)
            done = res == 0
    assert done
    out = np.zeros(size, np.uint8)
    assert REF.lib.wirehair_recover(codec, _ptr(out), size) == 0
    assert out[:4].tobytes() == b"\x28\xb5\x2f\xfd" or out[:4].tobytes()[0] in (0x50, 0x51, 0x52, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x5b, 0x5c, 0x5d, 0x5e, 0x5f)  # zstd or skippable-frame magic
    REF.lib.wirehair_free(codec)
