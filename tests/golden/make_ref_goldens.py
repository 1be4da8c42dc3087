#!/usr/bin/env python3
"""Writes tests/golden/ref_outputs.json: the reference's own results for the inputs of tests/test_oracle_vs_ref.py and of the
ScanState / Anchor checks in tests/test_scan_oracle.py, as SHA-256 digests (oracle_lib.digest).  The tests run the same input
sequences through the restatement and compare digests, so they need neither the reference checkout nor oracle/_ref.

    make -C oracle ref && python tests/golden/make_ref_goldens.py

RefSide drives oracle/_ref/libcimbar_ref.so (the reference's OpenCV-free sources compiled unmodified, oracle/ref_shim.cpp)
behind the calls of test_oracle_vs_ref.OracleSide."""
import ctypes as C
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import oracle_lib as ol                     # noqa: E402
import test_oracle_vs_ref as T              # noqa: E402
import test_scan_oracle as S                # noqa: E402
from oracle_lib import _ptr                 # noqa: E402

REF = ol.Ref()
L = REF.lib


class RefSide:
    def cell_positions(self, m, xs, ys):
        return L.ref_cell_positions(*REF.grid_args(m), _ptr(xs, C.c_int), _ptr(ys, C.c_int))

    def adjacent(self, m, xs, idx, out):
        L.ref_adjacent(*REF.grid_args(m), idx, _ptr(out, C.c_int))

    def interleave_reverse(self, args, out):
        L.ref_interleave_reverse(*args, _ptr(out, C.c_uint))

    def flood_walk(self, m, seed, noise, o, d, c):
        return L.ref_flood_walk_synthetic(*REF.grid_args(m), seed, noise, _ptr(o, C.c_uint16), _ptr(d, C.c_int8), _ptr(c))

    def fuzzy_ahash(self, bits, w, wx, wy, all_, out):
        L.ref_fuzzy_ahash(_ptr(bits), bits.size, w, wx, wy, all_, out)

    def rs_create(self, parity):
        return L.ref_rs_create(parity)

    def rs_destroy(self, h):
        L.ref_rs_destroy(h)

    def rs_encode(self, h, msg, out):
        return L.ref_rs_encode2(h, _ptr(msg), msg.size, _ptr(out))

    def rs_decoder(self, encoder, parity):
        return L.ref_rs_create(parity)

    def rs_decode(self, h, blk, out):
        return L.ref_rs_decode2(h, _ptr(blk), blk.size, _ptr(out))

    def rs_stream(self, parity, block, raw, sym_len):
        out = np.zeros((raw.size // block) * (block - parity) + 16, np.uint8)
        n = L.ref_rs_stream(parity, block, _ptr(raw), sym_len, _ptr(out))
        return out[:n]

    def rs_align(self, m, raw, sym_len, col_len):
        chunks = np.zeros((m.chunks_per_frame, m.chunk_size), np.uint8)
        used = C.c_uint(0)
        good = L.ref_rs_align_escrow(m.ecc_bytes, m.ecc_block_size, _ptr(raw), sym_len, col_len, m.chunk_size, m.chunks_per_frame,
                                     _ptr(chunks), C.byref(used))
        return good, used.value, chunks

    def md_pack(self, eid, size, bid, out):
        L.ref_md_pack(eid, size, bid, _ptr(out))

    def md_fields(self, a):
        return L.ref_md_file_size(_ptr(a)), L.ref_md_block_id(_ptr(a)), L.ref_md_encode_id(_ptr(a))


def ref_scanstate(kind, row):
    n = row.size
    res = (C.c_int * (n + 1))()
    L.ref_scanstate_run(kind, _ptr(np.ascontiguousarray(row)), n, res)
    want = [(x - res[x], x - 1, 0, 0) for x in range(n) if res[x] > 0]
    if res[n] > 0:
        want.append((n - res[n], n - 1, 0, 0))
    return want


def ref_anchor_op(a, b):
    ra, out = (C.c_int * 4)(*a), (C.c_longlong * 7)()
    L.ref_anchor_ops(ra, (C.c_int * 4)(*b), 32, out)
    merged = [tuple(ra)] if out[6] == 1 else [a, b]
    return merged, "%d+-%d,%d+-%d" % (out[0], out[2], out[1], out[3]), ((3 * out[5]) & 0xFFFFFFFF) // 8


def main():
    L.ref_scanstate_run.argtypes = [C.c_int, C.POINTER(C.c_uint8), C.c_int, C.POINTER(C.c_int)]
    L.ref_anchor_ops.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_longlong)]
    side, d = RefSide(), ol.digest
    gold = {
        "cell_positions_and_adjacency": {str(m): d(*T.cell_positions_and_adjacency(side, m)) for m in T.MODES},
        "interleave_reverse": {repr(a): d(T.interleave_reverse(side, a)) for a in T.INTERLEAVE_ARGS},
        "flood_walk": {"%d/%d" % (m, z): d(*T.flood_walks(side, m, z)) for m in T.WALK_MODES for z in T.WALK_NOISE},
        "fuzzy_ahash": d(T.fuzzy_ahashes(side)),
        "rs_known_answer": d(T.rs_known_answer(side)),
        "rs_decode": {"%d/%d" % pb: d(*T.rs_decode_outputs(T.rs_decode_trials(side, *pb))) for pb in T.RS_CODES},
        "rs_stream_and_aligned_chunks": {str(m): d(*T.rs_stream_and_aligned_chunks(side, m)) for m in T.STREAM_MODES},
        "fountain_metadata": d(*T.fountain_metadata(side)),
        "scanstate_patterns": d(S.scanstate_patterns(ref_scanstate)),
        "anchor_ops": d(S.anchor_ops(ref_anchor_op)),
    }
    with open(os.path.join(HERE, "ref_outputs.json"), "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
