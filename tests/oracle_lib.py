"""ctypes bindings for the CPU checker (oracle/liboracle.so) and, when built, the reference's own
OpenCV-free sources (oracle/_ref/libcimbar_ref.so).  TEST INFRASTRUCTURE ONLY: imported by tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline legs -- never by libcimbar_b200/."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

u8p = C.POINTER(C.c_uint8)


class Mode(C.Structure):
    _fields_ = [(n, C.c_int if n in ("mode_val", "fountain_chunks_scalar", "legacy_mode") else C.c_uint) for n in (
        "mode_val", "color_bits", "symbol_bits", "ecc_bytes", "ecc_block_size", "image_size_x", "image_size_y",
        "cell_size", "cell_spacing_x", "cell_spacing_y", "cell_offset", "cells_per_col_x", "cells_per_col_y",
        "fountain_chunks_scalar", "legacy_mode", "corner_padding_x", "corner_padding_y", "total_cells",
        "color_mode", "interleave_blocks", "interleave_partitions", "chunks_per_frame", "chunk_size")]


CELL_DTYPE = np.dtype([("order", "<u2"), ("symbol", "u1"), ("color", "u1"), ("drift_offset", "u1"),
                       ("distance", "u1"), ("x", "<i2"), ("y", "<i2"), ("drift_x", "i1"), ("drift_y", "i1"),
                       ("cooldown_in", "u1")], align=True)


def _ptr(a, t=C.c_uint8):
    return a.ctypes.data_as(C.POINTER(t))


def build_oracle():
    so = os.path.join(ORACLE_DIR, "liboracle.so")
    srcs = [os.path.join(ORACLE_DIR, f) for f in ("cimbar_oracle.c", "cimbar_oracle.h", "oracle_bench.c")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "liboracle.so"], stdout=subprocess.DEVNULL)
    return so


def build_ref():
    """oracle/_ref/libcimbar_ref.so: built from /root/reference where that exists, else the prebuilt file."""
    so = os.path.join(ORACLE_DIR, "_ref", "libcimbar_ref.so")
    if os.path.isdir("/root/reference"):
        srcs = [os.path.join(ORACLE_DIR, f) for f in ("ref_shim.cpp", "cimbar_oracle.c", "Makefile")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.check_call(["make", "-C", ORACLE_DIR, "ref"], stdout=subprocess.DEVNULL)
    return so if os.path.exists(so) else None


class Oracle:
    def __init__(self):
        self.lib = C.CDLL(build_oracle())
        L = self.lib
        L.cbo_mode_init.argtypes = [C.POINTER(Mode), C.c_int]
        L.cbo_capacity.argtypes = [C.POINTER(Mode), C.c_uint]
        L.cbo_capacity.restype = C.c_uint
        L.cbo_decode_raw.argtypes = [C.POINTER(Mode), u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p, C.c_void_p]
        L.cbo_decode.argtypes = [C.POINTER(Mode), u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p, u8p]
        L.cbo_decode_fountain.argtypes = [C.POINTER(Mode), u8p, C.c_int, C.c_int, C.c_int, u8p, C.POINTER(C.c_uint32)]
        L.cbo_rs_create.restype = C.c_void_p
        L.cbo_rs_create.argtypes = [C.c_uint]
        L.cbo_rs_destroy.argtypes = [C.c_void_p]
        L.cbo_rs_decode.argtypes = [C.c_void_p, u8p, C.c_uint, u8p]
        L.cbo_rs_encode.argtypes = [C.c_void_p, u8p, C.c_uint, u8p]
        L.cbo_rs_stream.argtypes = [C.c_uint, C.c_uint, u8p, C.c_uint, u8p, u8p]
        L.cbo_align_chunks.argtypes = [u8p, u8p, C.c_uint, C.c_uint, C.c_uint, u8p, C.POINTER(C.c_uint32)]
        L.cbo_align_chunks.restype = C.c_uint
        L.cbo_preprocess.argtypes = [u8p, C.c_int, C.c_int, C.c_int, u8p]
        L.cbo_rgb_to_gray.argtypes = [u8p, C.c_int, C.c_int, u8p]
        L.cbo_sharpen.argtypes = [u8p, C.c_int, C.c_int, u8p]
        L.cbo_adaptive_threshold.argtypes = [u8p, C.c_int, C.c_int, C.c_int, u8p]
        L.cbo_fuzzy_ahash.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64)]
        L.cbo_best_symbol.argtypes = [C.POINTER(C.c_uint64), C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        L.cbo_best_symbol.restype = C.c_uint
        L.cbo_best_color.argtypes = [C.c_float, C.c_float, C.c_float, C.c_uint, C.c_uint, C.POINTER(C.c_float)]
        L.cbo_best_color.restype = C.c_uint
        L.cbo_avg_color.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p]
        L.cbo_cell_positions.argtypes = [C.POINTER(Mode), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.cbo_adjacent.argtypes = [C.POINTER(Mode), C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.cbo_interleave_reverse.argtypes = [C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_uint)]
        L.cbo_flood_walk_synthetic.argtypes = [C.POINTER(Mode), C.c_uint, C.c_uint, C.POINTER(C.c_uint16), C.POINTER(C.c_int8), u8p]
        L.cbo_payload_to_cells.argtypes = [C.POINTER(Mode), u8p, C.c_uint, u8p]
        L.cbo_render_frame.argtypes = [C.POINTER(Mode), u8p, u8p]
        L.cbo_md_pack.argtypes = [C.c_uint8, C.c_uint, C.c_uint16, u8p]
        L.cbo_md_file_size.argtypes = [u8p]
        L.cbo_md_file_size.restype = C.c_uint
        L.cbo_md_block_id.argtypes = [u8p]
        L.cbo_md_block_id.restype = C.c_uint
        L.cbo_md_encode_id.argtypes = [u8p]
        L.cbo_md_encode_id.restype = C.c_uint
        L.cbo_bench_decode.argtypes = [C.c_int, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u8p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.cbo_bench_decode.restype = C.c_double
        L.cbo_set_ccm.argtypes = [C.POINTER(C.c_float)]
        L.cbo_get_ccm.argtypes = [C.POINTER(C.c_float)]
        L.cbo_adaptation_matrix.argtypes = [C.POINTER(C.c_float)] * 3
        L.cbo_simple_ccm.argtypes = [C.POINTER(Mode), u8p, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.cbo_moore_penrose_lsm.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_float)]
        L.cbo_init_ccm.argtypes = [C.POINTER(Mode), u8p, C.c_int, C.c_int, u8p, C.c_uint, C.POINTER(C.c_float)]
        L.cbo_decode_fountain_cc.argtypes = [C.POINTER(Mode), u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p, C.POINTER(C.c_uint32)]

    def mode(self, mode_val=68):
        m = Mode()
        self.lib.cbo_mode_init(C.byref(m), mode_val)
        return m

    def capacity(self, m, bits=0):
        return self.lib.cbo_capacity(C.byref(m), bits)

    def decode_raw(self, m, rgb, sharpen=False, want_cells=False, color_correction=0):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        out = np.zeros(self.capacity(m), dtype=np.uint8)
        cells = np.zeros(m.total_cells, dtype=CELL_DTYPE) if want_cells else None
        self.lib.cbo_decode_raw(C.byref(m), _ptr(rgb), w, h, int(sharpen), int(color_correction), _ptr(out),
                                cells.ctypes.data if want_cells else None)
        return (out, cells) if want_cells else out

    def set_ccm(self, m9):
        """CimbDecoder::update_color_correction for the calling thread's oracle state; None deactivates it"""
        if m9 is None:
            self.lib.cbo_set_ccm(None)
        else:
            a = np.ascontiguousarray(m9, dtype=np.float32).reshape(9)
            self.lib.cbo_set_ccm(_ptr(a, C.c_float))

    def adaptation_matrix(self, actual, desired):
        a, d, o = (np.asarray(actual, np.float32), np.asarray(desired, np.float32), np.zeros(9, np.float32))
        self.lib.cbo_adaptation_matrix(_ptr(a, C.c_float), _ptr(d, C.c_float), _ptr(o, C.c_float))
        return o.reshape(3, 3)

    def simple_ccm(self, m, rgb):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        o = np.zeros(9, np.float32)
        self.lib.cbo_simple_ccm(C.byref(m), _ptr(rgb), rgb.shape[1], rgb.shape[0], _ptr(o, C.c_float))
        return o.reshape(3, 3)

    def decode(self, m, rgb, use_ecc=True, sharpen=False):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        out = np.zeros(self.capacity(m), dtype=np.uint8)
        ok = np.zeros(128, dtype=np.uint8)
        n = self.lib.cbo_decode(C.byref(m), _ptr(rgb), w, h, int(sharpen), int(use_ecc), _ptr(out), _ptr(ok))
        nblocks = self.capacity(m) // m.ecc_block_size
        return out[:n].copy(), ok[:nblocks].copy()

    def decode_fountain(self, m, rgb, sharpen=False, color_correction=0):
        """Decoder::decode_fountain(img, stream, should_preprocess, color_correction); the CCM state is the calling thread's"""
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        chunks = np.zeros((m.chunks_per_frame, m.chunk_size), dtype=np.uint8)
        mask = C.c_uint32(0)
        good = self.lib.cbo_decode_fountain_cc(C.byref(m), _ptr(rgb), w, h, int(sharpen), int(color_correction), _ptr(chunks), C.byref(mask))
        return good, chunks, mask.value

    def get_ccm(self):
        a = np.zeros(9, np.float32)
        return a.reshape(3, 3) if self.lib.cbo_get_ccm(_ptr(a, C.c_float)) else None

    def moore_penrose_lsm(self, actual, desired):
        a = np.ascontiguousarray(actual, np.float32); d = np.ascontiguousarray(desired, np.float32); o = np.zeros(9, np.float32)
        self.lib.cbo_moore_penrose_lsm(_ptr(a, C.c_float), _ptr(d, C.c_float), a.shape[0], _ptr(o, C.c_float))
        return o.reshape(3, 3)

    def init_ccm(self, m, rgb, hdr6, radioactive):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h6 = np.ascontiguousarray(hdr6, dtype=np.uint8)
        o = np.zeros(9, np.float32)
        rc = self.lib.cbo_init_ccm(C.byref(m), _ptr(rgb), rgb.shape[1], rgb.shape[0], _ptr(h6), int(radioactive), _ptr(o, C.c_float))
        return o.reshape(3, 3) if rc else None

    def preprocess(self, rgb, sharpen=False):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        bits = np.zeros(w * h // 8 + 16, dtype=np.uint8)
        self.lib.cbo_preprocess(_ptr(rgb), w, h, int(sharpen), _ptr(bits))
        return bits[: w * h // 8]

    def payload_to_cells(self, m, payload):
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        cells = np.zeros(m.total_cells, dtype=np.uint8)
        self.lib.cbo_payload_to_cells(C.byref(m), _ptr(payload), payload.size, _ptr(cells))
        return cells

    def render_frame(self, m, cells):
        cells = np.ascontiguousarray(cells, dtype=np.uint8)
        rgb = np.zeros((m.image_size_y, m.image_size_x, 3), dtype=np.uint8)
        self.lib.cbo_render_frame(C.byref(m), _ptr(cells), _ptr(rgb))
        return rgb

    def rs_stream(self, parity, block, raw):
        raw = np.ascontiguousarray(raw, dtype=np.uint8)
        nb = raw.size // block
        out = np.zeros(nb * (block - parity), dtype=np.uint8)
        ok = np.zeros(nb, dtype=np.uint8)
        self.lib.cbo_rs_stream(parity, block, _ptr(raw), raw.size, _ptr(out), _ptr(ok))
        return out, ok

    def bench_decode(self, mode_val, frames, nthreads, stage=1):
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        n, h, w, _ = frames.shape
        cs = C.c_uint64(0)
        secs = self.lib.cbo_bench_decode(mode_val, _ptr(frames), n, w, h, nthreads, stage, None, 0, C.byref(cs))
        return secs, cs.value


class Ref:
    """The reference's own code (libcorrect, wirehair, flood walk, streams) behind oracle/ref_shim.cpp."""

    def __init__(self):
        so = build_ref()
        if so is None:
            raise FileNotFoundError("oracle/_ref/libcimbar_ref.so not built (needs /root/reference once)")
        self.lib = C.CDLL(so)
        L = self.lib
        L.ref_rs_create.restype = C.c_void_p
        L.ref_rs_create.argtypes = [C.c_uint]
        L.ref_rs_destroy.argtypes = [C.c_void_p]
        L.ref_rs_decode2.argtypes = [C.c_void_p, u8p, C.c_uint, u8p]
        L.ref_rs_encode2.argtypes = [C.c_void_p, u8p, C.c_uint, u8p]
        L.ref_cell_positions.argtypes = [C.c_uint] * 4 + [C.c_int, C.c_uint, C.c_uint, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.ref_adjacent.argtypes = [C.c_uint] * 4 + [C.c_int, C.c_uint, C.c_uint, C.c_int, C.POINTER(C.c_int)]
        L.ref_interleave_reverse.argtypes = [C.c_uint, C.c_uint, C.c_uint, C.POINTER(C.c_uint)]
        L.ref_flood_walk_synthetic.argtypes = [C.c_uint] * 4 + [C.c_int, C.c_uint, C.c_uint, C.c_uint, C.c_uint,
                                                                 C.POINTER(C.c_uint16), C.POINTER(C.c_int8), u8p]
        L.ref_fuzzy_ahash.argtypes = [u8p, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.POINTER(C.c_uint64)]
        L.ref_rs_align_escrow.argtypes = [C.c_uint, C.c_uint, u8p, C.c_uint, C.c_uint, C.c_uint, C.c_uint, u8p, C.POINTER(C.c_uint)]
        L.ref_rs_align_escrow.restype = C.c_uint
        L.ref_rs_stream.argtypes = [C.c_uint, C.c_uint, u8p, C.c_uint, u8p]
        L.ref_rs_stream.restype = C.c_uint
        L.ref_md_pack.argtypes = [C.c_uint8, C.c_uint, C.c_uint16, u8p]
        for f in ("ref_md_file_size", "ref_md_block_id", "ref_md_encode_id"):
            getattr(L, f).argtypes = [u8p]
            getattr(L, f).restype = C.c_uint
        # wirehair C API (src/third_party_lib/wirehair/include/wirehair/wirehair.h), linked unmodified
        L.wirehair_init_.argtypes = [C.c_int]
        L.wirehair_encoder_create.restype = C.c_void_p
        L.wirehair_encoder_create.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32]
        L.wirehair_encode.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        L.wirehair_decoder_create.restype = C.c_void_p
        L.wirehair_decoder_create.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
        L.wirehair_decode.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_uint32]
        L.wirehair_recover.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.wirehair_free.argtypes = [C.c_void_p]
        L.wirehair_init_(2)

    def grid_args(self, m, padding=0):
        return (m.cell_spacing_x, m.cell_spacing_y, m.cells_per_col_x, m.cells_per_col_y, m.cell_offset + padding,
                m.corner_padding_x, m.corner_padding_y)


def digest(*parts):
    """SHA-256 over the parts in order (arrays by their bytes, anything else by its repr): the form in which
    tests/golden/ref_outputs.json keeps the reference's results"""
    h = hashlib.sha256()
    for p in parts:
        h.update(np.ascontiguousarray(p).tobytes() if isinstance(p, np.ndarray) else repr(p).encode())
    return h.hexdigest()


def ref_outputs():
    """the reference's results for the inputs of the *_is_the_references / *_matches_* tests, written by
    tests/golden/make_ref_goldens.py from oracle/_ref (the reference's sources compiled unmodified)"""
    with open(os.path.join(GOLDEN_DIR, "ref_outputs.json")) as f:
        return json.load(f)


_manifest = None


def manifest():
    global _manifest
    if _manifest is None:
        with open(os.path.join(GOLDEN_DIR, "manifest.json")) as f:
            _manifest = json.load(f)
    return _manifest


def load_sample(name):
    """imread + BGR2RGB, as the reference's TestCimbar::loadSample (test/TestHelpers.h:8-18)."""
    import cv2
    ent = manifest()["samples"][name]
    if name == "b/scan2434.jpg":
        h, w, _ = ent["shape"]
        img = np.zeros((h, w, 3), dtype=np.uint8)
        img[:8, :8] = np.load(os.path.join(GOLDEN_DIR, ent["file"]))
        return img
    img = cv2.imread(os.path.join(GOLDEN_DIR, ent["file"]), cv2.IMREAD_COLOR)
    return np.ascontiguousarray(cv2.cvtColor(img, cv2.COLOR_BGR2RGB))
