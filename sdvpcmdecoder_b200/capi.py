"""ctypes binding of lib/libsdvpcm_b200.so (include/sdvpcm.h).

PyTorch is used only to own device memory and streams; every compute call goes through the C ABI.  There is no CPU
path: loading fails loudly when the library has not been built, and every compute call fails with SDV_ERR_CUDA
when there is no CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from ._build import LIB_PATH

SDV_OK, SDV_ERR_ARG, SDV_ERR_CUDA, SDV_ERR_UNSUPPORTED, SDV_ERR_NOMEM = 0, -1, -2, -3, -4
TYPE_PCM1, TYPE_PCM16X0, TYPE_STC007, TYPE_M2 = 0, 1, 2, 3
MODE_DRAFT, MODE_FAST, MODE_NORMAL, MODE_INSANE = 0, 1, 2, 3
RES_MODE_14BIT, RES_MODE_14BIT_AUTO, RES_MODE_16BIT_AUTO, RES_MODE_16BIT = 0, 1, 2, 3
SRV_NO, SRV_HEADER_LINE, SRV_CTRL_BLOCK = 0, 6, 7
LF_CRC_OK, LF_CRC_OK_IGN, LF_FORCED_BAD, LF_BW_SET, LF_COORDS_SET, LF_REF_SWEEP, LF_BY_EXT = 1, 2, 4, 8, 16, 32, 64
LF_COORD_SWEEP = 128
LF_MARKERS, LF_START_MARK, LF_STOP_MARK, LF_ALMOST_SILENT = 1 << 8, 1 << 9, 1 << 10, 1 << 12
SF_BLOCK_OK, SF_WORD_VALID, SF_WORD_FIXED = 1, 2, 4
BF_VALID, BF_BROKEN, BF_FIX_P, BF_FIX_Q, BF_SILENT, BF_UNSAFE = 1, 2, 4, 8, 16, 32

LINE_REC = np.dtype([("words", "<u2", (9,)), ("flags", "<u2"), ("ref", "u1"), ("black", "u1"), ("white", "u1"),
                     ("hyst", "u1"), ("data_start", "<i2"), ("data_stop", "<i2"), ("shift", "u1"),
                     ("service_type", "u1"), ("mark_stages", "u1"), ("reserved", "u1")])
LINE_AUX = np.dtype([("ref_low", "u1"), ("ref_high", "u1"), ("marker_start_bg", "<u2"), ("marker_start_ed", "<u2"),
                     ("marker_stop_ed", "<u2"), ("word_crc_mask", "<u2"), ("word_valid_mask", "<u2"), ("pad", "u1", (4,))])
BLOCK_REC = np.dtype([("words", "<u2", (8,)), ("line_crc", "u1"), ("word_valid", "u1"), ("audio_state", "u1"),
                      ("resolution", "u1"), ("flags", "u1"), ("reserved", "u1", (11,))])
PCM1_SUBLINE = np.dtype([("left", "<u2"), ("right", "<u2"), ("flags", "u1"), ("reserved", "u1", (3,))])
P1F_CRC_OK, P1F_BW_SET, P1F_PICKED_LEFT, P1F_PICKED_RIGHT = 1, 2, 4, 8
PCM1_FRAME_INFO = np.dtype([("odd_top", "<u2"), ("odd_bottom", "<u2"), ("even_top", "<u2"), ("even_bottom", "<u2"),
                            ("odd_data_lines", "<u2"), ("even_data_lines", "<u2"), ("header_present", "u1"),
                            ("emphasis_set", "u1"), ("reserved", "u1", (2,))])
assert PCM1_FRAME_INFO.itemsize == 16
SEAM = np.dtype([("f1_first", "<u4"), ("f1_size", "<u4"), ("f2_first", "<u4"), ("f2_size", "<u4")])
PCM16X0_FRAME_INFO = np.dtype([("sample_rate", "<u2"), ("emphasis", "u1"), ("code", "u1"), ("frame_votes", "u1"), ("reserved", "u1", (3,))])
PADDING = np.dtype([("padding", "<u2"), ("result", "u1"), ("last_pad_counter", "u1")])
STITCH_STATS = np.dtype([("index", "<u2"), ("valid", "<u2"), ("silent", "<u2"), ("unchecked", "<u2"), ("broken", "<u2"),
                         ("result", "u1"), ("reserved", "u1")])
STC007_FRAME_INFO = np.dtype([("start", "<i4"), ("pre", "<u2"), ("n1", "<u2"), ("inner", "<u2"), ("n2", "<u2"), ("outer", "<u2"),
                              ("skip1", "<u2"), ("skip2", "<u2"), ("odd_top", "<u2"), ("odd_bottom", "<u2"), ("even_top", "<u2"),
                              ("even_bottom", "<u2"), ("odd_data_lines", "<u2"), ("even_data_lines", "<u2"), ("odd_valid_lines", "<u2"),
                              ("even_valid_lines", "<u2"), ("inner_padding", "<u2"), ("outer_padding", "<u2"), ("field_order", "u1"),
                              ("video_std", "u1"), ("flags", "u1"), ("odd_res_mode", "u1"), ("even_res_mode", "u1"), ("reserved", "u1")])
assert STC007_FRAME_INFO.itemsize == 44
FA_INNER_OK, FA_OUTER_OK, FA_INNER_SILENCE, FA_OUTER_SILENCE, FA_ORDER_GUESSED, FA_MASK_INNER, FA_MASK_PREV_OUTER = 1, 2, 4, 8, 16, 32, 64
BF_CWD = 64          # sdv_block_rec.flags: isDataFixedByCWD
VID_UNKNOWN, VID_PAL, VID_NTSC = 0, 1, 2
ORDER_UNK, ORDER_TFF, ORDER_BFF = 0, 1, 2
PCM16X0_ALIGNMENT = np.dtype([("top_padding", "<i2", (2,)), ("cut_lines", "<i2", (2,)), ("lines", "<i2", (2,)), ("result", "u1", (2,)),
                              ("mask_seams", "u1"), ("reserved", "u1")])
assert PCM16X0_ALIGNMENT.itemsize == 16
DS_RET_NO_DATA, DS_RET_SILENCE, DS_RET_BROKE, DS_RET_NO_PAD, DS_RET_OK = range(5)
PCM16X0_SUBLINE = np.dtype([("words", "<u2", (3,)), ("flags", "u1"), ("picked_left", "u1")])
X0F_CRC_OK, X0F_HAS_DATA, X0F_PICKED_RIGHT = 1, 2, 8
assert PCM16X0_SUBLINE.itemsize == 8
assert LINE_REC.itemsize == 32 and LINE_AUX.itemsize == 16 and BLOCK_REC.itemsize == 32 and PCM1_SUBLINE.itemsize == 8


class BinConfig(C.Structure):
    _fields_ = [("pcm_type", C.c_uint8), ("mode", C.c_uint8), ("check_line_dup", C.c_uint8), ("reserved", C.c_uint8 * 13)]


class DeintConfig(C.Structure):
    _fields_ = [("res_mode", C.c_uint8), ("ignore_crc", C.c_uint8), ("force_check", C.c_uint8), ("p_corr", C.c_uint8),
                ("q_corr", C.c_uint8), ("broken_mask_dur", C.c_uint8), ("m2_format", C.c_uint8), ("countdown_in", C.c_uint8),
                ("cwd", C.c_uint8), ("reserved", C.c_uint8 * 7)]


class BinPreset(C.Structure):
    """sdv_bin_preset = bin_preset_t (binarizer.h:163-186)."""
    _fields_ = [("max_black_lvl", C.c_uint8), ("min_white_lvl", C.c_uint8), ("min_contrast", C.c_uint8), ("min_ref_lvl", C.c_uint8),
                ("max_ref_lvl", C.c_uint8), ("min_valid_crcs", C.c_uint8), ("mark_max_dist", C.c_uint8), ("left_bit_pick", C.c_uint8),
                ("right_bit_pick", C.c_uint8), ("en_force_coords", C.c_uint8), ("en_coord_search", C.c_uint8),
                ("en_first_line_dup", C.c_uint8), ("en_good_no_marker", C.c_uint8), ("reserved", C.c_uint8),
                ("horiz_start", C.c_int16), ("horiz_stop", C.c_int16), ("reserved2", C.c_uint8 * 14)]


class StitchConfig(C.Structure):
    _fields_ = [("video_std", C.c_uint8), ("field_order", C.c_uint8), ("resolution_16bit", C.c_uint8), ("file_start", C.c_uint8),
                ("file_end", C.c_uint8), ("mask_seams", C.c_uint8), ("fix_cut_above", C.c_uint8), ("max_unchecked_14bit", C.c_uint8),
                ("max_unchecked_16bit", C.c_uint8), ("reserved", C.c_uint8 * 7)]


class Countdown(C.Structure):
    _fields_ = [("countdown_in", C.c_uint8), ("countdown_out", C.c_uint8), ("depends_on_in", C.c_uint8), ("reserved", C.c_uint8),
                ("windows", C.c_uint32)]


class Geometry(C.Structure):
    _fields_ = [("lines_per_field", C.c_uint16), ("lead_in", C.c_uint16), ("reserved", C.c_uint16 * 6)]


class BinStats(C.Structure):
    _fields_ = [("lines_total", C.c_uint64), ("lines_fast", C.c_uint64), ("lines_chain", C.c_uint64),
                ("frames_skipped", C.c_uint64), ("kernel_launches", C.c_uint32), ("reserved", C.c_uint32)]


class Pcm16x0Config(C.Structure):
    _fields_ = [("ignore_crc", C.c_uint8), ("force_check", C.c_uint8), ("p_corr", C.c_uint8), ("ei_format", C.c_uint8),
                ("continue_file", C.c_uint8), ("reserved", C.c_uint8 * 3)]


class Pcm1StitchConfig(C.Structure):
    _fields_ = [("ignore_crc", C.c_uint8), ("bff", C.c_uint8), ("file_start", C.c_uint8), ("manual_offset", C.c_uint8),
                ("odd_offset", C.c_int8), ("even_offset", C.c_int8), ("reserved", C.c_uint8 * 2)]


class Pcm16x0Geometry(C.Structure):
    _fields_ = [("bff", C.c_uint8), ("top_padding_odd", C.c_uint8), ("top_padding_even", C.c_uint8),
                ("broken_mask_dur", C.c_uint8), ("reserved", C.c_uint8 * 4)]


class Timings(C.Structure):
    _fields_ = [("bulk_ms", C.c_float), ("deint_ms", C.c_float), ("bulk_lines", C.c_uint64), ("deint_blocks", C.c_uint64),
                ("bulk_launches", C.c_uint32), ("deint_launches", C.c_uint32), ("kernel_launches", C.c_uint32),
                ("reserved", C.c_uint32)]


EXPORTS = ("sdv_create", "sdv_destroy", "sdv_last_error", "sdv_version", "sdv_bin_decode_frames", "sdv_bin_on_first_frame", "sdv_deint_stc007",
           "sdv_stc007_frames_to_samples", "sdv_stc007_shard_to_samples", "sdv_stc007_block_count", "sdv_stc007_find_padding",
           "sdv_stc007_decode_tape_host", "sdv_bin_last_stats", "sdv_timings_read", "sdv_deint_pcm1", "sdv_deint_pcm16x0", "sdv_stc007_try_padding",
           "sdv_pcm1_frames_to_samples", "sdv_pcm16x0_frames_to_samples", "sdv_pcm16x0_frames_to_samples_info", "sdv_pcm1_decode_tape_host", "sdv_pcm16x0_decode_tape_host",
           "sdv_stc007_stitch_frames", "sdv_stc007_stitch_block_bound", "sdv_stc007_countdown", "sdv_stc007_countdown_copy", "sdv_pcm16x0_frames_to_samples_auto",
           "sdv_bin_default_fine_settings", "sdv_bin_get_fine_settings", "sdv_bin_set_fine_settings", "sdv_bin_decode_verify", "sdv_stc007_fuse_next_decode")

FIRST_FRAME_FN = C.CFUNCTYPE(None, C.c_void_p)
_lib = None


class SdvError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"sdvpcm error {code}: {msg}")
        self.code = code


def lib():
    """The CUDA library.  Raises if it has not been built: the product has no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a).  sdvpcmdecoder_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        vp, ci = C.c_void_p, C.c_int
        l.sdv_create.argtypes = [C.POINTER(vp), ci]
        l.sdv_destroy.argtypes = [vp]
        l.sdv_destroy.restype = None
        l.sdv_last_error.argtypes = [vp]
        l.sdv_last_error.restype = C.c_char_p
        l.sdv_bin_decode_frames.argtypes = [vp, C.POINTER(BinConfig), vp, ci, ci, ci, ci, vp, vp, vp]
        l.sdv_deint_stc007.argtypes = [vp, C.POINTER(DeintConfig), vp, ci, vp, vp, vp, vp]
        l.sdv_bin_on_first_frame.argtypes = [vp, FIRST_FRAME_FN, vp]
        l.sdv_stc007_frames_to_samples.argtypes = [vp, C.POINTER(DeintConfig), C.POINTER(Geometry), vp, ci, ci, vp, vp, vp, vp]
        l.sdv_stc007_shard_to_samples.argtypes = [vp, C.POINTER(DeintConfig), C.POINTER(Geometry), vp, ci, ci, vp, vp, vp, vp, vp]
        l.sdv_timings_read.argtypes = [vp, C.POINTER(Timings), ci]
        l.sdv_stc007_block_count.argtypes = [C.POINTER(Geometry), ci]
        l.sdv_stc007_decode_tape_host.argtypes = [vp, C.POINTER(BinConfig), C.POINTER(DeintConfig), C.POINTER(Geometry),
                                                  vp, ci, ci, ci, vp, vp, vp]
        l.sdv_bin_last_stats.argtypes = [vp, C.POINTER(BinStats)]
        l.sdv_deint_pcm1.argtypes = [vp, ci, vp, ci, vp, vp, vp]
        l.sdv_pcm16x0_frames_to_samples.argtypes = [vp, C.POINTER(Pcm16x0Config), C.POINTER(Pcm16x0Geometry), vp, ci, ci, vp, vp, vp, vp]
        l.sdv_pcm16x0_frames_to_samples_info.argtypes = [vp, C.POINTER(Pcm16x0Config), C.POINTER(Pcm16x0Geometry), vp, ci, ci, vp, vp, vp, vp, vp]
        l.sdv_pcm1_decode_tape_host.argtypes = [vp, C.POINTER(BinConfig), C.POINTER(Pcm1StitchConfig), vp, ci, ci, ci, vp, vp, vp]
        l.sdv_pcm16x0_decode_tape_host.argtypes = [vp, C.POINTER(BinConfig), C.POINTER(Pcm16x0Config), C.POINTER(Pcm16x0Geometry), vp, ci, ci, ci, vp, vp, vp]
        l.sdv_pcm1_frames_to_samples.argtypes = [vp, C.POINTER(Pcm1StitchConfig), vp, ci, ci, vp, vp, vp, vp]
        l.sdv_stc007_try_padding.argtypes = [vp, C.POINTER(DeintConfig), ci, ci, vp, vp, ci, ci, vp, vp]
        l.sdv_stc007_find_padding.argtypes = [vp, C.POINTER(DeintConfig), ci, ci, ci, ci, vp, vp, ci, vp, vp]
        l.sdv_deint_pcm16x0.argtypes = [vp, C.POINTER(Pcm16x0Config), vp, ci, vp, vp, vp, vp]
        l.sdv_stc007_stitch_frames.argtypes = [vp, C.POINTER(DeintConfig), C.POINTER(StitchConfig), vp, ci, ci, vp, vp, vp,
                                               C.POINTER(ci), C.POINTER(ci), vp, vp]
        l.sdv_pcm16x0_frames_to_samples_auto.argtypes = [vp, C.POINTER(Pcm16x0Config), C.POINTER(Pcm16x0Geometry), vp, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        l.sdv_stc007_stitch_block_bound.argtypes = [ci]
        l.sdv_stc007_countdown.argtypes = [vp, C.POINTER(Countdown), vp]
        l.sdv_stc007_countdown_copy.argtypes = [vp, vp, vp]
        l.sdv_bin_default_fine_settings.argtypes = [C.POINTER(BinPreset)]
        l.sdv_bin_get_fine_settings.argtypes = [vp, C.POINTER(BinPreset)]
        l.sdv_bin_set_fine_settings.argtypes = [vp, C.POINTER(BinPreset)]
        l.sdv_bin_decode_verify.argtypes = [vp, C.POINTER(ci)]
        l.sdv_stc007_fuse_next_decode.argtypes = [vp, C.POINTER(DeintConfig), C.POINTER(Geometry), vp, vp]
        _lib = l
    return _lib


class Handle:
    """One decoder context bound to one CUDA device (sdv_create / sdv_destroy)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        rc = lib().sdv_create(C.byref(self._h), int(device))
        if rc != SDV_OK:
            raise SdvError(rc, "sdv_create failed (no CUDA device? there is no CPU fallback)")
        self.device = int(device)

    def close(self):
        if self._h:
            lib().sdv_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != SDV_OK:
            raise SdvError(rc, lib().sdv_last_error(self._h).decode())

    @property
    def ptr(self):
        return self._h

    def timings(self, reset: bool = False) -> dict:
        """Accumulated device time of the bulk and deinterleave launches since the last reset (sdv_timings_read)."""
        t = Timings()
        self.check(lib().sdv_timings_read(self._h, C.byref(t), int(reset)))
        return {k: getattr(t, k) for k, _ in Timings._fields_}

    def last_stats(self) -> dict:
        s = BinStats()
        self.check(lib().sdv_bin_last_stats(self._h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in BinStats._fields_}
