"""Host-side mirror of the reference's operator surface for the batch-decode path, above the C ABI.

Class and method names follow the reference (VideoToDigital videotodigital.h:129-165, STC007Deinterleaver
stc007deinterleaver.h:159-173, STC007DataStitcher stc007datastitcher.h:286-352) so that a parity test reads like a
use of the reference; the difference is that one call takes a batch of frames resident in HBM instead of one line
from a queue.  All compute happens in the CUDA library; torch only owns the device buffers.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import capi
from .capi import (DeintConfig, BinConfig, Geometry, LINE_REC, LINE_AUX, BLOCK_REC, MODE_NORMAL, TYPE_STC007,
                   RES_MODE_14BIT, RES_MODE_16BIT)

VID_UNKNOWN, VID_PAL, VID_NTSC = 0, 1, 2            # FrameAsmDescriptor::VID_* (frametrimset.h:121-127)
LINES_PER_FIELD = {VID_PAL: 294, VID_NTSC: 245}     # config.h:80-81
LEAD_IN_LINES = 80                                   # STC007DataBlock::LINE_R2 (stc007datastitcher.cpp:4733-4737)


def _stream_ptr(stream):
    if stream is None:
        stream = torch.cuda.current_stream()
    return C.c_void_p(stream.cuda_stream)


def _dev_u8(t: torch.Tensor) -> torch.Tensor:
    if not (t.is_cuda and t.dtype == torch.uint8 and t.is_contiguous()):
        raise ValueError("expected a contiguous CUDA uint8 tensor")
    return t


def records_to_numpy(t: torch.Tensor, dtype) -> np.ndarray:
    """Device record buffer (uint8 [n, itemsize]) -> structured host array."""
    return t.cpu().numpy().reshape(-1).view(dtype)


class VideoToDigital:
    """Line decode over whole frames (VideoToDigital::doBinarize, videotodigital.cpp:698-1815)."""

    TYPE_PCM1, TYPE_PCM16X0, TYPE_STC007 = 0, 1, 2

    def __init__(self, handle: capi.Handle | None = None, device: int = 0):
        self.handle = handle or capi.Handle(device)
        self.pcm_type = TYPE_STC007
        self.mode = MODE_NORMAL
        self.check_line_dup = True
        self.chain_segments = 1     # > 1: decode the batch as that many independent files in parallel (sdv_bin_config)
        self.warm_start = True      # False: no speculative bulk launch with the previous call's presets (scheduling only)
        self.relay = True           # False: a damaged tape stays on the single sequential chain (scheduling only: relay mode is exact)

    def setPCMType(self, t):
        self.pcm_type = int(t)

    def setBinarizationMode(self, m):
        self.mode = int(m)

    def setCheckLineDup(self, flag):
        self.check_line_dup = bool(flag)

    def getDefaultFineSettings(self) -> "capi.BinPreset":
        p = capi.BinPreset()
        capi.lib().sdv_bin_default_fine_settings(C.byref(p))
        return p

    def getCurrentFineSettings(self) -> "capi.BinPreset":
        p = capi.BinPreset()
        self.handle.check(capi.lib().sdv_bin_get_fine_settings(self.handle.ptr, C.byref(p)))
        return p

    def setFineSettings(self, preset=None, **fields):
        """VideoToDigital::setFineSettings(bin_preset_t) (videotodigital.cpp:667-676): a capi.BinPreset, or the current settings
        with the given fields changed, e.g. setFineSettings(min_valid_crcs=3, mark_max_dist=10)."""
        p = preset if preset is not None else self.getCurrentFineSettings()
        for k, v in fields.items():
            setattr(p, k, int(v))
        self.handle.check(capi.lib().sdv_bin_set_fine_settings(self.handle.ptr, C.byref(p)))

    def setDefaultFineSettings(self):
        self.setFineSettings(self.getDefaultFineSettings())

    def verify(self) -> bool:
        """The answer to a doBinarize(lazy=True) call (sdv_bin_decode_verify): False = its records stand; True = a frame was not
        clean and the tape has been decoded again into the same buffer -- redo what was computed from the records."""
        r = C.c_int(0)
        self.handle.check(capi.lib().sdv_bin_decode_verify(self.handle.ptr, C.byref(r)))
        return bool(r.value)

    def doBinarize(self, luma: torch.Tensor, want_aux: bool = False, stream=None, out: torch.Tensor | None = None,
                   on_first_frame=None, continue_file: bool = False, lazy: bool = False):
        """luma: CUDA uint8 [F, H, W] (interlaced frames).  Returns the record buffer uint8 [F*H, 32] (and the
        auxiliary buffer uint8 [F*H, 16]) in the reference's stream order: per frame, odd-field rows then even-field rows
        (PCM-16x0: three sub-line records per row, [F*H*3, 32]).  continue_file: the batch continues the file of the previous
        call on the handle (same PCM type, geometry, mode and duplicate check), so a tape fed in batches decodes as in one call;
        any format (STC-007, M2, PCM-1, PCM-16x0)."""
        luma = _dev_u8(luma)
        f, h, w = luma.shape
        n = f * h * (3 if self.pcm_type == capi.TYPE_PCM16X0 else 1)
        recs = out if out is not None else torch.empty((n, LINE_REC.itemsize), dtype=torch.uint8, device=luma.device)
        assert recs.shape[0] >= n and recs.shape[1] == LINE_REC.itemsize
        aux = torch.empty((n, LINE_AUX.itemsize), dtype=torch.uint8, device=luma.device) if want_aux else None
        cfg = BinConfig(pcm_type=self.pcm_type, mode=self.mode, check_line_dup=int(self.check_line_dup))
        cfg.reserved[0], cfg.reserved[1] = self.chain_segments & 0xFF, (self.chain_segments >> 8) & 0xFF
        cfg.reserved[2] = (0 if self.warm_start else 1) | (0 if self.relay else 4) | (2 if lazy else 0)     # lazy: call verify() afterwards
        cfg.reserved[3] = 1 if continue_file else 0          # the batch continues the file of the previous call
        hook = None
        if on_first_frame is not None:
            # called as soon as the first frame's records are final (sdv_bin_on_first_frame): a shard starts its halo send here
            hook = capi.FIRST_FRAME_FN(lambda _user: on_first_frame())
            capi.lib().sdv_bin_on_first_frame(self.handle.ptr, hook, None)
        try:
            rc = capi.lib().sdv_bin_decode_frames(self.handle.ptr, C.byref(cfg), C.c_void_p(luma.data_ptr()), f, h, w, w,
                                                  C.c_void_p(recs.data_ptr()), C.c_void_p(aux.data_ptr()) if want_aux else None,
                                                  _stream_ptr(stream))
        finally:
            if hook is not None:
                capi.lib().sdv_bin_on_first_frame(self.handle.ptr, capi.FIRST_FRAME_FN(), None)
        self.handle.check(rc)
        return (recs, aux) if want_aux else recs

    def saveState(self, out: torch.Tensor | None = None, stream=None, pcm_type: int | None = None) -> torch.Tensor:
        """The open file of the line decode (what doBinarize(continue_file=True) would continue) as a canonical uint8 CUDA tensor
        of sdv_bin_chain_state_bytes() bytes (sdv_bin_chain_state_save): equal states give equal bytes.  pcm_type (default: this
        operator's) selects the STC-007 / M2 file or the PCM-1 / PCM-16x0 one.  No synchronisation."""
        n = int(capi.lib().sdv_bin_chain_state_bytes())
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=torch.device("cuda", self.handle.device))
        out = _dev_u8(out)
        assert out.numel() == n
        t = self.pcm_type if pcm_type is None else int(pcm_type)
        self.handle.check(capi.lib().sdv_bin_chain_state_save(self.handle.ptr, t, C.c_void_p(out.data_ptr()), _stream_ptr(stream)))
        return out

    def loadState(self, state: torch.Tensor, stream=None):
        """Make [state] (from saveState, on any handle or device) the open file of its kind on this handle: the next
        doBinarize(continue_file=True) with the saved PCM type, geometry, mode and duplicate check continues it exactly
        (sdv_bin_chain_state_load).  The handle's fine settings must be the ones the state was saved with."""
        state = _dev_u8(state)
        assert state.numel() == int(capi.lib().sdv_bin_chain_state_bytes())
        self.handle.check(capi.lib().sdv_bin_chain_state_load(self.handle.ptr, C.c_void_p(state.data_ptr()), _stream_ptr(stream)))

    def stats(self) -> dict:
        return self.handle.last_stats()


class _DeintSettings:
    def __init__(self):
        self.res_mode = RES_MODE_14BIT
        self.ignore_crc = False
        self.force_check = True
        self.p_corr = True
        self.q_corr = True
        self.broken_mask_dur = 0
        self.m2_format = False

    def setResMode(self, m):
        self.res_mode = int(m)

    def setIgnoreCRC(self, f):
        self.ignore_crc = bool(f)

    def setForcedErrorCheck(self, f):
        self.force_check = bool(f)

    def setPCorrection(self, f):
        self.p_corr = bool(f)
        if not self.p_corr:             # stc007deinterleaver.cpp:228-233
            self.q_corr = False

    def setQCorrection(self, f):
        self.q_corr = bool(f)
        if self.q_corr:                 # stc007deinterleaver.cpp:255-259
            self.p_corr = True

    def setM2SampleFormat(self, f):
        self.m2_format = bool(f)

    def setCWDCorrection(self, flag: bool):
        """STC007DataStitcher::setCWDCorrection (honoured by doFrameReassembleAuto; the reference's default is on, here it is off
        unless set: the preset-geometry calls have no frame queue for CWD to work on)."""
        self.cwd = bool(flag)

    def _cfg(self, countdown_in: int = 0, cwd: bool = False):
        if not 0 <= int(self.broken_mask_dur) <= 255 or not 0 <= int(countdown_in) <= 255:
            raise ValueError("broken-block mask duration / countdown must be 0..255 (uint8_t in the reference, stc007datastitcher.h)")
        return DeintConfig(res_mode=self.res_mode, ignore_crc=int(self.ignore_crc), force_check=int(self.force_check),
                           p_corr=int(self.p_corr), q_corr=int(self.q_corr), broken_mask_dur=int(self.broken_mask_dur),
                           m2_format=int(self.m2_format), countdown_in=int(countdown_in), cwd=int(bool(cwd)))


class STC007Deinterleaver(_DeintSettings):
    """STC007Deinterleaver::processBlock (stc007deinterleaver.cpp:286-1123) for every start line of an assembled line array."""

    def __init__(self, handle: capi.Handle | None = None, device: int = 0):
        super().__init__()
        self.handle = handle or capi.Handle(device)

    def processBlocks(self, lines: torch.Tensor, want_blocks: bool = True, stream=None, countdown_in: int = 0):
        """lines: CUDA uint8 [n, 32] line records; countdown_in: what the blocks before left of a broken-block window.  Returns (blocks uint8 [n-112, 32] | None, samples int16 [n-112, 6], flags uint8 [n-112, 6])."""
        lines = _dev_u8(lines)
        n = lines.shape[0]
        nb = max(n - 112, 0)
        dev = lines.device
        blocks = torch.empty((nb, BLOCK_REC.itemsize), dtype=torch.uint8, device=dev) if want_blocks else None
        samples = torch.empty((nb, 6), dtype=torch.int16, device=dev)
        flags = torch.empty((nb, 6), dtype=torch.uint8, device=dev)
        cfg = self._cfg(countdown_in)
        rc = capi.lib().sdv_deint_stc007(self.handle.ptr, C.byref(cfg), C.c_void_p(lines.data_ptr()), n,
                                         C.c_void_p(blocks.data_ptr()) if want_blocks else None,
                                         C.c_void_p(samples.data_ptr()), C.c_void_p(flags.data_ptr()), _stream_ptr(stream))
        self.handle.check(rc)
        return blocks, samples, flags


class PCM1Deinterleaver:
    """PCM1Deinterleaver::processBlock (pcm1deinterleaver.cpp:69-278) for the 8 interleave blocks of every field."""

    def __init__(self, handle: capi.Handle | None = None, device: int = 0):
        self.handle = handle or capi.Handle(device)
        self.ignore_crc = False

    def setIgnoreCRC(self, f):
        self.ignore_crc = bool(f)

    def processFields(self, sublines: torch.Tensor, stream=None):
        """sublines: CUDA uint8 [n_fields*735, 8] (capi.PCM1_SUBLINE).  Returns (samples int16 [n_fields*1470], flags uint8 [n_fields*1470])."""
        sublines = _dev_u8(sublines)
        assert sublines.shape[0] % 735 == 0 and sublines.shape[1] == capi.PCM1_SUBLINE.itemsize
        n_fields = sublines.shape[0] // 735
        samples = torch.empty(n_fields * 1470, dtype=torch.int16, device=sublines.device)
        flags = torch.empty(n_fields * 1470, dtype=torch.uint8, device=sublines.device)
        rc = capi.lib().sdv_deint_pcm1(self.handle.ptr, int(self.ignore_crc), C.c_void_p(sublines.data_ptr()), n_fields,
                                       C.c_void_p(samples.data_ptr()), C.c_void_p(flags.data_ptr()), _stream_ptr(stream))
        self.handle.check(rc)
        return samples, flags


class PCM1DataStitcher:
    """PCM1DataStitcher::doFrameReassemble with automatic line offset (pcm1datastitcher.cpp:202-1218,1382-1453): trim,
    split into sub-lines, pad to 735 per field, field order, deinterleave -- for all frames of a batch."""

    ORDER_TFF, ORDER_BFF = 1, 2                  # FrameAsmDescriptor::ORDER_*

    def __init__(self, handle: capi.Handle | None = None, device: int = 0):
        self.handle = handle or capi.Handle(device)
        self.ignore_crc = False
        self.field_order = self.ORDER_TFF
        self.auto_offset, self.odd_offset, self.even_offset = True, 0, 0

    def setIgnoreCRC(self, f):
        self.ignore_crc = bool(f)

    def setFieldOrder(self, order):
        self.field_order = self.ORDER_BFF if int(order) == self.ORDER_BFF else self.ORDER_TFF

    def setAutoLineOffset(self, f):
        self.auto_offset = bool(f)

    def setOddLineOffset(self, n):
        self.odd_offset = int(n)

    def setEvenLineOffset(self, n):
        self.even_offset = int(n)

    def doFrameReassemble(self, recs: torch.Tensor, n_frames: int, height: int, want_info: bool = False, stream=None,
                          file_start: bool = True):
        """recs: the PCM-1 line records of VideoToDigital.doBinarize (file_start: frame 0 opens the file).  Returns (samples int16 [n_frames*2940], flags uint8
        [n_frames*2940][, info uint8 [n_frames, 16] (capi.PCM1_FRAME_INFO)])."""
        recs = _dev_u8(recs)
        samples = torch.empty(n_frames * 2 * 1470, dtype=torch.int16, device=recs.device)
        flags = torch.empty(n_frames * 2 * 1470, dtype=torch.uint8, device=recs.device)
        info = torch.empty((n_frames, capi.PCM1_FRAME_INFO.itemsize), dtype=torch.uint8, device=recs.device) if want_info else None
        cfg = capi.Pcm1StitchConfig(ignore_crc=int(self.ignore_crc), bff=int(self.field_order == self.ORDER_BFF), file_start=int(file_start),
                                    manual_offset=int(not self.auto_offset), odd_offset=self.odd_offset, even_offset=self.even_offset)
        rc = capi.lib().sdv_pcm1_frames_to_samples(self.handle.ptr, C.byref(cfg), C.c_void_p(recs.data_ptr()), n_frames, height, C.c_void_p(samples.data_ptr()),
                                                   C.c_void_p(flags.data_ptr()), C.c_void_p(info.data_ptr()) if want_info else None,
                                                   _stream_ptr(stream))
        self.handle.check(rc)
        return (samples, flags, info) if want_info else (samples, flags)


class PCM16X0Deinterleaver:
    """PCM16X0Deinterleaver::processBlock (pcm16x0deinterleaver.cpp:128-912): SI format = the 35 data blocks of every
    105 sub-line interleave block; EI format = the 490 data blocks of every 1470 sub-line frame."""

    def __init__(self, handle: capi.Handle | None = None, device: int = 0):
        self.handle = handle or capi.Handle(device)
        self.ignore_crc, self.force_check, self.p_corr = False, True, True
        self.ei_format = False

    def setIgnoreCRC(self, f):
        self.ignore_crc = bool(f)

    def setForcedErrorCheck(self, f):
        self.force_check = bool(f)

    def setPCorrection(self, f):
        self.p_corr = bool(f)

    def setEIFormat(self, f=True):
        self.ei_format = bool(f)

    def setSIFormat(self):
        self.ei_format = False

    def processInterleaveBlocks(self, sublines: torch.Tensor, stream=None):
        """sublines: CUDA uint8 [n_units*105, 8] (SI) or [n_units*1470, 8] (EI) (capi.PCM16X0_SUBLINE).  Returns (samples int16
        [n, 6], flags uint8 [n, 6], states uint8 [n, 3])."""
        sublines = _dev_u8(sublines)
        unit, per = (1470, 490) if self.ei_format else (105, 35)
        assert sublines.shape[0] % unit == 0 and sublines.shape[1] == capi.PCM16X0_SUBLINE.itemsize
        n_itl = sublines.shape[0] // unit
        nb = n_itl * per
        dev = sublines.device
        samples = torch.empty((nb, 6), dtype=torch.int16, device=dev)
        flags = torch.empty((nb, 6), dtype=torch.uint8, device=dev)
        states = torch.empty((nb, 3), dtype=torch.uint8, device=dev)
        cfg = capi.Pcm16x0Config(ignore_crc=int(self.ignore_crc), force_check=int(self.force_check), p_corr=int(self.p_corr),
                                 ei_format=int(self.ei_format))
        rc = capi.lib().sdv_deint_pcm16x0(self.handle.ptr, C.byref(cfg), C.c_void_p(sublines.data_ptr()), n_itl,
                                          C.c_void_p(samples.data_ptr()), C.c_void_p(flags.data_ptr()),
                                          C.c_void_p(states.data_ptr()), _stream_ptr(stream))
        self.handle.check(rc)
        return samples, flags, states


class PCM16X0DataStitcher:
    """PCM16X0DataStitcher::doFrameReassemble for the SI format with preset vertical alignment (trim, false-positive CRC
    prescan, padding to 245 lines per field, field order, deinterleave + P correction, broken-block masking)."""

    ORDER_TFF, ORDER_BFF = 1, 2
    FORMAT_SI, FORMAT_EI = 1, 2                 # PCM16X0Deinterleaver::FORMAT_* (pcm16x0deinterleaver.h:72-78)

    def __init__(self, handle: capi.Handle | None = None, device: int = 0):
        self.handle = handle or capi.Handle(device)
        self.ignore_crc = False
        self.p_corr = True
        self.field_order = self.ORDER_TFF
        self.top_padding = (5, 5)               # odd, even field: lines above the first captured data line
        self.broken_mask_dur = 81               # UNCH_MASK_DURATION
        self.ei_format = False

    def setFormat(self, fmt):
        """PCM16X0DataStitcher::setFormat (pcm16x0datastitcher.cpp:5456-5490): FORMAT_SI or FORMAT_EI; FORMAT_AUTO (0) is a TODO
        in the reference (pcm16x0deinterleaver.h:74) and refused here.  doFrameReassembleAuto searches the EI alignment as the
        reference does; doFrameReassemble takes the top paddings given and deinterleaves the frame as one EI unit."""
        if int(fmt) not in (self.FORMAT_SI, self.FORMAT_EI):
            raise ValueError("PCM-16x0 format must be FORMAT_SI (1) or FORMAT_EI (2)")
        self.ei_format = int(fmt) == self.FORMAT_EI

    def setIgnoreCRC(self, f):
        self.ignore_crc = bool(f)

    def setPCorrection(self, f):
        self.p_corr = bool(f)

    def setFieldOrder(self, order):
        self.field_order = self.ORDER_BFF if int(order) == self.ORDER_BFF else self.ORDER_TFF

    def doFrameReassembleAuto(self, recs, n_frames, height, **kw):
        """The reference's own vertical alignment (findSIDataAlignment / findEIFrameStitching) instead of setTopPadding: see
        pcm16x0_reassemble_auto."""
        return pcm16x0_reassemble_auto(self, recs, n_frames, height, **kw)

    def setTopPadding(self, odd, even):
        self.top_padding = (int(odd), int(even))

    def setFineBrokeMask(self, n):
        if not 0 <= int(n) <= 255:
            raise ValueError("broken-block mask duration must be 0..255 (uint8_t broken_mask_dur, pcm16x0datastitcher.h)")
        self.broken_mask_dur = int(n)

    def doFrameReassemble(self, recs: torch.Tensor, n_frames: int, height: int, stream=None, mask_seams: torch.Tensor | None = None,
                          want_info: bool = False, continue_file: bool = False):
        """recs: the PCM-16x0 sub-line records of VideoToDigital.doBinarize; mask_seams: optional CUDA uint8 [n_frames], non-zero
        where the padding search was unsure about the frame.  Returns (samples int16 [n_frames*490, 6],
        flags uint8 [n_frames*490, 6]); with want_info also the control-bit decisions per frame (capi.PCM16X0_FRAME_INFO:
        sample rate, emphasis, code as the reference writes them into the frame's sample pairs).  continue_file: the frames
        continue those of the previous stitch call on the handle, whose control-bit votes then count for these."""
        recs = _dev_u8(recs)
        samples = torch.empty((n_frames * 490, 6), dtype=torch.int16, device=recs.device)
        flags = torch.empty((n_frames * 490, 6), dtype=torch.uint8, device=recs.device)
        cfg = capi.Pcm16x0Config(ignore_crc=int(self.ignore_crc), force_check=int(not self.ignore_crc), p_corr=int(self.p_corr),
                                 ei_format=int(self.ei_format), continue_file=int(continue_file))
        geo = capi.Pcm16x0Geometry(bff=int(self.field_order == self.ORDER_BFF), top_padding_odd=self.top_padding[0],
                                   top_padding_even=self.top_padding[1], broken_mask_dur=self.broken_mask_dur)
        info = torch.zeros((n_frames, capi.PCM16X0_FRAME_INFO.itemsize), dtype=torch.uint8, device=recs.device) if want_info else None
        rc = capi.lib().sdv_pcm16x0_frames_to_samples_info(self.handle.ptr, C.byref(cfg), C.byref(geo), C.c_void_p(recs.data_ptr()),
                                                           n_frames, height, C.c_void_p(mask_seams.data_ptr()) if mask_seams is not None else None,
                                                           C.c_void_p(samples.data_ptr()), C.c_void_p(flags.data_ptr()),
                                                           C.c_void_p(info.data_ptr()) if want_info else None, _stream_ptr(stream))
        self.handle.check(rc)
        if want_info:
            return samples, flags, info.cpu().numpy().reshape(-1).view(capi.PCM16X0_FRAME_INFO)
        return samples, flags


def pcm16x0_reassemble_auto(stitcher, recs: torch.Tensor, n_frames: int, height: int, stream=None, want_info: bool = False,
                            file_start: bool = True, mask_seams: bool = True, continue_file: bool = False):
    """PCM16X0DataStitcher::doFrameReassemble with the vertical alignment searched as the reference does
    (sdv_pcm16x0_frames_to_samples_auto): findSIDataAlignment, or findEIFrameStitching after stitcher.setFormat(FORMAT_EI).
    file_start=False keeps the padding history of the previous call; continue_file=True (with file_start=False) also its
    control-bit history, so a tape stitched in batches gives the output of one call.
    Returns (samples int16 [n_frames*490, 6], flags uint8 [n_frames*490, 6], alignment capi.PCM16X0_ALIGNMENT [n_frames][, info])."""
    recs = _dev_u8(recs)
    dev = recs.device
    samples = torch.empty((n_frames * 490, 6), dtype=torch.int16, device=dev)
    flags = torch.empty((n_frames * 490, 6), dtype=torch.uint8, device=dev)
    info = torch.empty((n_frames, capi.PCM16X0_FRAME_INFO.itemsize), dtype=torch.uint8, device=dev) if want_info else None
    align = np.zeros(max(n_frames, 1), capi.PCM16X0_ALIGNMENT)
    cfg = capi.Pcm16x0Config(ignore_crc=int(stitcher.ignore_crc), force_check=int(not stitcher.ignore_crc), p_corr=int(stitcher.p_corr),
                             ei_format=int(getattr(stitcher, "ei_format", False)), continue_file=int(continue_file))
    geo = capi.Pcm16x0Geometry(bff=int(stitcher.field_order == stitcher.ORDER_BFF), top_padding_odd=0, top_padding_even=0,
                               broken_mask_dur=int(stitcher.broken_mask_dur))
    rc = capi.lib().sdv_pcm16x0_frames_to_samples_auto(stitcher.handle.ptr, C.byref(cfg), C.byref(geo), C.c_void_p(recs.data_ptr()), n_frames, height,
                                                       int(file_start), int(mask_seams), C.c_void_p(samples.data_ptr()), C.c_void_p(flags.data_ptr()),
                                                       C.c_void_p(info.data_ptr()) if want_info else None, align.ctypes.data_as(C.c_void_p),
                                                       _stream_ptr(stream))
    stitcher.handle.check(rc)
    return (samples, flags, align[:n_frames], info) if want_info else (samples, flags, align[:n_frames])


class STC007DataStitcher(_DeintSettings):
    """Frame assembly with preset geometry + deinterleave + sample output
    (STC007DataStitcher::fillFrameForOutput / performDeinterleave / outputSamplePair, stc007datastitcher.cpp:4588-5388,6525-6885)."""

    def __init__(self, handle: capi.Handle | None = None, device: int = 0):
        super().__init__()
        self.handle = handle or capi.Handle(device)
        self.video_std = VID_PAL
        self.broken_mask_dur = 128          # stc007datastitcher.cpp:6894-7236 default
        self.lead_in = LEAD_IN_LINES

    def setVideoStandard(self, std):
        self.video_std = int(std)

    def setFieldOrder(self, order):
        """FrameAsmDescriptor::ORDER_*: 0 detect, 1 TFF, 2 BFF (used by the automatic alignment, doFrameReassembleAuto)."""
        self.field_order = int(order)

    def setResolutionPreset(self, bits16: bool | None):
        """STC007DataStitcher::setResolutionPreset: False = SAMPLE_RES_14BIT, True = SAMPLE_RES_16BIT, None = SAMPLE_RES_UNKNOWN
        (the resolution is detected per field; doFrameReassembleAuto only)."""
        self.res_auto = bits16 is None
        self.res_mode = RES_MODE_16BIT if bits16 else RES_MODE_14BIT

    def setFineMaskSeams(self, f):
        self.mask_seams = bool(f)

    def setFineTopLineFix(self, f):
        self.fix_cut_above = bool(f)

    def setFineMaxUnch14(self, n):
        self.max_unch14 = int(n) & 0xFF

    def setFineMaxUnch16(self, n):
        self.max_unch16 = int(n) & 0xFF

    def setFineBrokeMask(self, n):
        self.setBrokenMaskDuration(n)

    def setBrokenMaskDuration(self, n):
        if not 0 <= int(n) <= 255:
            raise ValueError("broken-block mask duration must be 0..255 (uint8_t broken_mask_dur, stc007datastitcher.h)")
        self.broken_mask_dur = int(n)

    def countdown(self, stream=None) -> dict:
        """Broken-block countdown state of the last deinterleave call on the handle (sdv_stc007_countdown)."""
        c = capi.Countdown()
        self.handle.check(capi.lib().sdv_stc007_countdown(self.handle.ptr, C.byref(c), _stream_ptr(stream)))
        return {"countdown_in": c.countdown_in, "countdown_out": c.countdown_out, "depends_on_in": bool(c.depends_on_in), "windows": c.windows}

    def countdown_to(self, state: torch.Tensor, stream=None):
        """Countdown state of the last deinterleave call as int32 [countdown_in, countdown_out, windows, depends_on_in] copied into
        the CUDA tensor [state] on the stream, without a host synchronisation (sdv_stc007_countdown_copy)."""
        assert state.is_cuda and state.dtype == torch.int32 and state.numel() >= 4
        self.handle.check(capi.lib().sdv_stc007_countdown_copy(self.handle.ptr, C.c_void_p(state.data_ptr()), _stream_ptr(stream)))
        return state

    def doFrameReassembleAuto(self, recs: torch.Tensor, n_frames: int, height: int, want_blocks: bool = False, stream=None,
                              file_start: bool = True, file_end: bool = True, video_std: int | None = None):
        """STC007DataStitcher::doFrameReassemble with the reference's own trim / padding / field-order decisions
        (sdv_stc007_stitch_frames).  video_std: 0 detect, 1 PAL, 2 NTSC (default: the preset of setVideoStandard).
        Returns (blocks | None, samples int16 [nb, 6], flags uint8 [nb, 6], info capi.STC007_FRAME_INFO [frames consumed])."""
        recs = _dev_u8(recs)
        cap = int(capi.lib().sdv_stc007_stitch_block_bound(n_frames))
        dev = recs.device
        blocks = torch.empty((cap, BLOCK_REC.itemsize), dtype=torch.uint8, device=dev) if want_blocks else None
        samples = torch.empty((cap, 6), dtype=torch.int16, device=dev)
        flags = torch.empty((cap, 6), dtype=torch.uint8, device=dev)
        info = np.zeros(max(n_frames, 1), capi.STC007_FRAME_INFO)
        std = {VID_PAL: 1, VID_NTSC: 2}.get(self.video_std, 0) if video_std is None else int(video_std)
        scfg = capi.StitchConfig(video_std=std, field_order=getattr(self, "field_order", 1),
                                 resolution_16bit=2 if getattr(self, "res_auto", False) else int(self.res_mode in (RES_MODE_16BIT, capi.RES_MODE_16BIT_AUTO)),
                                 file_start=int(file_start), file_end=int(file_end), mask_seams=int(getattr(self, "mask_seams", True)),
                                 fix_cut_above=int(getattr(self, "fix_cut_above", False)),
                                 max_unchecked_14bit=getattr(self, "max_unch14", 0x40), max_unchecked_16bit=getattr(self, "max_unch16", 0x20))
        cfg = self._cfg(cwd=getattr(self, "cwd", False))
        nb, nd = C.c_int(0), C.c_int(0)
        rc = capi.lib().sdv_stc007_stitch_frames(self.handle.ptr, C.byref(cfg), C.byref(scfg), C.c_void_p(recs.data_ptr()), n_frames, height,
                                                 C.c_void_p(blocks.data_ptr()) if want_blocks else None, C.c_void_p(samples.data_ptr()),
                                                 C.c_void_p(flags.data_ptr()), C.byref(nb), C.byref(nd), info.ctypes.data_as(C.c_void_p),
                                                 _stream_ptr(stream))
        self.handle.check(rc)
        return (blocks[:nb.value] if want_blocks else None), samples[:nb.value], flags[:nb.value], info[:nd.value]

    def saveState(self, out: torch.Tensor | None = None, stream=None) -> torch.Tensor:
        """The open file a doFrameReassembleAuto(file_end=False) call left on the handle, as a canonical uint8 CUDA tensor of
        sdv_stc007_stitch_state_bytes() bytes (sdv_stc007_stitch_state_save): equal states give equal bytes.  No synchronisation."""
        n = int(capi.lib().sdv_stc007_stitch_state_bytes())
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=torch.device("cuda", self.handle.device))
        out = _dev_u8(out)
        assert out.numel() == n
        self.handle.check(capi.lib().sdv_stc007_stitch_state_save(self.handle.ptr, C.c_void_p(out.data_ptr()), _stream_ptr(stream)))
        return out

    def loadState(self, state: torch.Tensor, stream=None):
        """Make [state] (from saveState, on any handle) the open file of this handle: the next doFrameReassembleAuto(file_start=False)
        continues it, with the CWD and resolution-detection settings it was saved with (sdv_stc007_stitch_state_load)."""
        state = _dev_u8(state)
        assert state.numel() == int(capi.lib().sdv_stc007_stitch_state_bytes())
        self.handle.check(capi.lib().sdv_stc007_stitch_state_load(self.handle.ptr, C.c_void_p(state.data_ptr()), _stream_ptr(stream)))

    def geometry(self) -> Geometry:
        return Geometry(lines_per_field=LINES_PER_FIELD[self.video_std], lead_in=self.lead_in)

    def block_count(self, n_frames: int) -> int:
        g = self.geometry()
        return int(capi.lib().sdv_stc007_block_count(C.byref(g), n_frames))

    def findPadding(self, recs: torch.Tensor, seams: np.ndarray, video_std: int | None = None, resolution_16bit: bool = False,
                    max_unchecked_14bit: int = 0x40, max_unchecked_16bit: int = 0x20, stream=None) -> np.ndarray:
        """STC007DataStitcher::findPadding (stc007datastitcher.cpp:1743-2054) for every seam: the padding sweep on the
        device, the reference's ranking and acceptance rules in the library.  Returns capi.PADDING [n_seams]
        (padding, DS_RET_* result, last_pad_counter)."""
        recs = _dev_u8(recs)
        seams = np.ascontiguousarray(seams, dtype=capi.SEAM)
        out = np.zeros(len(seams), dtype=capi.PADDING)
        cfg = self._cfg()
        std = self.video_std if video_std is None else video_std
        rc = capi.lib().sdv_stc007_find_padding(self.handle.ptr, C.byref(cfg), {VID_PAL: 1, VID_NTSC: 2}.get(std, 0), int(bool(resolution_16bit)),
                                                max_unchecked_14bit, max_unchecked_16bit, C.c_void_p(recs.data_ptr()),
                                                seams.ctypes.data_as(C.c_void_p), len(seams), out.ctypes.data_as(C.c_void_p), _stream_ptr(stream))
        self.handle.check(rc)
        return out

    def tryPadding(self, recs: torch.Tensor, seams: np.ndarray, n_paddings: int = 32, max_unchecked_14bit: int = 0x40,
                   max_unchecked_16bit: int = 0x20, stream=None) -> np.ndarray:
        """STC007DataStitcher::tryPadding (stc007datastitcher.cpp:1417-1740) for paddings 0..n_paddings-1 of every seam.
        recs: CUDA uint8 [n, 32] line records; seams: capi.SEAM array (ranges of recs).  Returns capi.STITCH_STATS [n_seams, n_paddings]."""
        recs = _dev_u8(recs)
        seams = np.ascontiguousarray(seams, dtype=capi.SEAM)
        sd = torch.from_numpy(seams.view(np.uint8).reshape(-1, capi.SEAM.itemsize).copy()).to(recs.device)
        out = torch.empty((len(seams) * n_paddings, capi.STITCH_STATS.itemsize), dtype=torch.uint8, device=recs.device)
        cfg = self._cfg()
        rc = capi.lib().sdv_stc007_try_padding(self.handle.ptr, C.byref(cfg), max_unchecked_14bit, max_unchecked_16bit,
                                               C.c_void_p(recs.data_ptr()), C.c_void_p(sd.data_ptr()), len(seams), n_paddings,
                                               C.c_void_p(out.data_ptr()), _stream_ptr(stream))
        self.handle.check(rc)
        return out.cpu().numpy().reshape(-1).view(capi.STITCH_STATS).reshape(len(seams), n_paddings)

    def fuseWithNextDecode(self, samples: torch.Tensor, flags: torch.Tensor, countdown_in: int = 0):
        """sdv_stc007_fuse_next_decode: the next VideoToDigital.doBinarize on this handle also finishes, inside its bulk pass, the
        data blocks that lie within one frame, into [samples] / [flags]; the following doFrameReassemble(..., samples=samples,
        flags=flags) with the same settings then only does what is left.  Results never depend on it."""
        assert samples.is_cuda and flags.is_cuda and samples.dtype == torch.int16 and flags.dtype == torch.uint8
        cfg, geo = self._cfg(countdown_in), self.geometry()
        self.handle.check(capi.lib().sdv_stc007_fuse_next_decode(self.handle.ptr, C.byref(cfg), C.byref(geo), C.c_void_p(samples.data_ptr()),
                                                                  C.c_void_p(flags.data_ptr())))

    def doFrameReassemble(self, recs: torch.Tensor, n_frames: int, height: int, want_blocks: bool = False, stream=None,
                          samples: torch.Tensor | None = None, flags: torch.Tensor | None = None,
                          halo: torch.Tensor | None = None, countdown_in: int = 0):
        """recs: CUDA uint8 [n_frames*height, 32] from VideoToDigital.doBinarize.  halo: the first 112 line records of
        the next shard of a frame-sharded tape (None on the last shard / unsharded tape).
        Returns (blocks | None, samples int16 [nb, 6], flags uint8 [nb, 6])."""
        recs = _dev_u8(recs)
        nb = self.block_count(n_frames)
        dev = recs.device
        blocks = torch.empty((nb, BLOCK_REC.itemsize), dtype=torch.uint8, device=dev) if want_blocks else None
        if samples is None:
            samples = torch.empty((nb, 6), dtype=torch.int16, device=dev)
        if flags is None:
            flags = torch.empty((nb, 6), dtype=torch.uint8, device=dev)
        assert samples.shape[0] >= nb and flags.shape[0] >= nb
        cfg, geo = self._cfg(countdown_in), self.geometry()
        rc = capi.lib().sdv_stc007_shard_to_samples(self.handle.ptr, C.byref(cfg), C.byref(geo), C.c_void_p(recs.data_ptr()),
                                                    n_frames, height, C.c_void_p(_dev_u8(halo).data_ptr()) if halo is not None else None,
                                                    C.c_void_p(blocks.data_ptr()) if want_blocks else None,
                                                    C.c_void_p(samples.data_ptr()), C.c_void_p(flags.data_ptr()), _stream_ptr(stream))
        self.handle.check(rc)
        return blocks, samples, flags


def decode_tape_host(handle: capi.Handle, luma: np.ndarray, mode: int = MODE_NORMAL, check_line_dup: bool = True,
                     video_std: int = VID_PAL, p_corr: bool = True, q_corr: bool = True, broken_mask_dur: int = 128,
                     want_flags: bool = True, want_recs: bool = False, samples_out: np.ndarray | None = None,
                     flags_out: np.ndarray | None = None):
    """The reference-facing whole-path call with HOST buffers (sdv_stc007_decode_tape_host): H2D, line decode,
    assembly, deinterleave + P/Q, D2H.  luma: uint8 [F, H, W] host array (pinned for best speed)."""
    assert luma.dtype == np.uint8 and luma.ndim == 3 and luma.flags.c_contiguous
    f, h, w = luma.shape
    geo = Geometry(lines_per_field=LINES_PER_FIELD[video_std], lead_in=LEAD_IN_LINES)
    nb = int(capi.lib().sdv_stc007_block_count(C.byref(geo), f))
    samples = samples_out if samples_out is not None else np.empty((nb, 6), dtype=np.int16)
    flags = (flags_out if flags_out is not None else np.empty((nb, 6), dtype=np.uint8)) if want_flags else None
    recs = np.empty(f * h, dtype=LINE_REC) if want_recs else None
    bcfg = BinConfig(pcm_type=TYPE_STC007, mode=mode, check_line_dup=int(check_line_dup))
    dcfg = DeintConfig(res_mode=RES_MODE_14BIT, ignore_crc=0, force_check=1, p_corr=int(p_corr), q_corr=int(q_corr),
                       broken_mask_dur=broken_mask_dur)
    rc = capi.lib().sdv_stc007_decode_tape_host(handle.ptr, C.byref(bcfg), C.byref(dcfg), C.byref(geo),
                                                luma.ctypes.data_as(C.c_void_p), f, h, w,
                                                samples.ctypes.data_as(C.c_void_p),
                                                flags.ctypes.data_as(C.c_void_p) if want_flags else None,
                                                recs.ctypes.data_as(C.c_void_p) if want_recs else None)
    handle.check(rc)
    return samples, flags, recs


def decode_tape_host_pcm1(handle: capi.Handle, luma: np.ndarray, mode: int = MODE_NORMAL, check_line_dup: bool = True,
                          bff: bool = False, ignore_crc: bool = False, offsets=None, want_recs: bool = False, continue_file: bool = False):
    """sdv_pcm1_decode_tape_host: PCM-1 host luma [F, H, W] -> (samples int16 [F*2940], flags uint8 [F*2940], recs).
    continue_file: the frames continue the file of the previous call on the handle (line decode and frame assembly)."""
    assert luma.dtype == np.uint8 and luma.ndim == 3 and luma.flags.c_contiguous
    f, h, w = luma.shape
    samples = np.empty(f * 2940, dtype=np.int16)
    flags = np.empty(f * 2940, dtype=np.uint8)
    recs = np.empty(f * h, dtype=LINE_REC) if want_recs else None
    bcfg = BinConfig(pcm_type=capi.TYPE_PCM1, mode=mode, check_line_dup=int(check_line_dup))
    bcfg.reserved[3] = int(continue_file)
    scfg = capi.Pcm1StitchConfig(ignore_crc=int(ignore_crc), bff=int(bff), file_start=int(not continue_file), manual_offset=int(offsets is not None),
                                 odd_offset=(offsets or (0, 0))[0], even_offset=(offsets or (0, 0))[1])
    rc = capi.lib().sdv_pcm1_decode_tape_host(handle.ptr, C.byref(bcfg), C.byref(scfg), luma.ctypes.data_as(C.c_void_p), f, h, w,
                                              samples.ctypes.data_as(C.c_void_p), flags.ctypes.data_as(C.c_void_p),
                                              recs.ctypes.data_as(C.c_void_p) if want_recs else None)
    handle.check(rc)
    return samples, flags, recs


def decode_tape_host_pcm16x0(handle: capi.Handle, luma: np.ndarray, mode: int = MODE_NORMAL, check_line_dup: bool = True,
                             bff: bool = False, ignore_crc: bool = False, p_corr: bool = True, top_padding=(5, 5),
                             broken_mask_dur: int = 81, want_recs: bool = False, continue_file: bool = False):
    """sdv_pcm16x0_decode_tape_host: PCM-16x0 (SI) host luma [F, H, W] -> (samples int16 [F*490, 6], flags uint8 [F*490, 6], recs).
    continue_file: the frames continue the file of the previous call on the handle (line decode and control-bit history)."""
    assert luma.dtype == np.uint8 and luma.ndim == 3 and luma.flags.c_contiguous
    f, h, w = luma.shape
    samples = np.empty((f * 490, 6), dtype=np.int16)
    flags = np.empty((f * 490, 6), dtype=np.uint8)
    recs = np.empty(f * h * 3, dtype=LINE_REC) if want_recs else None
    bcfg = BinConfig(pcm_type=capi.TYPE_PCM16X0, mode=mode, check_line_dup=int(check_line_dup))
    bcfg.reserved[3] = int(continue_file)
    dcfg = capi.Pcm16x0Config(ignore_crc=int(ignore_crc), force_check=int(not ignore_crc), p_corr=int(p_corr), continue_file=int(continue_file))
    geo = capi.Pcm16x0Geometry(bff=int(bff), top_padding_odd=top_padding[0], top_padding_even=top_padding[1], broken_mask_dur=broken_mask_dur)
    rc = capi.lib().sdv_pcm16x0_decode_tape_host(handle.ptr, C.byref(bcfg), C.byref(dcfg), C.byref(geo), luma.ctypes.data_as(C.c_void_p),
                                                 f, h, w, samples.ctypes.data_as(C.c_void_p), flags.ctypes.data_as(C.c_void_p),
                                                 recs.ctypes.data_as(C.c_void_p) if want_recs else None)
    handle.check(rc)
    return samples, flags, recs
