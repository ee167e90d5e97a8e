/* include/sdvpcm.h -- C ABI of the B200-native SDVPCM decode hot path (libsdvpcm_b200.so).
 *
 * This is the drop-in boundary for the per-frame decode path of Fagear/SDVPCMdecoder: what a maintainer binds
 * behind the reference's operator classes (see INTEGRATION.md).  Plain pointers and sizes only; every buffer is
 * caller-allocated; *_dev pointers are CUDA device memory, *_host pointers are host memory.  All entry points
 * return 0 on success or a negative SDV_ERR_* code; nothing throws across the boundary and there is NO CPU
 * fallback: without a CUDA device every compute call fails with SDV_ERR_CUDA.
 *
 * Reference interfaces replaced (file:line in the reference tree):
 *   sdv_bin_decode_frames      <- VideoToDigital::doBinarize per-frame loop body   videotodigital.cpp:825-1800
 *                                 = Binarizer::setSource/setOutput/setMode/.../processLine   binarizer.h:339-361,
 *                                   binarizer.cpp:443-1724, fed by the inter-line chain   videotodigital.cpp:1190-1522
 *   sdv_line_rec / sdv_line_aux<- STC007Line payload   stc007line.h:154-166, pcmline.h:132-160
 *   sdv_deint_stc007           <- STC007Deinterleaver::setInput/setOutput/setResMode/setIgnoreCRC/
 *                                 setForcedErrorCheck/setPCorrection/setQCorrection/processBlock
 *                                 stc007deinterleaver.h:159-173, stc007deinterleaver.cpp:286-1123
 *   sdv_block_rec              <- STC007DataBlock   stc007datablock.h:98-121
 *   sdv_stc007_frames_to_samples <- STC007DataStitcher::fillFrameForOutput (known paddings) + performDeinterleave +
 *                                 outputDataBlock/outputSamplePair   stc007datastitcher.cpp:4588-5388,6525-6627,6675-6885
 *   sdv_sample flags           <- PCMSample::{data_block_ok,word_valid,word_fixed}   pcmsamplepair.h:48-55
 */
#ifndef SDVPCM_H
#define SDVPCM_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDV_API __attribute__((visibility("default")))

/* ---- error codes */
enum { SDV_OK = 0, SDV_ERR_ARG = -1, SDV_ERR_CUDA = -2, SDV_ERR_UNSUPPORTED = -3, SDV_ERR_NOMEM = -4 };

/* ---- enumerations (values follow the reference) */
enum { SDV_TYPE_PCM1 = 0, SDV_TYPE_PCM16X0 = 1, SDV_TYPE_STC007 = 2, SDV_TYPE_M2 = 3 }; /* VideoToDigital::TYPE_* videotodigital.h:73-79
                                                                     (M2 = STC-007 lines with the M2 sample format) */
enum { SDV_MODE_DRAFT = 0, SDV_MODE_FAST = 1, SDV_MODE_NORMAL = 2, SDV_MODE_INSANE = 3 }; /* Binarizer::MODE_* binarizer.h:209-216 */
enum { SDV_SRV_NO = 0, SDV_SRV_HEADER_LINE = 6, SDV_SRV_CTRL_BLOCK = 7 };                /* PCMLine::SRVLINE_* pcmline.h:107-117 */
enum { SDV_RES_MODE_14BIT = 0, SDV_RES_MODE_14BIT_AUTO = 1, SDV_RES_MODE_16BIT_AUTO = 2, SDV_RES_MODE_16BIT = 3 };
                                                                                         /* STC007Deinterleaver::RES_MODE_* */
enum { SDV_AUD_ORIG = 0, SDV_AUD_FIX_P = 1, SDV_AUD_FIX_Q = 2, SDV_AUD_BROKEN = 3 };      /* STC007DataBlock::AUD_* */

/* ---- line record flags (sdv_line_rec.flags) */
enum
{
    SDV_LF_CRC_OK        = 1<<0,    /* PCMLine::isCRCValid()               (CRC matches and line not forced bad) */
    SDV_LF_CRC_OK_IGN    = 1<<1,    /* isCRCValidIgnoreForced()            */
    SDV_LF_FORCED_BAD    = 1<<2,    /* isForcedBad()                       */
    SDV_LF_BW_SET        = 1<<3,    /* hasBWSet()                          */
    SDV_LF_COORDS_SET    = 1<<4,    /* hasDataCoordSet()                   */
    SDV_LF_REF_SWEEP     = 1<<5,    /* isDataByRefSweep()                  */
    SDV_LF_BY_EXT        = 1<<6,    /* isDataBySkip()                      */
    SDV_LF_COORD_SWEEP   = 1<<7,    /* isDataByCoordSweep()  (PCM-1 / PCM-16x0: coordinates from the grid search) */
    SDV_LF_MARKERS       = 1<<8,    /* STC007Line::hasMarkers()            */
    SDV_LF_START_MARK    = 1<<9,
    SDV_LF_STOP_MARK     = 1<<10,
    SDV_LF_CONTROL_BIT   = 1<<11,   /* PCM16X0SubLine::control_bit         */
    SDV_LF_ALMOST_SILENT = 1<<12    /* isAlmostSilent()                    */
};

/* One decoded STC-007 line: 32 bytes, device resident.  Tier A = words + CRC flags; the rest is Tier B. */
typedef struct
{
    uint16_t words[9];          /* L R L R L R P Q (14-bit) + CRCC as read      stc007line.h:98-110 */
    uint16_t flags;             /* SDV_LF_* */
    uint8_t  ref, black, white, hyst;   /* ref_level, black_level, white_level, hysteresis_depth */
    int16_t  data_start, data_stop;     /* PCMLine::coords */
    uint8_t  shift;             /* shift_stage */
    uint8_t  service_type;      /* SDV_SRV_* */
    uint8_t  mark_stages;       /* mark_st_stage | mark_ed_stage<<4 */
    uint8_t  reserved;
} sdv_line_rec;

/* Optional Tier-B side record (16 bytes): fields the fast path can derive and only diagnostics need. */
typedef struct
{
    uint8_t  ref_low, ref_high;
    uint16_t marker_start_bg, marker_start_ed, marker_stop_ed;
    uint16_t word_crc_mask, word_valid_mask;    /* isWordCRCOk / isWordValid per word */
    uint8_t  pad[4];
} sdv_line_aux;

/* Binarizer fine settings   <- Binarizer::setFineSettings(bin_preset_t) / getDefaultFineSettings / getCurrentFineSettings
 * (binarizer.h:163-186,354-356; binarizer.cpp:48-65,394).  The nine numeric fields are honoured by every line decode path of
 * the handle (AGC limits, reference-level limits and sweep acceptance, marker search distance, bit-picker depth), and so is
 * en_coord_search (the PCM-1 / PCM-16x0 coordinate grid search) and en_first_line_dup (the first PCM line of a field forced bad
 * under the duplicate-line check, videotodigital.cpp:1199; with the switch off PCM-1 / PCM-16x0 frames all take the sequential
 * chain kernel); the other two switches and the forced coordinates are accepted at their default values only
 * (sdv_bin_set_fine_settings returns SDV_ERR_UNSUPPORTED otherwise: en_force_coords = 0, en_good_no_marker = 1). */
typedef struct
{
    uint8_t max_black_lvl;      /* 160  end point of the BLACK level search */
    uint8_t min_white_lvl;      /* 28   end point of the WHITE level search */
    uint8_t min_contrast;       /* 10   minimum WHITE - BLACK */
    uint8_t min_ref_lvl;        /* 7    lowest reference level */
    uint8_t max_ref_lvl;        /* 240  highest reference level */
    uint8_t min_valid_crcs;     /* 5    reference levels with the winning CRC a sweep needs */
    uint8_t mark_max_dist;      /* 6    percent of the line searched for START / STOP markers from either edge (STC-007) */
    uint8_t left_bit_pick;      /* 4    bits the bit picker may recover at the left edge (PCM-1 / PCM-16x0), at most 4 */
    uint8_t right_bit_pick;     /* 2    ... at the right edge, at most 2 */
    uint8_t en_force_coords, en_coord_search, en_first_line_dup, en_good_no_marker;     /* 0, 1, 1, 1 */
    uint8_t reserved;
    int16_t horiz_start, horiz_stop;    /* bin_preset_t::horiz_coords (used with en_force_coords only) */
    uint8_t reserved2[14];
} sdv_bin_preset;

/* Line decode configuration. */
typedef struct
{
    uint8_t pcm_type;           /* SDV_TYPE_STC007, SDV_TYPE_M2, SDV_TYPE_PCM1 or SDV_TYPE_PCM16X0 */
    uint8_t mode;               /* SDV_MODE_* */
    uint8_t check_line_dup;     /* VideoToDigital::setCheckLineDup */
    uint8_t reserved[13];       /* reserved[0] | reserved[1]<<8 = chain_segments: 0/1 = the tape is one file (the reference's
                                   semantics); S > 1 = decode it as S independent files of n_frames/S frames each, in parallel
                                   (each segment equals the reference run on that piece; for heavily damaged tapes)
                                   reserved[2] bit 0 = 1: no warm start (do not launch the bulk pass speculatively with the
                                   presets the previous call on this handle ended with; scheduling only, results are identical)
                                   reserved[2] bit 1 = 1: lazy verification (STC-007 / M2, not with reserved[3]): when the warm start hits, the call
                                   returns without waiting for the bulk pass to confirm that it took every frame; whatever uses the records
                                   may be enqueued behind it right away; sdv_bin_decode_verify() must be called before the next decode on
                                   the handle and before the results are relied on (it decodes the tape again if a frame was not clean)
                                   reserved[2] bit 2 = 1: no relay mode (a tape whose chain does not settle within 64 frames is decoded by many
                                   chains at once, each verified to have started from the true chain state; scheduling only, results are
                                   identical to the single sequential chain)
                                   reserved[3] bit 0 = 1 (STC-007 / M2 / PCM-1 / PCM-16x0): the call CONTINUES the file of the previous call
                                   on this handle instead of opening a new one: the chain state (Binarizer presets fed back by
                                   setGoodParameters, the coordinate histories of the last 9 lines and 16 frames, videotodigital.cpp:
                                   707-710,1366-1522; for PCM-1 / PCM-16x0 also the prescan's reference level, and frame 0 is not the
                                   file's first: no NEW_FILE line in its prescan) carries over, so a tape fed in batches decodes exactly
                                   as in one call, records and aux.  STC-007 / M2 and PCM-1 / PCM-16x0 keep one open file each: a call of
                                   the one kind neither opens nor closes the other's.  Every call that does not continue opens a new file;
                                   a continuing call needs the PCM type, H, W, mode and check_line_dup of the open file, else it fails
                                   with SDV_ERR_ARG.  A call that fails while decoding and a change of the fine settings
                                   (sdv_bin_set_fine_settings) close the file; n_frames = 0 leaves it as it is.  PCM-1 / PCM-16x0: not
                                   with chain_segments > 1 (SDV_ERR_ARG) */
} sdv_bin_config;

/* One deinterleaved data block (32 bytes). */
typedef struct
{
    uint16_t words[8];          /* L0 R0 L1 R1 L2 R2 P0 Q0 after correction */
    uint8_t  line_crc;          /* isWordLineCRCOk bit mask */
    uint8_t  word_valid;        /* isWordValid bit mask */
    uint8_t  audio_state;       /* SDV_AUD_* */
    uint8_t  resolution;        /* 0 = 14 bit, 1 = 16 bit */
    uint8_t  flags;             /* bit0 isBlockValid, 1 isDataBroken, 2 fixed by P, 3 fixed by Q, 4 isSilent, 5 marked unsafe */
    uint8_t  reserved[11];
} sdv_block_rec;

typedef struct
{
    uint8_t res_mode;           /* SDV_RES_MODE_* (setResMode) */
    uint8_t ignore_crc;         /* setIgnoreCRC */
    uint8_t force_check;        /* setForcedErrorCheck */
    uint8_t p_corr, q_corr;     /* setPCorrection / setQCorrection */
    uint8_t broken_mask_dur;    /* STC007DataStitcher broken_mask_dur (default 128), used by sdv_stc007_frames_to_samples */
    uint8_t m2_format;          /* setM2SampleFormat: M2 range/sign expansion of the samples (stc007datablock.cpp:507-562) */
    uint8_t countdown_in;       /* STC007DataStitcher::broken_countdown (stc007datastitcher.cpp:79,6785-6863) as the blocks BEFORE this call
                                   left it: 0 at a file start; for the later shards of a frame-sharded tape the countdown_out of the
                                   shard before (sdv_stc007_countdown) */
    uint8_t cwd;                /* STC007DataStitcher::setCWDCorrection (the reference's default is ON): Cross-Word Decoding, performCWD
                                   (stc007datastitcher.cpp:5905-6398) over every queued frame until a pass repairs nothing more, then the
                                   deinterleaver with its CWD stage (stc007deinterleaver.cpp:638-712).  Honoured by sdv_stc007_stitch_frames
                                   (the path with the reference's own frame assembly, where the queue CWD works on exists); the
                                   preset-geometry entry points reject it */
    uint8_t reserved[7];
} sdv_deint_config;

/* Per-sample flags written next to the int16 samples. */
enum { SDV_SF_BLOCK_OK = 1<<0, SDV_SF_WORD_VALID = 1<<1, SDV_SF_WORD_FIXED = 1<<2 };

/* Fixed frame geometry for assembling decoded lines into the deinterleaver input (what
 * STC007DataStitcher::fillFrameForOutput produces once trim and paddings are known). */
typedef struct
{
    uint16_t lines_per_field;   /* 294 (PAL) / 245 (NTSC): config.h:80-81 */
    uint16_t lead_in;           /* empty lines queued at file start: 80 (STC007DataBlock::LINE_R2, stc007datastitcher.cpp:4733) */
    uint16_t reserved[6];
} sdv_stc007_geometry;

typedef struct sdv_handle sdv_handle;

/* ---- lifetime */
SDV_API int  sdv_create(sdv_handle **out, int cuda_device);
SDV_API void sdv_destroy(sdv_handle *h);
SDV_API const char *sdv_last_error(sdv_handle *h);
SDV_API int  sdv_version(void);

/* ---- line decode operator (device buffers, stream ordered).
 * luma_dev: u8 [n_frames][H][stride] interlaced frames (odd field = rows 0,2,..; even field = rows 1,3,..).
 * recs_dev: [n_frames*H] records in the reference's stream order (per frame: odd-field rows, then even-field rows).
 * aux_dev : optional (NULL to skip).  The chain state starts empty (as after NEW_FILE) on every call unless the configuration
 *   asks to continue the previous call's file (reserved[3]).
 * PCM-1 (PCM1Line): words[0..5] = L2 R2 L4 R4 L6 R6 (13 bit), words[6] = CRCC, mark_stages = picked_bits_left |
 *   picked_bits_right<<4, service_type SDV_SRV_HEADER_LINE for the header line.
 * PCM-16x0 (PCM16X0SubLine): THREE records per video line ([n_frames*H*3], parts left, middle, right): words[0..2] =
 *   R1P1L1 L2P2R2 R3P3L3, words[3] = CRCC, words[4] = queue_order, reserved = line_part, SDV_LF_CONTROL_BIT, mark_stages as
 *   for PCM-1. */
SDV_API int sdv_bin_decode_frames(sdv_handle *h, const sdv_bin_config *cfg, const uint8_t *luma_dev, int n_frames, int H, int W,
                                  int stride, sdv_line_rec *recs_dev, sdv_line_aux *aux_dev, void *cuda_stream);

/* ---- fine settings of the handle's Binarizer (see sdv_bin_preset).  They stay until changed; a new handle has the defaults. */
SDV_API int sdv_bin_default_fine_settings(sdv_bin_preset *out);
SDV_API int sdv_bin_get_fine_settings(sdv_handle *h, sdv_bin_preset *out);
SDV_API int sdv_bin_set_fine_settings(sdv_handle *h, const sdv_bin_preset *in);

/* ---- the answer to a lazy decode call (sdv_bin_config.reserved[2] bit 1): waits for the bulk pass of that call; *redone = 0: its
 * records stand; *redone = 1: a frame was not clean, the tape has been decoded again into the same buffers (which therefore must
 * still be the caller's) and everything computed from the records since has to be computed again.  No-op without a pending call. */
SDV_API int sdv_bin_decode_verify(sdv_handle *h, int *redone);

/* ---- the open file of the line decode as a portable blob of sdv_bin_chain_state_bytes() bytes in device memory (4-byte aligned),
 * so that a decode can be checkpointed and resumed on another handle or device, or split over frame shards with a verified
 * hand-off (sharding.decode_shard).  The blob is canonical: equal bytes mean that every later call decodes the same records and
 * aux.  Layout (little endian; chain_state.cuh CS_* / CSH_* / CSB_*):
 *   [0, 64)    header: magic "SDCS" (u32), version (u16), PCM type (u16), size (u32), H, W (u16), mode, duplicate-line check,
 *              M2 sample format (u8), then at 32 the handle's sdv_bin_preset fine settings, verbatim;
 *   [64, 292)  the chain state at the frame boundary: the Binarizer presets (BinState), field state, duplicate check, M2 flag,
 *              the prescan's reference level (PCM-1 / PCM-16x0), the history counts, the words of the previous line, the frame
 *              average and the 9-line (PCM-16x0: 27 sub-line) and 16-frame coordinate histories;
 *   the rest zero, as are history entries past their counts.  Counters and PCM-16x0's running pair G of the bulk pass
 *   (scheduling only, derived from the history on load) are not part of it.
 * _save: the open file of [pcm_type]'s kind (STC-007 / M2: the one sdv_bin_decode_frames keeps for those two, PCM-1 / PCM-16x0:
 * the other) -> state_dev, one launch on the stream, no synchronisation.  _load: checks the blob on the host, then makes it the
 * open file of its kind on this handle, keyed by the blob's PCM type, H, W, mode and duplicate check: the next call with
 * sdv_bin_config.reserved[3] bit 0 and that key continues it exactly as the saved handle would have; synchronises the stream.
 * SDV_ERR_ARG: save without an open file of that kind; save or load while a lazy call awaits sdv_bin_decode_verify; load of a blob
 * with a wrong magic, version or size, an out-of-range field or bytes not in canonical form; load when the handle's fine
 * settings differ from the blob's. */
SDV_API int sdv_bin_chain_state_bytes(void);
SDV_API int sdv_bin_chain_state_save(sdv_handle *h, int pcm_type, void *state_dev, void *cuda_stream);
SDV_API int sdv_bin_chain_state_load(sdv_handle *h, const void *state_dev, void *cuda_stream);

/* ---- optional hook: [fn] is called from inside sdv_bin_decode_frames() (same thread) as soon as the records of the FIRST
 * frame are final -- on an STC-007 call with a warm handle that is while the bulk pass over the other frames is still
 * running on the device; on every other path it is called once before the function returns.  A frame-sharded decoder
 * starts sending its first 112 line records to the previous shard from here (VideoToDigital has no counterpart: the
 * reference's stitcher simply sees the lines in order).  Work the hook enqueues must not wait for [cuda_stream]'s later
 * work.  fn = NULL removes the hook. */
typedef void (*sdv_first_frame_fn)(void *user);
SDV_API int sdv_bin_on_first_frame(sdv_handle *h, sdv_first_frame_fn fn, void *user);

/* ---- deinterleave operator: one block per start line s in [0, n_lines-112) of the assembled line array.
 * blocks_dev / samples_dev ([n_blocks][6] int16) / sample_flags_dev ([n_blocks][6]) may each be NULL. */
SDV_API int sdv_deint_stc007(sdv_handle *h, const sdv_deint_config *cfg, const sdv_line_rec *asm_lines_dev, int n_lines,
                             sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev, void *cuda_stream);

/* ---- decoded frames -> samples with a known frame geometry (assembly fused into the deinterleave gather).
 * Block b (0 <= b < *n_blocks) starts at assembled line b; assembled stream = lead_in empty lines, then per field
 * its H/2 decoded lines followed by (lines_per_field - H/2) empty lines; 112 empty lines close the file.
 * n_blocks = lead_in + n_frames*2*lines_per_field. */
SDV_API int sdv_stc007_frames_to_samples(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_geometry *geo,
                                         const sdv_line_rec *recs_dev, int n_frames, int H,
                                         sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev,
                                         void *cuda_stream);
SDV_API int sdv_stc007_block_count(const sdv_stc007_geometry *geo, int n_frames);

/* ---- fused deinterleave: arms the handle so that the NEXT sdv_bin_decode_frames call (STC-007, at most 576 lines per frame) also
 * finishes -- inside its bulk pass, from the line words the decoding warp still holds on chip -- every data block whose eight
 * lines lie in one frame (2 x lines-per-field - 112 of the 2 x lines-per-field blocks that start in a frame), writing them where
 * the following sdv_stc007_frames_to_samples / sdv_stc007_shard_to_samples call with the SAME cfg, geo, record and output buffers
 * would; that call then only does the blocks that are left (those reaching into the next frame, the first frame, lead-in / halo /
 * tail) and the countdown windows.  Standard setting only (14 bit, forced parity check, P + Q, CRC respected, no M2, no CWD, no
 * block records): anything else, or a decode that did not come out of one clean bulk pass, silently leaves all the work to the
 * deinterleave call -- results are the same either way. */
SDV_API int sdv_stc007_fuse_next_decode(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_geometry *geo,
                                        int16_t *samples_dev, uint8_t *sample_flags_dev);

/* ---- the same for one shard of a frame-sharded tape (one GPU of several): halo_dev = the first 112 line records of the
 * NEXT shard (the cross-frame interleave span 7*16 lines, stc007datablock.h:44-58), NULL on the last shard; lead_in is
 * 80 on the first shard and 0 on the others.  Block counts and layouts as above. */
SDV_API int sdv_stc007_shard_to_samples(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_geometry *geo,
                                        const sdv_line_rec *recs_dev, int n_frames, int H, const sdv_line_rec *halo_dev,
                                        sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev,
                                        void *cuda_stream);

/* ---- the broken-block countdown of the LAST deinterleave call on this handle (sdv_deint_stc007, sdv_stc007_frames_to_samples,
 * sdv_stc007_shard_to_samples, sdv_stc007_stitch_frames): the reference's stitcher keeps its countdown from frame to frame
 * (broken_countdown is a member, stc007datastitcher.cpp:79), so a BROKEN block near the end of one call / shard masks up to
 * broken_mask_dur blocks of the next.  countdown_out goes into the next call's sdv_deint_config.countdown_in.
 * depends_on_in = 1: a BROKEN block lies within the first broken_mask_dur blocks, i.e. countdown_out was computed with
 * countdown_in and a different countdown_in may change it (a sharded decoder that ran the shards concurrently with
 * countdown_in = 0 has to redo only the shards for which the shard before reports countdown_out > 0).  Synchronises the stream. */
typedef struct { uint8_t countdown_in, countdown_out, depends_on_in, reserved; uint32_t windows; } sdv_countdown;
SDV_API int sdv_stc007_countdown(sdv_handle *h, sdv_countdown *out, void *cuda_stream);
/* The same four numbers as int32 {countdown_in, countdown_out, windows, depends_on_in} copied device to device on the stream
 * (no synchronisation): for a sharded decoder that gathers them over NCCL straight from device memory. */
SDV_API int sdv_stc007_countdown_copy(sdv_handle *h, int32_t *state_dev, void *cuda_stream);

/* ---- decoded frames -> samples with the reference's OWN vertical alignment   <- STC007DataStitcher::doFrameReassemble
 * (stc007datastitcher.cpp:7250-7479) = findFramesTrim (259-734), splitFramesToFields (737-985), detectVideoStandard (2773-2925),
 * findFieldStitching (2929-4276: the previous frame's paddings re-tried with tryPadding, else findPadding for the seam
 * between the fields and the seam to the next frame, field order by trial when it is not preset), getAssemblyFieldOrder
 * (4278-4423), fillFrameForOutput (4588-5388), performDeinterleave (6675-6885: seam masking 6738-6771, broken-block
 * countdown 6778-6862) and outputDataBlock.  Trims, seam sweeps and the deinterleave pass are device work over all frames of
 * the call; the frame-to-frame decisions (a few bytes per frame, each depending on the frame before) are host code inside
 * the library.  The audio resolution is a preset (14 or 16 bit, setResolutionPreset) or detected per field; CWD as sdv_deint_config.cwd says
 * (prescanFrame 6401-6452: the frames CWD can touch at all -- those with a line it may patch -- are walked chain by chain on the device,
 * sdv_block_rec.flags bit 6 = isDataFixedByCWD).
 * recs_dev: the [n_frames*H] line records of sdv_bin_decode_frames.  The assembled stream is: 80 empty lines at a file
 * start, per frame what fillFrameForOutput queues (2 x lines-per-field lines: first field, inner padding, second field,
 * outer padding), 112 empty lines at a file end; block b starts at stream line b, *n_blocks_out = lines - 112 of them.
 * file_start = 0 continues the file of the previous call on this handle (its frame state, countdown and the last 112
 * queued lines are kept in the handle); file_end = 0 leaves the LAST frame of the call unprocessed, as the reference does
 * until it has seen the frame after it: pass it again as the first frame of the next call (*n_frames_done tells how many
 * frames were consumed).  Output buffers must hold sdv_stc007_stitch_block_bound(n_frames) blocks.  info_host (may be NULL):
 * one FrameAsmSTC007 summary per consumed frame.  Synchronises the stream. */
typedef struct
{
    uint8_t video_std;              /* setVideoStandard: 0 detect by line count / 1 PAL / 2 NTSC (FrameAsmDescriptor::VID_*) */
    uint8_t field_order;            /* setFieldOrder: 0 detect / 1 TFF / 2 BFF (FrameAsmDescriptor::ORDER_*) */
    uint8_t resolution_16bit;       /* setResolutionPreset: 0 = SAMPLE_RES_14BIT, 1 = SAMPLE_RES_16BIT (sdv_deint_config.res_mode must then be
                                       SDV_RES_MODE_14BIT / _16BIT), 2 = SAMPLE_RES_UNKNOWN: the resolution is detected per field as the reference
                                       does it (getFieldResolution 996-1195: every block of a field tried as 14- and as 16-bit data;
                                       detectAudioResolution 2207-2770 with its 65-entry history; the deinterleaver mode of every block and
                                       every seam from the fields it touches, getDataBlockResolution 1272-1414) and res_mode is not used */
    uint8_t file_start, file_end;
    uint8_t mask_seams;             /* setFineMaskSeams (default on) */
    uint8_t fix_cut_above;          /* setFineTopLineFix (default off) */
    uint8_t max_unchecked_14bit, max_unchecked_16bit;   /* setFineMaxUnch14 / 16 (defaults 0x40 / 0x20) */
    uint8_t reserved[7];
} sdv_stc007_stitch_config;
typedef struct
{
    int32_t  start;                 /* stream line of the frame's first line */
    uint16_t pre, n1, inner, n2, outer;     /* empty lines in front, lines of field 1, inner padding, lines of field 2, outer padding */
    uint16_t skip1, skip2;          /* lines of the trimmed fields left out at their top */
    uint16_t odd_top, odd_bottom, even_top, even_bottom;    /* findFramesTrim: first / last line number with data */
    uint16_t odd_data_lines, even_data_lines, odd_valid_lines, even_valid_lines;
    uint16_t inner_padding, outer_padding;  /* as FrameAsmSTC007 keeps them after fillFrameForOutput */
    uint8_t  field_order, video_std;
    uint8_t  flags;                 /* SDV_FA_* */
    uint8_t  odd_res_mode, even_res_mode;   /* FrameAsmSTC007::odd_resolution / even_resolution: SDV_RES_MODE_* of the two fields */
    uint8_t  reserved;
} sdv_stc007_frame_info;
enum { SDV_FA_INNER_OK = 1, SDV_FA_OUTER_OK = 2, SDV_FA_INNER_SILENCE = 4, SDV_FA_OUTER_SILENCE = 8, SDV_FA_ORDER_GUESSED = 16,
       SDV_FA_MASK_INNER = 32, SDV_FA_MASK_PREV_OUTER = 64 };
SDV_API int sdv_stc007_stitch_block_bound(int n_frames);
SDV_API int sdv_stc007_stitch_frames(sdv_handle *h, const sdv_deint_config *cfg, const sdv_stc007_stitch_config *scfg,
                                     const sdv_line_rec *recs_dev, int n_frames, int H,
                                     sdv_block_rec *blocks_dev, int16_t *samples_dev, uint8_t *sample_flags_dev,
                                     int *n_blocks_out, int *n_frames_done, sdv_stc007_frame_info *info_host, void *cuda_stream);

/* ---- the open file of sdv_stc007_stitch_frames as a portable blob of sdv_stc007_stitch_state_bytes() bytes in device memory
 * (4-byte aligned): the previous frame's state, the field-order and resolution histories, the broken-block countdown, the 112
 * queued lines with their CWD-patched copies, and whether CWD and resolution detection were on.  The form is canonical -- rings
 * rotated to position 0, frame numbers counted from the first frame after the state, unused bytes zero -- so two states with the
 * same future compare equal byte for byte.  _save: the handle's open file (a call with file_end = 0 left it; SDV_ERR_ARG without
 * one) -> state_dev, one launch on the stream, no synchronisation.  _load: state_dev -> the handle's open file, so the next call
 * may pass file_start = 0, on this handle or another one on any device; synchronises the stream.  A blob of another magic,
 * version or size fails with SDV_ERR_ARG, and so does a continuing call after a load whose sdv_deint_config.cwd or detected
 * resolution (resolution_16bit = 2) differs from the saved state's.  file_start = 1 still resets everything. */
SDV_API int sdv_stc007_stitch_state_bytes(void);
SDV_API int sdv_stc007_stitch_state_save(sdv_handle *h, void *state_dev, void *cuda_stream);
SDV_API int sdv_stc007_stitch_state_load(sdv_handle *h, const void *state_dev, void *cuda_stream);

/* ---- whole path with HOST buffers (what the reference-facing plugin calls): H2D luma, line decode, assembly,
 * deinterleave + P/Q, D2H samples.  samples_host [n_blocks][6] int16, flags_host [n_blocks][6] (may be NULL),
 * recs_host [n_frames*H] (may be NULL). */
SDV_API int sdv_stc007_decode_tape_host(sdv_handle *h, const sdv_bin_config *bcfg, const sdv_deint_config *dcfg,
                                        const sdv_stc007_geometry *geo, const uint8_t *luma_host, int n_frames, int H, int W,
                                        int16_t *samples_host, uint8_t *flags_host, sdv_line_rec *recs_host);

/* ---- field-seam padding sweep   <- STC007DataStitcher::tryPadding(field1, f1_size, field2, f2_size, padding, stats)
 * stc007datastitcher.cpp:1417-1740, evaluated for paddings 0..n_paddings-1 of every seam in one launch (what findPadding,
 * 1743-2054, asks for one padding at a time).  A seam = two fields given as ranges of the line record array (the
 * trimmed field line vectors of splitFramesToFields).  stats_dev [n_seams][n_paddings]: FieldStitchStats (frametrimset.h:
 * 97-114; sort them with its operator< on the host) + the DS_RET_* code.  max_unchecked_*: the stitcher's
 * max_unchecked_14b_blocks / max_unchecked_16b_blocks (defaults 0x40 / 0x20). */
typedef struct { uint32_t f1_first, f1_size, f2_first, f2_size; } sdv_seam;
typedef struct { uint16_t index, valid, silent, unchecked, broken; uint8_t result; uint8_t reserved; } sdv_stitch_stats;
enum { SDV_DS_RET_NO_DATA = 0, SDV_DS_RET_SILENCE = 1, SDV_DS_RET_BROKE = 2, SDV_DS_RET_NO_PAD = 3, SDV_DS_RET_OK = 4 };
/* ---- field-seam padding decision   <- STC007DataStitcher::findPadding(field1, f1_size, field2, f2_size, in_std,
 * in_resolution, &padding)   stc007datastitcher.cpp:1743-2054, for every seam of [seams_host] at once: one sweep launch
 * (16 or 32 paddings per seam), then the reference's ranking (FieldStitchStats::operator<, frametrimset.cpp:312-371) and
 * acceptance rules on the host.  video_std: 0 unknown / 1 PAL / 2 NTSC (FrameAsmDescriptor::VID_*, frametrimset.h);
 * resolution_16bit: in_resolution == STC007DataBlock::RES_16BIT.  out_host[s].padding = the accepted padding, or the
 * standard's default (lines per field - f1_size) when result != SDV_DS_RET_OK; last_pad_counter as the member of that
 * name.  Synchronises the stream. */
typedef struct { uint16_t padding; uint8_t result; uint8_t last_pad_counter; } sdv_padding;
SDV_API int sdv_stc007_find_padding(sdv_handle *h, const sdv_deint_config *cfg, int video_std, int resolution_16bit,
                                    int max_unchecked_14bit, int max_unchecked_16bit, const sdv_line_rec *recs_dev,
                                    const sdv_seam *seams_host, int n_seams, sdv_padding *out_host, void *cuda_stream);
SDV_API int sdv_stc007_try_padding(sdv_handle *h, const sdv_deint_config *cfg, int max_unchecked_14bit, int max_unchecked_16bit,
                                   const sdv_line_rec *recs_dev, const sdv_seam *seams_dev, int n_seams, int n_paddings,
                                   sdv_stitch_stats *stats_dev, void *cuda_stream);

/* ---- PCM-1 deinterleave operator   <- PCM1Deinterleaver::setInput/setOutput/setIgnoreCRC/processBlock(itl_block, 0)
 * pcm1deinterleaver.h:79-84, pcm1deinterleaver.cpp:69-278, for all 8 interleave blocks of n_fields fields.
 * sublines_dev: [n_fields*735] (PCM1SubLine payload, pcm1subline.h:78-90); a field = 245 lines x 3 sub-lines, already
 * padded to 735 by the caller (PCM1DataStitcher::fillFrameForOutput).  Output per field: 1470 words in block order
 * (7 x 184 + 182): samples_dev int16 [n_fields*1470] (13 -> 16 bit, pcm1datablock.cpp:309-345), sample_flags_dev
 * [n_fields*1470] (SDV_SF_BLOCK_OK | SDV_SF_WORD_VALID; may be NULL). */
typedef struct
{
    uint16_t left, right;       /* 13-bit words */
    uint8_t  flags;             /* SDV_P1F_* */
    uint8_t  reserved[3];
} sdv_pcm1_subline;
enum { SDV_P1F_CRC_OK = 1, SDV_P1F_BW_SET = 2, SDV_P1F_PICKED_LEFT = 4, SDV_P1F_PICKED_RIGHT = 8 };
SDV_API int sdv_deint_pcm1(sdv_handle *h, int ignore_crc, const sdv_pcm1_subline *sublines_dev, int n_fields,
                           int16_t *samples_dev, uint8_t *sample_flags_dev, void *cuda_stream);

/* ---- PCM-1: decoded frames -> samples   <- PCM1DataStitcher::doFrameReassemble (automatic or preset line offsets)
 * (findFrameTrim / splitFrameToFields / findFramePadding / fillFirst+SecondFieldForOutput / performDeinterleave,
 * pcm1datastitcher.cpp:202-1218,1382-1453).  recs_dev: the [n_frames*H] PCM-1 line records of sdv_bin_decode_frames.
 * Every frame gives two fields of 735 sub-lines (trimmed to the data lines, padded at the top, or at the bottom when the
 * header line precedes the data), fields in the preset order (bff = 0: odd field first), each deinterleaved into 1470
 * samples: samples_dev int16 [n_frames*2*1470], sample_flags_dev likewise (may be NULL), info_dev [n_frames] (may be NULL).
 * file_start != 0: frame 0 is the first frame of the file (the reference forgets its header/emphasis detection when it
 * resets its state on NEW_FILE, pcm1datastitcher.cpp:1671-1675); 0 for the later shards of a frame-sharded tape. */
typedef struct
{
    uint16_t odd_top, odd_bottom, even_top, even_bottom;    /* first / last data line of the field (index in the field) */
    uint16_t odd_data_lines, even_data_lines;
    uint8_t  header_present, emphasis_set;                  /* findFrameTrim: header line ahead of / behind the data */
    uint8_t  reserved[2];
} sdv_pcm1_frame_info;
typedef struct
{
    uint8_t ignore_crc;         /* setIgnoreCRC */
    uint8_t bff;                /* setFieldOrder: 0 = odd field first */
    uint8_t file_start;         /* frame 0 opens the file */
    uint8_t manual_offset;      /* setAutoLineOffset(false): use the two offsets below instead of the automatic alignment */
    int8_t  odd_offset, even_offset;    /* setOddLineOffset / setEvenLineOffset: > 0 skips lines at the top, < 0 pads */
    uint8_t reserved[2];
} sdv_pcm1_stitch_config;
SDV_API int sdv_pcm1_frames_to_samples(sdv_handle *h, const sdv_pcm1_stitch_config *cfg, const sdv_line_rec *recs_dev, int n_frames,
                                       int H, int16_t *samples_dev, uint8_t *sample_flags_dev, sdv_pcm1_frame_info *info_dev,
                                       void *cuda_stream);

/* ---- PCM-16x0 (SI format) deinterleave operator   <- PCM16X0Deinterleaver::setInput/setOutput/setIgnoreCRC/
 * setForcedErrorCheck/setPCorrection/setSIFormat/processBlock(line_sh, even_order)  pcm16x0deinterleaver.h:126-135,
 * pcm16x0deinterleaver.cpp:128-912, called as PCM16X0DataStitcher::performDeinterleave does (pcm16x0datastitcher.cpp:
 * 5204-5346): for each interleave block of 105 sub-lines, data block i = 0..34 from sub-lines i, i+35, i+70 with
 * even_order = (i odd).  sublines_dev [n_itl_blocks*105] (PCM16X0SubLine payload, pcm16x0subline.h:116-125, line-major:
 * line 0 LEFT, MIDDLE, RIGHT, line 1 LEFT ...).  Output per data block: samples_dev int16 [n][6] = (L,R) of sub-blocks
 * 1..3; sample_flags_dev [n][6] (SDV_SF_*, may be NULL); states_dev [n][3] PCM16X0DataBlock::AUD_* (may be NULL);
 * n = 35*n_itl_blocks. */
typedef struct
{
    uint16_t words[3];          /* WORD_R1P1L1, WORD_L2P2R2, WORD_R3P3L3 */
    uint8_t  flags;             /* SDV_X0F_* */
    uint8_t  picked_left;       /* picked_bits_left */
} sdv_pcm16x0_subline;
enum { SDV_X0F_CRC_OK = 1, SDV_X0F_HAS_DATA = 2 /* coordinates valid and black/white set */, SDV_X0F_CONTROL_BIT = 4 /* PCM16X0SubLine::control_bit */,
       SDV_X0F_PICKED_RIGHT = 8 };
typedef struct { uint8_t ignore_crc, force_check, p_corr, ei_format /* setEIFormat: units of 1470 sub-lines (one frame), 490 data
                 blocks from sub-lines i, i+490, i+980 (pcm16x0datablock.h:41,70-72); n_itl_blocks then counts frames */,
                 continue_file /* stitch calls: the control-bit history of the previous stitch call goes on (see _info) */,
                 reserved[3]; } sdv_pcm16x0_config;
SDV_API int sdv_deint_pcm16x0(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_subline *sublines_dev,
                              int n_itl_blocks, int16_t *samples_dev, uint8_t *sample_flags_dev, uint8_t *states_dev,
                              void *cuda_stream);

/* ---- PCM-16x0 (SI format): decoded frames -> samples with a PRESET vertical alignment   <- PCM16X0DataStitcher::
 * doFrameReassemble (pcm16x0datastitcher.cpp:5652-5858) = findFrameTrim, splitFrameToFields, prescanForFalsePosCRCs,
 * fillFrameForOutput, performDeinterleave (incl. the unsafe marking of the broken_mask_dur data blocks from a BROKEN one
 * on) and outputDataBlock; the top padding of each field, which the reference searches for (findSIDataAlignment), is
 * given by the caller.  recs_dev: the [n_frames*H*3] sub-line records of sdv_bin_decode_frames.  Per frame 490 data
 * blocks (2 fields x 7 interleave blocks x 35): samples_dev int16 [n_frames*490][6] = (L,R) of sub-blocks 1..3,
 * sample_flags_dev likewise (SDV_SF_*, may be NULL).  mask_seams_dev (may be NULL = never): one byte per frame, non-zero
 * where the caller's padding search was unsure (FrameAsmPCM16x0 padding_ok false on a non-silent frame): the data blocks of
 * that frame are marked unsafe until three fully valid ones have been seen (setFineMaskSeams, 5230-5246).
 * cfg->ei_format = 1: the same assembly, the frame deinterleaved as one EI unit (data block b from sub-lines b, b+490, b+980). */
typedef struct
{
    uint8_t bff;                /* 0: odd field first (TFF) */
    uint8_t top_padding_odd, top_padding_even;      /* lines of padding above the first data line (FrameAsmPCM16x0) */
    uint8_t broken_mask_dur;    /* setFineBrokeMask, default 81 (UNCH_MASK_DURATION) */
    uint8_t reserved[4];
} sdv_pcm16x0_geometry;
SDV_API int sdv_pcm16x0_frames_to_samples(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_geometry *geo,
                                          const sdv_line_rec *recs_dev, int n_frames, int H, const uint8_t *mask_seams_dev,
                                          int16_t *samples_dev, uint8_t *sample_flags_dev, void *cuda_stream);

/* ---- the same plus the control-bit decisions of every frame   <- PCM16X0DataStitcher::collectCtrlBitStats,
 * updateCtrlBitStats, getProbableSampleRate / EmphasesBit / CodeBit (pcm16x0datastitcher.cpp:4745-4913, 4126-4348) as
 * applied at the end of fillFrameForOutput (4711-4741): the control bits of lines 0..3 of the 14 interleave blocks of the
 * assembled frame (middle sub-lines with a valid CRC; bit 0 = active) are put to the vote; a frame with at least two votes
 * on emphasis, sample rate and code takes its own result, any other frame the majority of the last 65 frames.
 * sample_rate / emphasis / code are what the reference then writes into the frame's PCMSamplePairs and data blocks (f1_srate,
 * f1_emph, f1_code, before setSampleRatePreset overrides the rate) -- including its quirk that the fall-back values of
 * emphasis and code have the opposite sense of the voted ones (4169-4287).  The history starts empty on every call unless
 * cfg->continue_file = 1: then the votes of the last 64 frames of the previous PCM-16x0 stitch call on this handle (and of the
 * calls it continued) stand in front of frame 0, so a tape stitched in batches gets the decisions of one call.  Every stitch call
 * (sdv_pcm16x0_frames_to_samples, _info, _auto, with or without info) keeps its votes on the handle; continue_file without an
 * earlier stitch call, or after one in the other format (ei_format), fails with SDV_ERR_ARG. */
enum { SDV_X0I_VALID = 1, SDV_X0I_EMPHASIS = 2, SDV_X0I_44100 = 4, SDV_X0I_EI_FORMAT = 8, SDV_X0I_CODE = 16 };
typedef struct
{
    uint16_t sample_rate;       /* 44100 / 44056 */
    uint8_t  emphasis, code;
    uint8_t  frame_votes;       /* SDV_X0I_*: this frame's own vote (collectCtrlBitStats); VALID = isOrderEven() */
    uint8_t  reserved[3];
} sdv_pcm16x0_frame_info;
SDV_API int sdv_pcm16x0_frames_to_samples_info(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_geometry *geo,
                                               const sdv_line_rec *recs_dev, int n_frames, int H, const uint8_t *mask_seams_dev,
                                               int16_t *samples_dev, uint8_t *sample_flags_dev, sdv_pcm16x0_frame_info *info_dev,
                                               void *cuda_stream);

/* ---- the same with the vertical alignment searched as the reference does   <- PCM16X0DataStitcher::findSIDataAlignment
 * (pcm16x0datastitcher.cpp:2246-2377) = findSIPadding per field (1557-2245): trySIPadding (1129-1556) for the paddings 0..34,
 * the zeroed control bits (findZeroControlBitOffset, 868-1055), the interleave block the field starts in (estimateBlockNumber,
 * 1058-1126), the 65-field history of accepted paddings (getProbablePadding), cutFieldTop; a frame whose search is not sure
 * and not silent gets its first data blocks masked (setFineMaskSeams).  The per-field scan is device work, the decisions host
 * code inside the library.  geo's top paddings are ignored.  align_host (may be NULL): what was decided, per frame.
 * file_start = 0 keeps the padding history of the previous call on the handle; cfg->continue_file = 1 (with file_start = 0 only,
 * else SDV_ERR_ARG) also the control-bit history, as in _info.  Synchronises the stream.
 * cfg->ei_format = 1: the EI format   <- PCM16X0DataStitcher::findEIFrameStitching (3588-4117): the padding of the history
 * tried first, else findEIPadding (2649-2994: tryEIPadding, 2380-2646, for the 81 paddings between the two fields of the
 * frame), conditionEIFramePadding (2997-3464) or, without a padding, findEIDataAlignment per field (3467-3585); data block b
 * of the frame from sub-lines b, b+490, b+980 (performDeinterleave, 5181-5186).  For EI frames sdv_pcm16x0_alignment.result =
 * { DS_RET_* of the padding search, padding between the fields or 0xFF }.  A change of format between calls drops the history. */
typedef struct
{
    int16_t  top_padding[2], cut_lines[2], lines[2];    /* odd, even field: padding on top, lines dropped at the head, lines kept */
    uint8_t  result[2];                                 /* SDV_DS_RET_* of findSIPadding */
    uint8_t  mask_seams;                                /* !padding_ok && !silence */
    uint8_t  reserved;
} sdv_pcm16x0_alignment;
SDV_API int sdv_pcm16x0_frames_to_samples_auto(sdv_handle *h, const sdv_pcm16x0_config *cfg, const sdv_pcm16x0_geometry *geo,
                                               const sdv_line_rec *recs_dev, int n_frames, int H, int file_start, int mask_seams,
                                               int16_t *samples_dev, uint8_t *sample_flags_dev, sdv_pcm16x0_frame_info *info_dev,
                                               sdv_pcm16x0_alignment *align_host, void *cuda_stream);

/* ---- whole path with HOST buffers for PCM-1 and PCM-16x0 (SI), as sdv_stc007_decode_tape_host: H2D luma, line decode,
 * frame assembly, deinterleave, D2H.  samples_host int16 [n_frames*2*1470] (735 sample pairs per field, fields in output
 * order), flags_host likewise (may be NULL), recs_host [n_frames*H] / [n_frames*H*3] (may be NULL).  The configurations go to
 * the calls unchanged: a capture streams through in batches with bcfg->reserved[3] bit 0 set on every batch after the first,
 * and scfg->file_start = 0 / dcfg->continue_file = 1 there. */
SDV_API int sdv_pcm1_decode_tape_host(sdv_handle *h, const sdv_bin_config *bcfg, const sdv_pcm1_stitch_config *scfg,
                                      const uint8_t *luma_host, int n_frames, int H, int W, int16_t *samples_host,
                                      uint8_t *flags_host, sdv_line_rec *recs_host);
SDV_API int sdv_pcm16x0_decode_tape_host(sdv_handle *h, const sdv_bin_config *bcfg, const sdv_pcm16x0_config *dcfg,
                                         const sdv_pcm16x0_geometry *geo, const uint8_t *luma_host, int n_frames, int H, int W,
                                         int16_t *samples_host, uint8_t *flags_host, sdv_line_rec *recs_host);

/* ---- statistics of the last sdv_bin_decode_frames call (for tests and the bench's launch accounting) */
typedef struct
{
    uint64_t lines_total;
    uint64_t lines_fast;        /* decoded by the bulk speculative kernel and kept */
    uint64_t lines_chain;       /* (re)decoded by the sequential chain kernel */
    uint64_t frames_skipped;    /* frames the chain kernel skipped as neutral */
    uint32_t kernel_launches;
    uint32_t reserved;
} sdv_bin_stats;
SDV_API int sdv_bin_last_stats(sdv_handle *h, sdv_bin_stats *out);

/* ---- accumulated device time of the bulk line-decode launches and of the (first-pass) deinterleave launches since the
 * last reset, measured with CUDA events the library records on the caller's stream around each of those launches; blocks
 * until the last such launch has finished.  For roofline accounting. */
typedef struct
{
    float    bulk_ms, deint_ms;     /* sums over the launches */
    uint64_t bulk_lines;            /* video lines handed to the bulk launches */
    uint64_t deint_blocks;          /* data blocks produced by the deinterleave launches */
    uint32_t bulk_launches, deint_launches;
    uint32_t kernel_launches;       /* every kernel the library launched since the last reset */
    uint32_t reserved;
} sdv_timings;
SDV_API int sdv_timings_read(sdv_handle *h, sdv_timings *out, int reset);

#ifdef __cplusplus
}
#endif
#endif
