// chain_state.cuh -- the line-decode chain state of an open file as a blob (sdv_bin_chain_state_save / _load).
//
// What a decode call with sdv_bin_config.reserved[3] bit 0 reads from the handle: the chain context of the open STC-007 / M2
// file (ChainCtx) or of the open PCM-1 / PCM-16x0 file (P1ChainCtx / X0ChainCtx), at a frame boundary.  The blob is canonical:
// it holds exactly what decides the records and aux of every later frame -- for STC-007 what chain_state_equal() compares, for
// the PCM formats its counterparts plus the prescan's reference level -- in a fixed little-endian byte layout, history entries
// past their counts and every unused byte zero.  Two states with the same future therefore compare equal with memcmp.
// Counters, the per-frame lists (empty at a frame boundary) and the per-field / per-line counters (reset before they are read
// again) are left out; unpacking zeroes them.  PCM-16x0's running pair G (X0ChainCtx::run_g) is left out too: it only decides
// which frames the chain may take from the bulk pass (a frame is taken only when the whole coordinate history equals G, and then
// the bulk records are what the chain would decode), so unpacking derives it from the history.
#pragma once
#include "pcm16x0_chain.cuh"

namespace sdv {

enum { CS_MAGIC = 0x53434453u /* "SDCS" */, CS_VERSION = 1, CS_BYTES = 512, CS_HDR = 64 };
// Header (built on the host from the handle's key and fine settings).
enum { CSH_MAGIC = 0 /* u32 */, CSH_VERSION = 4 /* u16 */, CSH_TYPE = 6 /* u16 SDV_TYPE_* */, CSH_SIZE = 8 /* u32 */,
       CSH_H = 12 /* u16 */, CSH_W = 14 /* u16 */, CSH_MODE = 16 /* u8 */, CSH_DUP = 17 /* u8 duplicate-line check */,
       CSH_M2 = 18 /* u8 M2 sample format */, CSH_FINE = 32 /* sdv_bin_preset, 32 bytes, as sdv_bin_get_fine_settings gives it */ };
// Chain state (packed on the device).
enum { CSB_BIN = 64       /* BinState: def_black, def_white, def_ref, mode (u8), def_coord (2 x i16), max_hyst, max_shift (u8) */,
       CSB_FIELD = 76     /* field_state, line_dup, m2, prescan_ref (PCM-1 / PCM-16x0; 0 for STC-007) */,
       CSB_COUNTS = 80    /* n_last, n_long, n_fv, n_fi (i32; the last two are 0 at a frame boundary) */,
       CSB_WORDS = 96     /* last_words: STC-007 8, PCM-1 6, PCM-16x0 3 x 3 (u16, up to 9) */,
       CSB_AVG = 116      /* frame_avg (2 x i16) */,
       CSB_LAST = 120     /* last_valid: n_last of up to 27 pairs (PCM-16x0: 3 x 9) */,
       CSB_LONG = 228     /* long_valid: n_long of up to 16 pairs */,
       CSB_END = 292 };
enum { CS_KIND_STC = 0, CS_KIND_P1 = 1, CS_KIND_X0 = 2 };
static_assert(((int)CSB_LAST+4*COORD_HISTORY_DEPTH*3==(int)CSB_LONG)&&((int)CSB_LONG+4*COORD_LONG_HISTORY==(int)CSB_END)&&((int)CSB_END<=(int)CS_BYTES), "chain blob layout");
struct ChainBlobHdr { u32 w[CS_HDR/4]; };

SDV_HD void cs_put16(u8 *b, int at, u32 v) { b[at] = (u8)v; b[at+1] = (u8)(v>>8); }
SDV_HD void cs_put32(u8 *b, int at, u32 v) { cs_put16(b, at, v&0xFFFFu); cs_put16(b, at+2, v>>16); }
SDV_HD u32 cs_get16(const u8 *b, int at) { return (u32)b[at]|((u32)b[at+1]<<8); }
SDV_HD u32 cs_get32(const u8 *b, int at) { return cs_get16(b, at)|(cs_get16(b, at+2)<<16); }
SDV_HD void cs_put_coord(u8 *b, int at, Coord c) { cs_put16(b, at, (u16)c.start); cs_put16(b, at+2, (u16)c.stop); }
SDV_HD Coord cs_get_coord(const u8 *b, int at) { Coord c; c.start = (i16)(u16)cs_get16(b, at); c.stop = (i16)(u16)cs_get16(b, at+2); return c; }

// The part every format shares.  [b]: the whole blob, its body zero beforehand.
SDV_HD void cs_pack_common(u8 *b, const BinState &s, u8 field_state, u8 line_dup, u8 m2, u8 prescan_ref, const u16 *words, int n_words,
                           const Coord *last, int n_last, const Coord *lng, int n_long, Coord avg, int n_fv, int n_fi)
{
    b[CSB_BIN] = s.def_black; b[CSB_BIN+1] = s.def_white; b[CSB_BIN+2] = s.def_ref; b[CSB_BIN+3] = s.mode;
    cs_put_coord(b, CSB_BIN+4, s.def_coord); b[CSB_BIN+8] = s.max_hyst; b[CSB_BIN+9] = s.max_shift;
    b[CSB_FIELD] = field_state; b[CSB_FIELD+1] = line_dup; b[CSB_FIELD+2] = m2; b[CSB_FIELD+3] = prescan_ref;
    cs_put32(b, CSB_COUNTS, (u32)n_last); cs_put32(b, CSB_COUNTS+4, (u32)n_long); cs_put32(b, CSB_COUNTS+8, (u32)n_fv); cs_put32(b, CSB_COUNTS+12, (u32)n_fi);
    for(int i=0;i<n_words;i++) cs_put16(b, CSB_WORDS+2*i, words[i]);
    cs_put_coord(b, CSB_AVG, avg);
    for(int i=0;i<n_last;i++) cs_put_coord(b, CSB_LAST+4*i, last[i]);
    for(int i=0;i<n_long;i++) cs_put_coord(b, CSB_LONG+4*i, lng[i]);
}
// Its inverse; the counts are clamped to the capacities (a blob load checks them first, see cs_blob_kind).
SDV_HD void cs_unpack_common(const u8 *b, BinState *s, u8 *field_state, u8 *line_dup, u16 *words, int n_words, Coord *last, int cap_last,
                             int *n_last, Coord *lng, int *n_long, Coord *avg)
{
    s->def_black = b[CSB_BIN]; s->def_white = b[CSB_BIN+1]; s->def_ref = b[CSB_BIN+2]; s->mode = b[CSB_BIN+3];
    s->def_coord = cs_get_coord(b, CSB_BIN+4); s->max_hyst = b[CSB_BIN+8]; s->max_shift = b[CSB_BIN+9];
    *field_state = b[CSB_FIELD]; *line_dup = b[CSB_FIELD+1];
    const int nl = (int)cs_get32(b, CSB_COUNTS), ng = (int)cs_get32(b, CSB_COUNTS+4);
    const int n_l = (nl<0) ? 0 : ((nl>cap_last) ? cap_last : nl), n_g = (ng<0) ? 0 : ((ng>COORD_LONG_HISTORY) ? COORD_LONG_HISTORY : ng);
    *n_last = n_l; *n_long = n_g;
    for(int i=0;i<n_words;i++) words[i] = (u16)cs_get16(b, CSB_WORDS+2*i);
    *avg = cs_get_coord(b, CSB_AVG);
    for(int i=0;i<cap_last;i++) last[i] = (i<n_l) ? cs_get_coord(b, CSB_LAST+4*i) : coord_none();
    for(int i=0;i<COORD_LONG_HISTORY;i++) lng[i] = (i<n_g) ? cs_get_coord(b, CSB_LONG+4*i) : coord_none();
}

SDV_HD void cs_pack_stc(const ChainCtx *x, u8 *b)
{
    cs_pack_common(b, x->bin, x->field_state, x->line_dup, x->m2, 0, x->last_words, 8, x->last_valid, x->n_last, x->long_valid, x->n_long,
                   x->frame_avg, x->n_fv, x->n_fi);
}
SDV_HD void cs_pack_p1(const P1ChainCtx *x, u8 *b)
{
    cs_pack_common(b, x->bin, x->field_state, x->line_dup, 0, x->prescan_ref, x->last_words, 6, x->last_valid, x->n_last, x->long_valid, x->n_long,
                   x->frame_avg, x->n_fv, x->n_fi);
}
SDV_HD void cs_pack_x0(const X0ChainCtx *x, u8 *b)
{
    cs_pack_common(b, x->bin, x->field_state, x->line_dup, 0, x->prescan_ref, &x->last_words[0][0], 9, x->last_valid, x->n_last, x->long_valid,
                   x->n_long, x->frame_avg, x->n_fv, x->n_fi);
}

// Blob -> context at a frame boundary: the state the blob holds, counters and per-frame lists empty.
SDV_HD void cs_unpack_stc(const u8 *b, ChainCtx *x)
{
    cs_unpack_common(b, &x->bin, &x->field_state, &x->line_dup, x->last_words, 8, x->last_valid, COORD_HISTORY_DEPTH, &x->n_last,
                     x->long_valid, &x->n_long, &x->frame_avg);
    x->m2 = b[CSB_FIELD+2]; x->pad0 = 0;
    x->n_fv = x->n_fi = 0;
    x->next_frame = 0; x->stable = 0; x->first_unclean = 0; x->any_broken = 0;
    x->lines_chain = x->lines_chain_fast = x->lines_swept = 0;
}
SDV_HD void cs_unpack_p1(const u8 *b, P1ChainCtx *x)
{
    cs_unpack_common(b, &x->bin, &x->field_state, &x->line_dup, x->last_words, 6, x->last_valid, COORD_HISTORY_DEPTH, &x->n_last,
                     x->long_valid, &x->n_long, &x->frame_avg);
    x->prescan_ref = b[CSB_FIELD+3]; x->pad0 = 0;
    x->n_fv = x->n_fi = 0;
    x->good_in_field = x->pcm_in_field = 0;
    x->lines_chain = x->lines_search = 0;
}
// PCM-16x0: G from the history -- the pair the whole history holds in the steady state the bulk pass serves (so a clean tape
// stays on the bulk pass after a load), its median otherwise.
SDV_HD P1Preset cs_derive_run_g(const X0ChainCtx *x)
{
    P1Preset g;
    g.coords = (x->n_last>0) ? median_small(x->last_valid, x->n_last) : x->frame_avg;
    g.valid = coord_valid(g.coords) ? 1 : 0; g.ref = x->prescan_ref; g.pad[0] = g.pad[1] = 0;
    return g;
}
SDV_HD void cs_unpack_x0(const u8 *b, X0ChainCtx *x)
{
    cs_unpack_common(b, &x->bin, &x->field_state, &x->line_dup, &x->last_words[0][0], 9, x->last_valid, COORD_HISTORY_DEPTH*3, &x->n_last,
                     x->long_valid, &x->n_long, &x->frame_avg);
    x->prescan_ref = b[CSB_FIELD+3]; x->force_bad_line = 0;
    x->n_fv = x->n_fi = 0;
    x->good_in_field = x->pcm_in_field = x->line_in_field = 0;
    x->run_g = cs_derive_run_g(x);
}

// Is [b] a blob of this build whose chain state is in range (header fields, mode-derived Binarizer limits, counts, field
// state)?  The caller also checks that the body is canonical (unpack + pack gives the same bytes).  -> CS_KIND_* or -1.
SDV_HD int cs_blob_kind(const u8 *b)
{
    if((cs_get32(b, CSH_MAGIC)!=CS_MAGIC)||(cs_get16(b, CSH_VERSION)!=CS_VERSION)||(cs_get32(b, CSH_SIZE)!=CS_BYTES)) return -1;
    const int type = (int)cs_get16(b, CSH_TYPE), H = (int)cs_get16(b, CSH_H), W = (int)cs_get16(b, CSH_W);
    const int mode = b[CSH_MODE], dup = b[CSH_DUP], m2 = b[CSH_M2];
    if((H<2)||(H&1)||(H>SDV_MAX_H)||(W<BITS_IN_LINE)||(W>SDV_MAX_W)||(mode>SDV_MODE_INSANE)||(dup>1)||(m2>1)) return -1;
    for(int i=CSH_M2+1;i<CSH_FINE;i++) if(b[i]) return -1;
    int kind = -1;
    if(type==SDV_TYPE_STC007) kind = CS_KIND_STC;
    else if(type==SDV_TYPE_M2) kind = CS_KIND_STC;
    else if(type==SDV_TYPE_PCM1) kind = CS_KIND_P1;
    else if(type==SDV_TYPE_PCM16X0) kind = CS_KIND_X0;
    if((kind<0)||(m2!=((type==SDV_TYPE_M2) ? 1 : 0))) return -1;
    BinState ref; bin_set_mode(&ref, mode);
    if((b[CSB_BIN+3]!=ref.mode)||(b[CSB_BIN+8]!=ref.max_hyst)||(b[CSB_BIN+9]!=ref.max_shift)) return -1;
    if((b[CSB_FIELD]>FIELD_UNSAFE)||(b[CSB_FIELD+1]!=dup)||(b[CSB_FIELD+2]!=((kind==CS_KIND_STC) ? m2 : 0))) return -1;
    if((kind==CS_KIND_STC)&&(b[CSB_FIELD+3]!=0)) return -1;
    const int cap = (kind==CS_KIND_X0) ? COORD_HISTORY_DEPTH*3 : COORD_HISTORY_DEPTH;
    const int nl = (int)cs_get32(b, CSB_COUNTS), ng = (int)cs_get32(b, CSB_COUNTS+4);
    if((nl<0)||(nl>cap)||(ng<0)||(ng>COORD_LONG_HISTORY)||(cs_get32(b, CSB_COUNTS+8)!=0)||(cs_get32(b, CSB_COUNTS+12)!=0)) return -1;
    return kind;
}

#if defined(__CUDACC__)
// Header (by value) | the chain state packed from the device context [ctx] of kind [kind] -> blob, in one block.
__global__ void __launch_bounds__(128) chain_state_pack_kernel(ChainBlobHdr hdr, int kind, const void *ctx, u32 *blob)
{
    __shared__ u32 s[CS_BYTES/4];
    for(int i=threadIdx.x;i<CS_BYTES/4;i+=blockDim.x) s[i] = 0;
    __syncthreads();
    if(threadIdx.x==0)
    {
#pragma unroll
        for(int j=0;j<CS_HDR/4;j++) s[j] = hdr.w[j];
        u8 *b = (u8 *)s;
        if(kind==CS_KIND_STC) cs_pack_stc((const ChainCtx *)ctx, b);
        else if(kind==CS_KIND_P1) cs_pack_p1((const P1ChainCtx *)ctx, b);
        else cs_pack_x0((const X0ChainCtx *)ctx, b);
    }
    __syncthreads();
    for(int i=threadIdx.x;i<CS_BYTES/4;i+=blockDim.x) blob[i] = s[i];
}
// The chain state of a (checked) blob -> the device context [ctx] of kind KIND.  (One instance per kind: with the three bodies in
// one kernel ptxas puts a few registers on the stack.)
template<int KIND>
__global__ void __launch_bounds__(128) chain_state_unpack_kernel(const u32 *blob, void *ctx)
{
    __shared__ u32 s[CS_BYTES/4];
    for(int i=threadIdx.x;i<CS_BYTES/4;i+=blockDim.x) s[i] = blob[i];
    __syncthreads();
    if(threadIdx.x==0)
    {
        const u8 *b = (const u8 *)s;
        if(KIND==CS_KIND_STC) cs_unpack_stc(b, (ChainCtx *)ctx);
        else if(KIND==CS_KIND_P1) cs_unpack_p1(b, (P1ChainCtx *)ctx);
        else cs_unpack_x0(b, (X0ChainCtx *)ctx);
    }
}
#endif

}   // namespace sdv
