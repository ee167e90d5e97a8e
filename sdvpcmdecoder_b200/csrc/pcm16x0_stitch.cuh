// pcm16x0_stitch.cuh -- PCM16X0DataStitcher on the device: decoded sub-lines of one frame -> two fields of 735 sub-lines -> 490 data
// blocks (SI: 14 interleave blocks of 35; EI: one unit per frame) -> 1470 sample pairs, and the scans its padding searches decide over.
//
// Follows PCM16X0DataStitcher::doFrameReassemble (pcm16x0datastitcher.cpp:5652-5858): findFrameTrim (213-563: first/last line of
// each field with data -- black/white levels found, or a valid CRC once more than six interleave blocks' worth of lines (210) of
// the field are valid), splitFrameToFields (566-750), prescanForFalsePosCRCs (753-833: a line whose only valid part is a bit-picked
// outer part is forced bad), fillFrameForOutput (4594-4700: top padding, data, bottom padding to 245 lines, fields in the preset
// order), performDeinterleave (5165-5447: every data block through the deinterleaver, the blocks after a BROKEN one marked unsafe
// for broken_mask_dur blocks, PCM16X0DataBlock::markAsUnsafe, pcm16x0datablock.cpp:186-225) and outputDataBlock (4973-5117).
// The vertical alignment is either given by the caller (x0_stitch_frame_cta with top paddings) or found as the reference finds it:
// x0_sipad_scan_cta / x0_eipad_scan_cta compute what findSIPadding (1557-2245) / findEIFrameStitching (3588-4117) decide over, the
// decisions are host code of the library (pcm16x0_stitch_host.h).  One thread block per frame (per field for the SI scan).
#pragma once
#include "pcm16x0_deint.cuh"

namespace sdv {

enum { X0S_LINES_PF = 245, X0S_SUBLINES_PF = 735, X0S_MIN_GOOD = 35*(7-1)*3 /* MIN_GOOD_SUBLINES_PF, pcm16x0datastitcher.h:135-136 */, X0S_BLOCKS_FRAME = 2*7*35 };

struct X0AsmScratch
{
    int good[2], top[2], bottom[2];
    u8 broken[X0S_BLOCKS_FRAME];        // data block is BROKEN and not silent
    u8 counts[X0S_BLOCKS_FRAME];        // data block counts towards valid_cnt of the seam masking
    sdv_pcm16x0_subline sub[2*X0S_SUBLINES_PF];
};

SDV_HD void x0s_atomic_add(int *p, int v)
{
#if defined(__CUDA_ARCH__)
    atomicAdd(p, v);
#else
    *p += v;
#endif
}
SDV_HD void x0s_atomic_min(int *p, int v)
{
#if defined(__CUDA_ARCH__)
    atomicMin(p, v);
#else
    if(v<*p) *p = v;
#endif
}
SDV_HD void x0s_atomic_max(int *p, int v)
{
#if defined(__CUDA_ARCH__)
    atomicMax(p, v);
#else
    if(v>*p) *p = v;
#endif
}

// PCM16X0DataBlock::markAsUnsafe on the register block.
SDV_HD void x0_mark_unsafe(X0Block *b)
{
    for(int i=0;i<3;i++)
    {
        const u32 c3 = (b->crc>>(3*i))&7u;
        const int err_audio = 2-(int)((c3&1u)+((c3>>2)&1u));
        const bool full_bad = (((c3>>X0_LINE_2)&1u)==0)&&(err_audio>0);
        if(b->state[i]!=X0_AUD_BROKEN)
        {
            const u32 m1 = 1u<<(3*i+X0_LINE_1), m3 = 1u<<(3*i+X0_LINE_3);
            b->valid &= ~(m1|m3);
            if(!full_bad) b->valid |= b->crc&(m1|m3);
            b->state[i] = X0_AUD_ORIG;
        }
    }
}
SDV_HD bool x0_block_silent(const X0Block *b)
{
    for(int sb=0;sb<3;sb++) { if(b->words[sb][X0_LINE_1]!=0) return false; if(b->words[sb][X0_LINE_3]!=0) return false; }
    return true;
}
// valid_cnt of performDeinterleave counts: not silent, every audio word valid, no bit-picked word in sub-block 1.
SDV_HD bool x0_block_counts(const X0Block *b)
{
    const bool all_valid = ((b->valid&0x5u)==0x5u)&&(((b->valid>>3)&0x5u)==0x5u)&&(((b->valid>>6)&0x5u)==0x5u);
    return (!x0_block_silent(b))&&all_valid&&(b->picked_left==0)&&(b->picked_crc==0);
}
// The unsafe marking of performDeinterleave for data block q of the frame (seam masking, broken-block masking).
SDV_HD bool x0s_unsafe(const X0AsmScratch *s, int q, bool silent, bool mask_seams, int broken_mask_dur)
{
    if(silent) return false;
    bool unsafe = false;
    if(mask_seams)
    {
        int cnt = 0;
        for(int d=0;(d<=q)&&(cnt<3);d++) cnt += s->counts[d];
        if(cnt<3) unsafe = true;
    }
    if(broken_mask_dur>0) for(int d=0;(d<broken_mask_dur)&&(q-d>=0);d++) if(s->broken[q-d]) { unsafe = true; break; }
    return unsafe;
}
SDV_HD bool x0_block_broken(const X0Block *b) { return (b->state[0]==X0_AUD_BROKEN)||(b->state[1]==X0_AUD_BROKEN)||(b->state[2]==X0_AUD_BROKEN); }

SDV_HD void x0s_emit(const X0Block *b, i16 *smp, u8 *fl)
{
    i16 s6[6]; u8 f6[6];
    x0_output(b, s6, f6, (u8 *)0);
    for(int i=0;i<6;i++) { smp[i] = s6[i]; if(fl) fl[i] = f6[i]; }
}

// fr: the H*3 sub-line records of the frame (stream order: odd field, then even field; three parts per line).
// samples / sflags: [490][6] of this frame.
// mask_seams: the reference's padding search was not sure about this frame (padding_ok false, frame not silent).
// PCM16X0DataStitcher::collectCtrlBitStats (pcm16x0datastitcher.cpp:4745-4913) over the assembled frame in s->sub: the
// middle sub-lines of lines 0..3 of each of the 14 interleave blocks vote on emphasis / 44.1 kHz / EI format / code
// (control bit 0 = active; only sub-lines with a valid CRC vote).
SDV_HD u8 x0_ctrl_votes(const X0AsmScratch *s)
{
    int act[4] = { 0, 0, 0, 0 }, cnt[4] = { 0, 0, 0, 0 };
    for(int iblk=0;iblk<14;iblk++)
        for(int k=0;k<4;k++)
        {
            const sdv_pcm16x0_subline *l = s->sub+(size_t)iblk*X0_SUBLINES_ITL+1+3*k;
            if(l->flags&SDV_X0F_CRC_OK) { cnt[k]++; if(!(l->flags&SDV_X0F_CONTROL_BIT)) act[k]++; }
        }
    u8 v = 0;
    if(act[0]>cnt[0]/2) v |= SDV_X0I_EMPHASIS;
    if(act[1]>cnt[1]/2) v |= SDV_X0I_44100;
    if(act[2]>cnt[2]/2) v |= SDV_X0I_EI_FORMAT;
    if(act[3]>cnt[3]/2) v |= SDV_X0I_CODE;
    if((cnt[0]>=2)&&(cnt[1]>=2)&&(cnt[3]>=2)) v |= SDV_X0I_VALID;
    return v;
}
enum { X0_CTRL_HISTORY = 64 };       // frames before the current one whose votes count (updateCtrlBitStats keeps 65 with it)
// What frame f works with (f1_srate, f1_emph, f1_code at the end of fillFrameForOutput, 4711-4741): its own vote, or the
// majority over the last 65 frames (updateCtrlBitStats + getProbable*, 4126-4348; ties and an empty history give 44056 Hz /
// true / true -- the fall-back booleans are "bit is 1", the opposite sense of the voted ones).  hist: the votes of the
// X0_CTRL_HISTORY frames before frame 0 of the call (hist[X0_CTRL_HISTORY-1] = the frame just before), NULL = none.
SDV_HD void x0_ctrl_effective(sdv_pcm16x0_frame_info *info, int f, const u8 *hist = 0)
{
    const u8 v = info[f].frame_votes;
    sdv_pcm16x0_frame_info o = info[f];
    if(v&SDV_X0I_VALID)
    {
        o.sample_rate = (v&SDV_X0I_44100) ? 44100 : 44056;
        o.emphasis = (v&SDV_X0I_EMPHASIS) ? 1 : 0;
        o.code = (v&SDV_X0I_CODE) ? 1 : 0;
    }
    else
    {
        int e_on = 0, e_off = 0, c_code = 0, c_audio = 0, r441 = 0, r440 = 0;
        for(int g=(hist||(f>=X0_CTRL_HISTORY)) ? (f-X0_CTRL_HISTORY) : 0;g<=f;g++)
        {
            const u8 h = (g<0) ? hist[X0_CTRL_HISTORY+g] : info[g].frame_votes;
            if(!(h&SDV_X0I_VALID)) continue;
            if(h&SDV_X0I_EMPHASIS) e_on++; else e_off++;
            if(h&SDV_X0I_CODE) c_code++; else c_audio++;
            if(h&SDV_X0I_44100) r441++; else r440++;
        }
        o.sample_rate = (r440<r441) ? 44100 : 44056;
        o.emphasis = (e_off<e_on) ? 0 : 1;
        o.code = (((c_code==0)&&(c_audio==0))||(c_code<c_audio)) ? 1 : 0;
    }
    info[f].sample_rate = o.sample_rate; info[f].emphasis = o.emphasis; info[f].code = o.code;
}

// Vertical alignment of one field as findSIPadding leaves it: lines of padding on top, lines of the trimmed field dropped at
// its head (cutFieldTop), lines taken (-1: all the trimmed field has).
struct X0FieldGeo { i16 top_pad, cut, lines, pad; };

SDV_HD void x0_stitch_frame_cta(const Cta &c, const sdv_line_rec *fr, int H, bool bff, int top_pad_odd, int top_pad_even, X0Cfg cfg,
                                int broken_mask_dur, bool mask_seams, X0AsmScratch *s, i16 *samples, u8 *sflags,
                                sdv_pcm16x0_frame_info *info = 0, const X0FieldGeo *geo = 0 /*[2]: odd, even field*/, bool ei = false,
                                u8 *vote = 0 /*where the frame's control-bit vote is kept for the next call, may be NULL*/)
{
    const int hf = H/2;
    const int BIG = 1<<30;
    c.sync();
    if(c.tid==0) for(int f=0;f<2;f++) { s->good[f] = 0; s->top[f] = BIG; s->bottom[f] = -1; }
    c.sync();
    // ---- findFrameTrim
    for(int i=c.tid;i<2*hf;i+=c.n)
    {
        const int f = i/hf;
        const sdv_line_rec *r = fr+(size_t)i*3;
        if((r[0].flags|r[1].flags|r[2].flags)&SDV_LF_CRC_OK) x0s_atomic_add(&s->good[f], 3);
    }
    c.sync();
    for(int i=c.tid;i<2*hf;i+=c.n)
    {
        const int f = i/hf, k = i-f*hf;
        const sdv_line_rec *r = fr+(size_t)i*3;
        const u16 any = (u16)(r[0].flags|r[1].flags|r[2].flags);
        const bool skip_bad = s->good[f]>X0S_MIN_GOOD;
        if(skip_bad ? ((any&SDV_LF_CRC_OK_IGN)!=0) : ((any&SDV_LF_BW_SET)!=0)) { x0s_atomic_min(&s->top[f], k); x0s_atomic_max(&s->bottom[f], k); }
    }
    c.sync();
    // ---- splitFrameToFields + prescanForFalsePosCRCs + fillFrameForOutput
    for(int i=c.tid;i<2*X0S_LINES_PF;i+=c.n)
    {
        const int slot = i/X0S_LINES_PF, line = i-slot*X0S_LINES_PF;
        const int f = bff ? (1-slot) : slot;
        int top = s->top[f], bottom = s->bottom[f];
        if((bottom>=0)&&(bottom==top)) bottom = -1;             // the line that sets the top does not set the bottom (pcm16x0datastitcher.cpp:318-386)
        int n = (bottom>=0) ? (bottom-top+1) : 0;
        if(n>X0S_LINES_PF) n = X0S_LINES_PF;
        int top_pad = (f==0) ? top_pad_odd : top_pad_even;
        if(geo)
        {   // the alignment the padding search found: cut at the head of the field, fewer lines, its own top padding
            top_pad = geo[f].top_pad; top += geo[f].cut; n -= geo[f].cut;
            if((geo[f].lines>=0)&&(geo[f].lines<n)) n = geo[f].lines;
            if(n<0) n = 0;
        }
        const int j = line-top_pad;
        sdv_pcm16x0_subline o[3];
        for(int part=0;part<3;part++) { o[part].words[0] = o[part].words[1] = o[part].words[2] = 0; o[part].flags = 0; o[part].picked_left = 0; }
        if((j>=0)&&(j<n))
        {
            const sdv_line_rec *r = fr+((size_t)f*hf+top+j)*3;
            bool ok[3];
            for(int part=0;part<3;part++) ok[part] = (r[part].flags&SDV_LF_CRC_OK)!=0;
            const bool pl = (r[0].mark_stages&0x0F)!=0, pr = (r[2].mark_stages&0xF0)!=0;
            const bool forced = (ok[0]&&(!ok[1])&&(!ok[2])&&pl)||((!ok[0])&&(!ok[1])&&ok[2]&&pr);
            for(int part=0;part<3;part++)
            {
                o[part].words[0] = r[part].words[0]; o[part].words[1] = r[part].words[1]; o[part].words[2] = r[part].words[2];
                u8 fl = 0;
                if(ok[part]&&!forced) fl |= SDV_X0F_CRC_OK;
                Coord cc; cc.start = r[part].data_start; cc.stop = r[part].data_stop;
                if(coord_valid(cc)&&(r[part].flags&SDV_LF_BW_SET)) fl |= SDV_X0F_HAS_DATA;
                if(r[part].mark_stages&0xF0) fl |= SDV_X0F_PICKED_RIGHT;
                if(r[part].flags&SDV_LF_CONTROL_BIT) fl |= SDV_X0F_CONTROL_BIT;
                o[part].flags = fl;
                o[part].picked_left = (u8)(r[part].mark_stages&0x0F);
            }
        }
        for(int part=0;part<3;part++) s->sub[(size_t)i*3+part] = o[part];
    }
    c.sync();
    if((info||vote)&&(c.tid==0))
    {
        sdv_pcm16x0_frame_info o; o.sample_rate = 0; o.emphasis = o.code = 0; o.frame_votes = x0_ctrl_votes(s);
        o.reserved[0] = o.reserved[1] = o.reserved[2] = 0;
        if(info) *info = o;
        if(vote) *vote = o.frame_votes;
    }
    // ---- performDeinterleave: data block q = 35*m + i from sub-lines i, i+35, i+70 of interleave block m (SI format);
    //      data block q from sub-lines q, q+490, q+980 of the frame (EI format, 5181-5186)
    for(int base=0;base<X0S_BLOCKS_FRAME;base+=c.n)
    {
        const int q = base+c.tid;
        X0Block blk;
        bool live = q<X0S_BLOCKS_FRAME;
        if(live)
        {
            const int m = q/X0_BLOCKS_ITL, i = q-m*X0_BLOCKS_ITL;
            const sdv_pcm16x0_subline *b0 = ei ? (s->sub+q) : (s->sub+(size_t)m*X0_SUBLINES_ITL+i);
            const int ofs = ei ? X0_OFS_EI : X0_OFS;
            x0_process_block(&blk, b0, b0+ofs, b0+2*ofs, ((ei ? q : i)&1)!=0, cfg);
            s->broken[q] = (x0_block_broken(&blk)&&!x0_block_silent(&blk)) ? 1 : 0;
            s->counts[q] = x0_block_counts(&blk) ? 1 : 0;
        }
        if(c.n>=X0S_BLOCKS_FRAME)
        {
            c.sync();
            if(live)
            {
                if(x0s_unsafe(s, q, x0_block_silent(&blk), mask_seams, broken_mask_dur)) x0_mark_unsafe(&blk);
                x0s_emit(&blk, samples+(size_t)q*6, sflags ? sflags+(size_t)q*6 : (u8 *)0);
            }
        }
    }
    if(c.n<X0S_BLOCKS_FRAME)
    {   // small "block" (host build): second pass recomputes every data block
        c.sync();
        for(int q=c.tid;q<X0S_BLOCKS_FRAME;q+=c.n)
        {
            X0Block blk;
            const int m = q/X0_BLOCKS_ITL, i = q-m*X0_BLOCKS_ITL;
            const sdv_pcm16x0_subline *b0 = ei ? (s->sub+q) : (s->sub+(size_t)m*X0_SUBLINES_ITL+i);
            const int ofs = ei ? X0_OFS_EI : X0_OFS;
            x0_process_block(&blk, b0, b0+ofs, b0+2*ofs, ((ei ? q : i)&1)!=0, cfg);
            if(x0s_unsafe(s, q, x0_block_silent(&blk), mask_seams, broken_mask_dur)) x0_mark_unsafe(&blk);
            x0s_emit(&blk, samples+(size_t)q*6, sflags ? sflags+(size_t)q*6 : (u8 *)0);
        }
    }
    c.sync();
}


// ------------------------------------------------------------------------------------------------ SI padding search (device part)
// PCM16X0DataStitcher::findSIPadding (pcm16x0datastitcher.cpp:1557-2245) needs, per field: trySIPadding (1129-1556) for the
// paddings 0..34, findZeroControlBitOffset (868-1055) and estimateBlockNumber (1058-1126).  All three are functions of the
// trimmed field alone; x0_sipad_scan_cta computes them for one field, the decision (with its 65-field padding history) is
// host work (X0PadChain).
enum { X0S_MAX_PAD_SI = 35, X0S_BURST_SI = 34, X0S_MIN_VALID_SI = 17, X0S_MIN_FILL_SI = 105, X0S_ILINE_DELIM = 45 };
struct X0PadScan
{
    sdv_stitch_stats st[X0S_MAX_PAD_SI];    // trySIPadding per padding: index, valid, silent, unchecked, broken, DS_RET_*
    i16 zero_ofs;                           // findZeroControlBitOffset(from the top), with findSIPadding's one-line adjustment
    u8  iblk_num;                           // estimateBlockNumber
    u8  pad0;
    u16 n_sub;                              // sub-lines of the trimmed field
    u16 top;                                // first line of the field with data (index in the field), as findFrameTrim
};
struct X0PadScratch
{
    int good[2], top[2], bottom[2];
    int n_sub;
    u8 flags[7*X0_BLOCKS_ITL];
    sdv_stitch_stats ib[7];
    sdv_pcm16x0_subline sub[X0S_SUBLINES_PF];
    u16 line_no[X0S_LINES_PF];
};
// One sub-line of the trimmed field as splitFrameToFields + prescanForFalsePosCRCs leave it.
SDV_HD void x0s_field_line(const sdv_line_rec *r /*[3]*/, sdv_pcm16x0_subline *o /*[3]*/)
{
    bool ok[3];
    for(int part=0;part<3;part++) ok[part] = (r[part].flags&SDV_LF_CRC_OK)!=0;
    const bool pl = (r[0].mark_stages&0x0F)!=0, pr = (r[2].mark_stages&0xF0)!=0;
    const bool forced = (ok[0]&&(!ok[1])&&(!ok[2])&&pl)||((!ok[0])&&(!ok[1])&&ok[2]&&pr);
    for(int part=0;part<3;part++)
    {
        o[part].words[0] = r[part].words[0]; o[part].words[1] = r[part].words[1]; o[part].words[2] = r[part].words[2];
        u8 fl = 0;
        if(ok[part]&&!forced) fl |= SDV_X0F_CRC_OK;
        Coord cc; cc.start = r[part].data_start; cc.stop = r[part].data_stop;
        if(coord_valid(cc)&&(r[part].flags&SDV_LF_BW_SET)) fl |= SDV_X0F_HAS_DATA;
        if(r[part].mark_stages&0xF0) fl |= SDV_X0F_PICKED_RIGHT;
        if(r[part].flags&SDV_LF_CONTROL_BIT) fl |= SDV_X0F_CONTROL_BIT;
        o[part].flags = fl;
        o[part].picked_left = (u8)(r[part].mark_stages&0x0F);
    }
}
// Sub-line q of the padding queue: [pad] empty lines, the field, empty lines up to 735 (what findSIPadding builds and shifts).
SDV_HD const sdv_pcm16x0_subline *x0s_queue(const X0PadScratch *s, const sdv_pcm16x0_subline *empty, int pad, int q)
{
    const int j = q-3*pad;
    return ((j>=0)&&(j<s->n_sub)) ? &s->sub[j] : empty;
}
// field: 0 = odd, 1 = even.  fr: the H*3 sub-line records of the frame.
SDV_HD void x0_sipad_scan_cta(const Cta &c, const sdv_line_rec *fr, int H, int field, X0Cfg cfg, X0PadScratch *s, X0PadScan *out)
{
    const int hf = H/2;
    const int BIG = 1<<30;
    c.sync();
    if(c.tid==0) { s->good[field] = 0; s->top[field] = BIG; s->bottom[field] = -1; }
    c.sync();
    // ---- findFrameTrim for this field (as x0_stitch_frame_cta)
    for(int k=c.tid;k<hf;k+=c.n)
    {
        const sdv_line_rec *r = fr+((size_t)field*hf+k)*3;
        if((r[0].flags|r[1].flags|r[2].flags)&SDV_LF_CRC_OK) x0s_atomic_add(&s->good[field], 3);
    }
    c.sync();
    for(int k=c.tid;k<hf;k+=c.n)
    {
        const sdv_line_rec *r = fr+((size_t)field*hf+k)*3;
        const u16 any = (u16)(r[0].flags|r[1].flags|r[2].flags);
        const bool skip_bad = s->good[field]>X0S_MIN_GOOD;
        if(skip_bad ? ((any&SDV_LF_CRC_OK_IGN)!=0) : ((any&SDV_LF_BW_SET)!=0)) { x0s_atomic_min(&s->top[field], k); x0s_atomic_max(&s->bottom[field], k); }
    }
    c.sync();
    int top = s->top[field], bottom = s->bottom[field];
    if((bottom>=0)&&(bottom==top)) bottom = -1;
    int n = (bottom>=0) ? (bottom-top+1) : 0;
    if(n>X0S_LINES_PF) n = X0S_LINES_PF;
    for(int j=c.tid;j<n;j+=c.n)
    {
        x0s_field_line(fr+((size_t)field*hf+top+j)*3, &s->sub[3*j]);
        s->line_no[j] = (u16)(2*(top+j)+1+field);
    }
    if(c.tid==0) s->n_sub = 3*n;
    c.sync();
    const int n_sub = 3*n;
    sdv_pcm16x0_subline empty; empty.words[0] = empty.words[1] = empty.words[2] = 0; empty.flags = 0; empty.picked_left = 0;
    cfg.force_check = 1; cfg.p_corr = 1;                        // pad_checker.setForcedErrorCheck(true), setPCorrection(true)
    // ---- trySIPadding for every padding
    for(int pad=0;pad<X0S_MAX_PAD_SI;pad++)
    {
        for(int q=c.tid;q<7*X0_BLOCKS_ITL;q+=c.n)
        {
            const int m = q/X0_BLOCKS_ITL, i = q-m*X0_BLOCKS_ITL, st = m*X0_SUBLINES_ITL+i;
            X0Block blk;
            x0_process_block(&blk, x0s_queue(s, &empty, pad, st), x0s_queue(s, &empty, pad, st+X0_OFS), x0s_queue(s, &empty, pad, st+2*X0_OFS), (i&1)!=0, cfg);
            const bool broken = x0_block_broken(&blk), silent = x0_block_silent(&blk);
            const bool all_valid = ((blk.valid&0x5u)==0x5u)&&(((blk.valid>>3)&0x5u)==0x5u)&&(((blk.valid>>6)&0x5u)==0x5u);      // isBlockValid(): no audio word left invalid
            const bool can_force = (!broken)&&((blk.crc&0x1FFu)==0x1FFu);                                                        // canForceCheck(): not BROKEN, no CRC error at all
            const bool fix_p = (blk.state[0]==X0_AUD_FIX_P)||(blk.state[1]==X0_AUD_FIX_P)||(blk.state[2]==X0_AUD_FIX_P);
            s->flags[q] = (u8)((all_valid&&(!silent)&&can_force ? 1 : 0)|(silent ? 2 : 0)|(((!can_force)||fix_p) ? 4 : 0)|(broken ? 8 : 0));
        }
        c.sync();
        for(int m=c.tid;m<7;m+=c.n)
        {   // the burst counters of one interleave block
            int vc = 0, sc = 0, uc = 0, bc = 0, vm = 0, sm = 0, um = 0, bm = 0;
            for(int i=0;i<X0_BLOCKS_ITL;i++)
            {
                const u8 f = s->flags[m*X0_BLOCKS_ITL+i];
                if(f&1) vc++; else if(vc>vm) vm = vc;
                if(f&2) { sc++; if(sc>=X0S_BURST_SI) vc = 0; } else { if(sc>sm) sm = sc; sc = 0; }
                if(f&4) { uc++; if(uc>X0S_BURST_SI) vc = 0; } else { if(uc>um) um = uc; uc = 0; }
                if(f&8) { bc++; if(bc>=1) vc = 0; } else { if(bc>bm) bm = bc; bc = 0; }
            }
            if(vc>vm) vm = vc;
            if(sc>sm) sm = sc;
            if(uc>um) um = uc;
            if(bc>bm) bm = bc;
            sdv_stitch_stats o; o.index = (u16)m; o.valid = (u16)vm; o.silent = (u16)sm; o.unchecked = (u16)um; o.broken = (u16)bm; o.result = 0; o.reserved = 0;
            s->ib[m] = o;
        }
        c.sync();
        if(c.tid==0)
        {   // the first and the last interleave block are left out, the rest share the worst BROKEN burst, the best one speaks
            u16 top_broken = 0;
            for(int m=1;m<=5;m++) if(s->ib[m].broken>top_broken) top_broken = s->ib[m].broken;
            int best = 1;
            for(int m=2;m<=5;m++)
            {
                const sdv_stitch_stats &a = s->ib[m], &b = s->ib[best];
                bool less;
                if(a.valid!=b.valid) less = a.valid>b.valid;
                else if(a.unchecked!=b.unchecked) less = a.unchecked<b.unchecked;
                else if(a.silent!=b.silent) less = a.silent<b.silent;
                else less = a.index<b.index;
                if(less) best = m;
            }
            sdv_stitch_stats o = s->ib[best];
            o.index = (u16)pad; o.broken = top_broken;
            if(o.unchecked>X0S_BURST_SI) o.result = SDV_DS_RET_NO_PAD;
            else if(o.valid==0) o.result = SDV_DS_RET_NO_PAD;
            else if(o.silent>X0S_BURST_SI) o.result = SDV_DS_RET_SILENCE;
            else if(o.broken>=1) o.result = SDV_DS_RET_BROKE;
            else o.result = SDV_DS_RET_OK;
            out->st[pad] = o;
        }
        c.sync();
    }
    // ---- findZeroControlBitOffset(field, f_size, from the top) + the adjustment findSIPadding makes + estimateBlockNumber
    if(c.tid==0)
    {
        int best_cnt = 0, best_ofs = 0, run = 0;
        for(int ofs=1+3;ofs-3<n_sub-3;ofs+=3)          // buf_start_ofs: 1 -> 4, 7, ... while the value before the increment is < f_size-3
        {
            int zc = 0;
            for(int m=0;m<7;m++)
            {
                const int q = ofs+m*X0_SUBLINES_ITL;
                if(q>=n_sub) break;
                if((s->sub[q].flags&SDV_X0F_CRC_OK)&&!(s->sub[q].flags&SDV_X0F_CONTROL_BIT)) zc++;
            }
            if(zc>best_cnt) { best_cnt = zc; best_ofs = ofs-1; }
            run++;
            if(run>(X0_BLOCKS_ITL*3/2)) break;
        }
        int zero_ofs = (best_cnt>0) ? best_ofs : -1;
        if((zero_ofs>=0)&&((zero_ofs+3+1)<n_sub))
        {
            const sdv_pcm16x0_subline &l = s->sub[zero_ofs+3+1];
            if((l.flags&SDV_X0F_CRC_OK)&&!(l.flags&SDV_X0F_CONTROL_BIT)) zero_ofs += 3;
        }
        int iblk = 6;
        if(zero_ofs<n_sub)
        {
            if(zero_ofs<0) iblk = 0;
            else
            {
                const int ln = s->line_no[zero_ofs/3];
                if(ln<X0S_ILINE_DELIM) iblk = 0;
                else if(ln<X0S_ILINE_DELIM+70) iblk = 1;
                else if(ln<X0S_ILINE_DELIM+140) iblk = 2;
                else if(ln<X0S_ILINE_DELIM+210) iblk = 3;
                else if(ln<X0S_ILINE_DELIM+280) iblk = 4;
                else if(ln<X0S_ILINE_DELIM+350) iblk = 5;
            }
        }
        out->zero_ofs = (i16)zero_ofs; out->iblk_num = (u8)iblk; out->pad0 = 0; out->n_sub = (u16)n_sub; out->top = (u16)((top==BIG) ? 0 : top);
    }
    c.sync();
}

// ------------------------------------------------------------------------------------------------ EI padding search (device part)
// PCM16X0DataStitcher::findEIFrameStitching (pcm16x0datastitcher.cpp:3588-4117) decides over: tryEIPadding (2380-2646) for the
// 81 paddings between the two fields of the frame (findEIPadding, 2649-2994; the padding the history proposes is one of them),
// and per field findZeroControlBitOffset from the bottom (868-1055) with estimateBlockNumber (1058-1126) for
// conditionEIFramePadding (2997-3464) / findEIDataAlignment (3467-3585).  x0_eipad_scan_cta computes them for one frame; the
// decisions are host work (X0PadChain::frame_ei).
enum { X0S_MAX_PAD_EI = 81, X0S_BURST_EI = 243, X0S_MIN_VALID_EI = 163, X0S_MIN_FILL_EI = 246, X0S_EI_GROUP = 16, X0S_EI_MAXB = 736,
       X0S_EI_LEAD = 2*X0_OFS_EI+1 };
struct X0EIScan
{
    sdv_stitch_stats st[X0S_MAX_PAD_EI];    // tryEIPadding per padding (lines between the fields): index, valid, silent, unchecked, broken, DS_RET_*
    i16 zero_ofs[2];                        // findZeroControlBitOffset(from the bottom) of the odd / even field
    u8  iblk[2];                            // estimateBlockNumber for that offset
    u16 n_sub[2];                           // sub-lines of the trimmed field
    u16 top[2];                             // first line of the field with data
};
struct X0EIScratch
{
    int good[2], top[2], bottom[2];
    int n_sub[2];
    u8 flags[X0S_EI_GROUP][X0S_EI_MAXB];
    sdv_pcm16x0_subline sub[2][X0S_SUBLINES_PF];
    u16 line_no[2][X0S_LINES_PF];
};
// fr: the H*3 sub-line records of the frame.  bff: the even field comes first in the frame.
SDV_HD void x0_eipad_scan_cta(const Cta &c, const sdv_line_rec *fr, int H, bool bff, X0Cfg cfg, X0EIScratch *s, X0EIScan *out)
{
    const int hf = H/2;
    const int BIG = 1<<30;
    c.sync();
    if(c.tid==0) for(int f=0;f<2;f++) { s->good[f] = 0; s->top[f] = BIG; s->bottom[f] = -1; }
    c.sync();
    // ---- findFrameTrim (as x0_stitch_frame_cta)
    for(int i=c.tid;i<2*hf;i+=c.n)
    {
        const sdv_line_rec *r = fr+(size_t)i*3;
        if((r[0].flags|r[1].flags|r[2].flags)&SDV_LF_CRC_OK) x0s_atomic_add(&s->good[i/hf], 3);
    }
    c.sync();
    for(int i=c.tid;i<2*hf;i+=c.n)
    {
        const int f = i/hf, k = i-f*hf;
        const sdv_line_rec *r = fr+(size_t)i*3;
        const u16 any = (u16)(r[0].flags|r[1].flags|r[2].flags);
        const bool skip_bad = s->good[f]>X0S_MIN_GOOD;
        if(skip_bad ? ((any&SDV_LF_CRC_OK_IGN)!=0) : ((any&SDV_LF_BW_SET)!=0)) { x0s_atomic_min(&s->top[f], k); x0s_atomic_max(&s->bottom[f], k); }
    }
    c.sync();
    for(int f=0;f<2;f++)
    {
        int top = s->top[f], bottom = s->bottom[f];
        if((bottom>=0)&&(bottom==top)) bottom = -1;
        int n = (bottom>=0) ? (bottom-top+1) : 0;
        if(n>X0S_LINES_PF) n = X0S_LINES_PF;
        for(int j=c.tid;j<n;j+=c.n)
        {
            x0s_field_line(fr+((size_t)f*hf+top+j)*3, &s->sub[f][3*j]);
            s->line_no[f][j] = (u16)(2*(top+j)+1+f);
        }
        if(c.tid==0) s->n_sub[f] = 3*n;
    }
    c.sync();
    const int f1 = bff ? 1 : 0, f2 = 1-f1;
    const int n1 = s->n_sub[f1], n2 = s->n_sub[f2];
    sdv_pcm16x0_subline empty; empty.words[0] = empty.words[1] = empty.words[2] = 0; empty.flags = 0; empty.picked_left = 0;
    cfg.force_check = 1; cfg.p_corr = 1;                        // pad_checker.setForcedErrorCheck(true), setPCorrection(true) (2708-2711)
    // ---- tryEIPadding for every padding: the queue is field 1, 3*pad empty sub-lines, field 2; data block b = sub-lines b, b+490, b+980
    for(int g0=0;g0<X0S_MAX_PAD_EI;g0+=X0S_EI_GROUP)
    {
        const int gn = (X0S_MAX_PAD_EI-g0<X0S_EI_GROUP) ? (X0S_MAX_PAD_EI-g0) : X0S_EI_GROUP;
        for(int idx=c.tid;idx<gn*X0S_EI_MAXB;idx+=c.n)
        {
            const int k = idx/X0S_EI_MAXB, b = idx-k*X0S_EI_MAXB, pad = g0+k;
            const int gap = n1+3*pad, size = gap+n2;
            if(b>=size-X0S_EI_LEAD) continue;
            const sdv_pcm16x0_subline *l[3];
            for(int w=0;w<3;w++)
            {
                const int q = b+w*X0_OFS_EI;
                l[w] = (q<n1) ? &s->sub[f1][q] : ((q<gap) ? &empty : &s->sub[f2][q-gap]);
            }
            X0Block blk;
            x0_process_block(&blk, l[0], l[1], l[2], (b&1)!=0, cfg);
            const bool broken = x0_block_broken(&blk), silent = x0_block_silent(&blk);
            const bool all_valid = ((blk.valid&0x5u)==0x5u)&&(((blk.valid>>3)&0x5u)==0x5u)&&(((blk.valid>>6)&0x5u)==0x5u);
            const bool can_force = (!broken)&&((blk.crc&0x1FFu)==0x1FFu);
            const bool fix_p = (blk.state[0]==X0_AUD_FIX_P)||(blk.state[1]==X0_AUD_FIX_P)||(blk.state[2]==X0_AUD_FIX_P);
            s->flags[k][b] = (u8)((all_valid&&(!silent)&&can_force ? 1 : 0)|(silent ? 2 : 0)|(((!can_force)||fix_p) ? 4 : 0)|(broken ? 8 : 0));
        }
        c.sync();
        for(int k=c.tid;k<gn;k+=c.n)
        {   // the burst counters of one padding
            const int pad = g0+k, size = n1+3*pad+n2, nb = size-X0S_EI_LEAD;
            sdv_stitch_stats o; o.index = 0; o.valid = 0; o.silent = o.unchecked = o.broken = 0xFF; o.result = SDV_DS_RET_NO_DATA; o.reserved = 0;    // FieldStitchStats::clear, frametrimset.cpp:374
            if(size>=X0_OFS_EI)
            {
                int vc = 0, sc = 0, uc = 0, bc = 0, vm = 0, sm = 0, um = 0, bm = 0;
                for(int b=0;b<nb;b++)
                {
                    const u8 f = s->flags[k][b];
                    if(f&1) vc++; else if(vc>vm) vm = vc;
                    if(f&2) { sc++; if(sc>=X0S_BURST_EI) vc = 0; } else { if(sc>sm) sm = sc; sc = 0; }
                    if(f&4) { uc++; if(uc>X0S_BURST_EI) vc = 0; } else { if(uc>um) um = uc; uc = 0; }
                    if(f&8) { bc++; if(bc>=1) vc = 0; } else { if(bc>bm) bm = bc; bc = 0; }
                }
                if(vc>vm) vm = vc;
                if(sc>sm) sm = sc;
                if(uc>um) um = uc;
                if(bc>bm) bm = bc;
                if(nb>0) { o.index = (u16)pad; o.valid = (u16)vm; o.silent = (u16)sm; o.unchecked = (u16)um; o.broken = (u16)bm; }
                if(um>X0S_BURST_EI) o.result = SDV_DS_RET_NO_PAD;
                else if(vm==0) o.result = SDV_DS_RET_NO_PAD;
                else if(sm>X0S_BURST_EI) o.result = SDV_DS_RET_SILENCE;
                else if(bm>=1) o.result = SDV_DS_RET_BROKE;
                else o.result = SDV_DS_RET_OK;
            }
            out->st[pad] = o;
        }
        c.sync();
    }
    // ---- findZeroControlBitOffset(field, f_size, from the bottom) + estimateBlockNumber, per field
    for(int f=c.tid;f<2;f+=c.n)
    {
        const int n_sub = s->n_sub[f];
        int best_cnt = 0, best_ofs = 0, run = 0;
        for(int bso=n_sub+1-3;bso>=0;bso-=3)
        {
            int zc = 0;
            for(int m=0;m<7;m++)
            {
                const int q = bso-m*X0_SUBLINES_ITL;
                if(q<0) break;
                if((s->sub[f][q].flags&SDV_X0F_CRC_OK)&&!(s->sub[f][q].flags&SDV_X0F_CONTROL_BIT)) zc++;
            }
            if(zc>best_cnt) { best_cnt = zc; best_ofs = bso-1; }
            run++;
            if(run>(X0_BLOCKS_ITL*3/2)) break;
        }
        const int zero_ofs = (best_cnt>0) ? best_ofs : -1;
        int iblk = 6;
        if(zero_ofs<n_sub)
        {
            if(zero_ofs<0) iblk = 0;
            else
            {
                const int ln = s->line_no[f][zero_ofs/3];
                if(ln<X0S_ILINE_DELIM) iblk = 0;
                else if(ln<X0S_ILINE_DELIM+70) iblk = 1;
                else if(ln<X0S_ILINE_DELIM+140) iblk = 2;
                else if(ln<X0S_ILINE_DELIM+210) iblk = 3;
                else if(ln<X0S_ILINE_DELIM+280) iblk = 4;
                else if(ln<X0S_ILINE_DELIM+350) iblk = 5;
            }
        }
        out->zero_ofs[f] = (i16)zero_ofs; out->iblk[f] = (u8)iblk; out->n_sub[f] = (u16)n_sub; out->top[f] = (u16)((s->top[f]==BIG) ? 0 : s->top[f]);
    }
    c.sync();
}

#if defined(__CUDACC__)
// The control-bit votes of the last X0_CTRL_HISTORY frames of the file as the call leaves them, into hist_out: the frames of the call,
// in front of them the tail of hist_in (the same of the call before; NULL = the call opens the history).  Returns where frame f's
// vote goes, NULL when it is not among the last ones.
__device__ __forceinline__ u8 *x0_votes_carry(const Cta &c, int f, int n_frames, const u8 *hist_in, u8 *hist_out)
{
    if(f==0) for(int i=c.tid;i<X0_CTRL_HISTORY-n_frames;i+=c.n) hist_out[i] = hist_in ? hist_in[n_frames+i] : (u8)0;
    return (f+X0_CTRL_HISTORY>=n_frames) ? hist_out+(X0_CTRL_HISTORY-n_frames+f) : (u8 *)0;
}
__global__ void __launch_bounds__(512) pcm16x0_stitch_kernel(const sdv_line_rec *recs, int n_frames, int H, int bff, int top_pad_odd,
                                                             int top_pad_even, X0Cfg cfg, int broken_mask_dur, const u8 *mask_seams,
                                                             i16 *samples, u8 *sflags, sdv_pcm16x0_frame_info *info, int ei,
                                                             const u8 *hist_in, u8 *hist_out)
{
    __shared__ X0AsmScratch s;
    const int f = blockIdx.x;
    if(f>=n_frames) return;
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    u8 *vote = x0_votes_carry(c, f, n_frames, hist_in, hist_out);
    x0_stitch_frame_cta(c, recs+(size_t)f*H*3, H, bff!=0, top_pad_odd, top_pad_even, cfg, broken_mask_dur, mask_seams ? (mask_seams[f]!=0) : false, &s,
                        samples+(size_t)f*X0S_BLOCKS_FRAME*6, sflags ? sflags+(size_t)f*X0S_BLOCKS_FRAME*6 : (u8 *)0, info ? info+f : (sdv_pcm16x0_frame_info *)0,
                        (const X0FieldGeo *)0, ei!=0, vote);
}
// One block per (frame, field): the padding scan of x0_sipad_scan_cta.
__global__ void __launch_bounds__(256) pcm16x0_sipad_kernel(const sdv_line_rec *recs, int n_frames, int H, X0Cfg cfg, X0PadScan *out)
{
    __shared__ X0PadScratch s;
    const int f = blockIdx.x>>1, field = blockIdx.x&1;
    if(f>=n_frames) return;
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    x0_sipad_scan_cta(c, recs+(size_t)f*H*3, H, field, cfg, &s, out+blockIdx.x);
}
// The frame stitcher with the alignment of every field given per frame (geo[2*f], geo[2*f+1]: odd, even field).
__global__ void __launch_bounds__(512) pcm16x0_stitch_geo_kernel(const sdv_line_rec *recs, int n_frames, int H, int bff, const X0FieldGeo *geo, X0Cfg cfg,
                                                                 int broken_mask_dur, const u8 *mask_seams, i16 *samples, u8 *sflags, sdv_pcm16x0_frame_info *info,
                                                                 int ei, const u8 *hist_in, u8 *hist_out)
{
    __shared__ X0AsmScratch s;
    const int f = blockIdx.x;
    if(f>=n_frames) return;
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    u8 *vote = x0_votes_carry(c, f, n_frames, hist_in, hist_out);
    x0_stitch_frame_cta(c, recs+(size_t)f*H*3, H, bff!=0, 0, 0, cfg, broken_mask_dur, mask_seams ? (mask_seams[f]!=0) : false, &s,
                        samples+(size_t)f*X0S_BLOCKS_FRAME*6, sflags ? sflags+(size_t)f*X0S_BLOCKS_FRAME*6 : (u8 *)0, info ? info+f : (sdv_pcm16x0_frame_info *)0,
                        geo+2*(size_t)f, ei!=0, vote);
}
// One block per frame: the EI padding scan of x0_eipad_scan_cta.
__global__ void __launch_bounds__(256) pcm16x0_eipad_kernel(const sdv_line_rec *recs, int n_frames, int H, int bff, X0Cfg cfg, X0EIScan *out)
{
    __shared__ X0EIScratch s;
    const int f = blockIdx.x;
    if(f>=n_frames) return;
    Cta c = { (int)threadIdx.x, (int)blockDim.x };
    x0_eipad_scan_cta(c, recs+(size_t)f*H*3, H, bff!=0, cfg, &s, out+f);
}
__global__ void pcm16x0_ctrl_history_kernel(sdv_pcm16x0_frame_info *info, int n_frames, const u8 *hist)
{
    const int f = blockIdx.x*blockDim.x+threadIdx.x;
    if(f<n_frames) x0_ctrl_effective(info, f, hist);     // reads frame_votes of 65 frames, writes the other fields of its own
}
#endif

}   // namespace sdv
