// stc007_stitch.cuh -- STC-007 frame assembly with the reference's own vertical alignment (STC007DataStitcher).
//
// The reference walks the tape one frame at a time (doFrameReassemble, stc007datastitcher.cpp:7250-7479):
//   findFramesTrim (259-734)         first / last line with PCM data per field           -> trim_frame_cta (device, all frames)
//   splitFramesToFields (737-985)    the four trimmed field vectors of frames A and B      -> FieldTrim: an index range, never copied
//   findFieldStitching (2929-4276)   paddings between the fields: a state machine around   -> Stitcher::find_field_stitching (host; the
//                                    tryPadding / findPadding                                 seam statistics come from the seam kernel)
//   fillFrameForOutput (4588-5388)   field 1 + inner padding + field 2 + outer padding      -> Stitcher::fill_frame -> FrameAsm (48 bytes)
//   performDeinterleave (6675-6885)  one data block per assembled line, seam masking,       -> stc007_deint_kernel over the FrameAsm map
//                                    broken-block countdown
// Everything per frame that touches line data runs on the device for all frames at once; what is left on the host is the
// frame-to-frame decision chain over a few bytes per frame (it depends on the previous frame's outcome).
#pragma once
#include "sdv_common.cuh"
#include "stc007_deint.cuh"

namespace sdv {

enum { ST_LINES_PF_NTSC = 245, ST_LINES_PF_PAL = 294, ST_BUF_SIZE_FIELD = 294 };            // config.h:80-81, stc007datastitcher.h:181
enum { ST_MIN_GOOD_LINES_PF = ST_LINES_PF_NTSC-8, ST_MIN_FILL_LINES_PF = 56 };              // stc007datastitcher.h:182-183
enum { ST_LINES_PF_MAX_PAL = ST_LINES_PF_PAL+16, ST_LINES_PF_MAX_NTSC = ST_LINES_PF_PAL-32 };  // stc007datastitcher.h:172-173
enum { ST_VID_UNKNOWN = 0, ST_VID_PAL = 1, ST_VID_NTSC = 2 };                               // FrameAsmDescriptor::VID_*
enum { ST_ORDER_UNK = 0, ST_ORDER_TFF = 1, ST_ORDER_BFF = 2 };                              // FrameAsmDescriptor::ORDER_*
enum { ST_LEAD_IN = 80, ST_TAIL = 112 };                                                     // STC007DataBlock::LINE_R2 / MIN_DEINT_DATA
enum { ST_NO_HOLE = 0xFFFF };

// One trimmed field of a frame = the non-service lines with line numbers in [top, bottom] (splitFramesToFields): records
// first .. of the field's H/2 records, [data_lines] of them; a service line (Control Block) inside the range is skipped
// (hole = its position in the vector; the reference cannot hold more than one per field on any real tape, a second one is
// reported through [holes]).
struct FieldTrim
{
    u16 top, bottom;        // line numbers in the frame (odd field 1,3,.. / even field 2,4,..); 0,0 = no data found
    u16 first;              // index in the field of the first data line
    u16 data_lines;         // lines in the vector (at most ST_BUF_SIZE_FIELD)
    u16 valid_lines;        // of them with a valid CRC
    u16 hole;               // vector position at which one record has to be skipped, ST_NO_HOLE if none
    u16 holes;              // number of service lines inside [top, bottom]
    u16 max_line;           // largest line number of a non-service line of the field (detectVideoStandard)
};
struct FrameTrim { FieldTrim odd, even; };      // 32 bytes per frame

// Record index (in the field's H/2 records) of vector element k.
SDV_HD int field_vec_index(const FieldTrim &t, int k) { return (int)t.first+k+((k>=(int)t.hole) ? 1 : 0); }

// findFramesTrim + splitFramesToFields for one field of one frame: [recs] = the field's hf records, parity 0 = odd field.
// Cooperative: every thread of the group calls it; [scr] = 8 ints of shared scratch.  Result valid in thread 0.
SDV_HD void trim_field_cta(const Cta &c, const sdv_line_rec *recs, int hf, int parity, int *scr, FieldTrim *out)
{
    // pass 1: lines with a valid CRC (isCRCValid) decide whether markers alone qualify a line as data
    if(c.tid==0) { scr[0] = 0; scr[1] = 0x7FFFFFFF; scr[2] = -1; scr[3] = 0; scr[4] = 0; scr[5] = 0; scr[6] = 0x7FFFFFFF; scr[7] = 0; }
    c.sync();
    int good = 0;
    for(int j=c.tid;j<hf;j+=c.n)
    {
        const sdv_line_rec *r = recs+j;
        if((r->service_type==SDV_SRV_NO)&&(r->flags&SDV_LF_CRC_OK)) good++;
    }
#if defined(__CUDA_ARCH__)
    if(good) atomicAdd(&scr[0], good);
#else
    scr[0] += good;
#endif
    c.sync();
    const bool skip_bad = scr[0]>ST_MIN_GOOD_LINES_PF;
    // pass 2: first / last qualifying line
    int lo = 0x7FFFFFFF, hi = -1, mx = 0;
    for(int j=c.tid;j<hf;j+=c.n)
    {
        const sdv_line_rec *r = recs+j;
        if(r->service_type!=SDV_SRV_NO) continue;
        mx = j+1;
        const bool q = ((r->flags&SDV_LF_CRC_OK_IGN)!=0)||((!skip_bad)&&((r->flags&SDV_LF_MARKERS)!=0));
        if(q) { if(j<lo) lo = j; if(j>hi) hi = j; }
    }
#if defined(__CUDA_ARCH__)
    if(hi>=0) { atomicMin(&scr[1], lo); atomicMax(&scr[2], hi); }
    if(mx) atomicMax(&scr[7], mx);
#else
    if(hi>=0) { if(lo<scr[1]) scr[1] = lo; if(hi>scr[2]) scr[2] = hi; }
    if(mx>scr[7]) scr[7] = mx;
#endif
    c.sync();
    lo = scr[1]; hi = scr[2];
    // the vector: non-service lines of [lo, hi], at most ST_BUF_SIZE_FIELD of them
    int n_srv = 0, first_srv = 0x7FFFFFFF;
    if(hi>=0)
    {
        for(int j=lo+c.tid;j<=hi;j+=c.n)
            if(recs[j].service_type!=SDV_SRV_NO) { n_srv++; if(j<first_srv) first_srv = j; }
#if defined(__CUDA_ARCH__)
        if(n_srv) { atomicAdd(&scr[3], n_srv); atomicMin(&scr[6], first_srv); }
#else
        scr[3] += n_srv; if(first_srv<scr[6]) scr[6] = first_srv;
#endif
    }
    c.sync();
    int n_data = 0, hole = ST_NO_HOLE;
    if(hi>=0)
    {
        n_data = hi-lo+1-scr[3];
        if(scr[3]>0) hole = scr[6]-lo;
        if(n_data>ST_BUF_SIZE_FIELD) n_data = ST_BUF_SIZE_FIELD;
        // valid lines among the vector's elements
        int v = 0;
        for(int k=c.tid;k<n_data;k+=c.n)
        {
            const sdv_line_rec *r = recs+lo+k+((k>=hole) ? 1 : 0);
            if((r->service_type==SDV_SRV_NO)&&(r->flags&SDV_LF_CRC_OK)) v++;
        }
#if defined(__CUDA_ARCH__)
        if(v) atomicAdd(&scr[4], v);
#else
        scr[4] += v;
#endif
    }
    c.sync();
    if(c.tid==0)
    {
        FieldTrim t;
        t.top = t.bottom = t.first = t.data_lines = t.valid_lines = 0; t.hole = ST_NO_HOLE; t.holes = 0;
        t.max_line = (u16)(scr[7] ? (2*(scr[7]-1)+1+parity) : 0);
        if(hi>=0)
        {
            t.top = (u16)(2*lo+1+parity); t.bottom = (u16)(2*hi+1+parity);
            t.first = (u16)lo; t.data_lines = (u16)n_data; t.valid_lines = (u16)scr[4];
            t.hole = (u16)hole; t.holes = (u16)scr[3];
        }
        *out = t;
    }
    c.sync();
}

// ------------------------------------------------------------------------------------------------ assembled frame
// What fillFrameForOutput queues for one frame: [pre] empty lines, n1 lines of the first field from element skip1 on,
// [inner] empty lines, n2 lines of the second field from element skip2 on, [outer] empty lines.  line0[s] = the line number
// the first line of segment s carries (line numbers step by 2 inside a segment); data segments carry their own.
struct FrameAsm
{
    i32 start;              // position of the frame's first line in the assembled stream of this call
    u16 pre, n1, inner, n2, outer;
    u16 skip1, skip2;
    u16 line0_pre, line0_inner, line0_outer;
    u8  first_even;         // the first field is the even one (BFF)
    u8  mask;               // bit 0: inner seam not trusted (mask blocks across it); bit 1: the seam to the previous frame not trusted
    u16 first1, first2;     // FieldTrim::first of the two fields (in assembly order)
    u16 hole1, hole2;       // FieldTrim::hole
    u16 total;              // lines of the frame in the stream
    u16 reserved;
};

// One line of the assembled stream: record (NULL = empty line), source frame (index+1; 0 = lead-in) and line number.
struct AsmLine { const sdv_line_rec *rec; i32 frame; i32 line; };

SDV_HD AsmLine frame_asm_line(const FrameAsm &fa, int fi, int k, const sdv_line_rec *recs, int H)
{   // line k (0 <= k < fa.total) of frame fi
    AsmLine a; a.rec = 0; a.frame = fi+1; a.line = 0;
    const int hf = H/2;
    if(k<fa.pre) { a.line = fa.line0_pre+2*k; return a; }
    k -= fa.pre;
    if(k<fa.n1)
    {
        const int e = fa.skip1+k, j = fa.first1+e+((e>=fa.hole1) ? 1 : 0);
        a.rec = recs+(size_t)fi*H+(fa.first_even ? hf : 0)+j;
        a.line = 2*j+1+(fa.first_even ? 1 : 0);
        return a;
    }
    k -= fa.n1;
    if(k<fa.inner) { a.line = fa.line0_inner+2*k; return a; }
    k -= fa.inner;
    if(k<fa.n2)
    {
        const int e = fa.skip2+k, j = fa.first2+e+((e>=fa.hole2) ? 1 : 0);
        a.rec = recs+(size_t)fi*H+(fa.first_even ? 0 : hf)+j;
        a.line = 2*j+1+(fa.first_even ? 0 : 1);
        return a;
    }
    k -= fa.n2;
    a.line = fa.line0_outer+2*k;
    return a;
}

// The assembled stream of one call: [lead] empty lines (frame 0), the frames, [tail] empty lines (frame n_frames+1), or --
// when the call continues a file -- [carry] = the last 112 lines the previous call left in the queue come first.
struct StitchMap
{
    const sdv_line_rec *recs; const FrameAsm *fa; int n_frames, H;
    int lead; int lead_line0;           // file start: 80 empty lines, numbered from lead_line0
    int tail;                           // file end: 112 empty lines numbered 1, 3, ..
    const sdv_line_rec *carry; const i32 *carry_meta; int n_carry;  // continuation: records + (frame, line) pairs of the carried lines
    i32 frame_base;                     // frame number of frame 0 of this call minus 1
    i32 frame_len;                      // usual length of a frame in the stream (2 x lines per field): first guess of the frame search
    long long n_lines;
    // audio resolution detected per field (detectAudioResolution): step_res[4*f..] = the deinterleaver modes of frame f's odd / even
    // field and of the odd / even field of the frame behind it, as they stand while frame f is assembled; NULL = the preset
    // of the call (DeintCfg::res_mode).  f0_res: the modes of the frame before frame 0 of this call (at a file start: of the lead-in).
    const u8 *step_res; u8 f0_res[2];
};
// STC007DataStitcher::getDataBlockResolution (stc007datastitcher.cpp:1272-1414) while frame [step] of the call is assembled:
// the mode of the field that holds a line (frame number, line number) -- frames other than the one before, the one assembled
// and the one behind it are unknown to the reference at that moment and count as 14 bit.
SDV_HD u8 stitch_line_res(const StitchMap &m, int step, i32 frame, i32 line)
{
    const int fi = frame-m.frame_base-1;                // index in this call
    const int par = (line&1) ? 0 : 1;
    if(fi==step+1) return m.step_res[4*step+2+par];
    if(fi==step) return m.step_res[4*step+par];
    if(fi==step-1) return (step>0) ? m.step_res[4*(step-1)+par] : m.f0_res[par];
    return SDV_RES_MODE_14BIT;
}

// Frame that holds assembled line a (lead <= a-n_carry < lead+sum of totals): frames are 2*lines_per_field long unless a
// field was cut short, so the guess a/(average) is off by a few frames at most.
SDV_HD int stitch_find_frame(const StitchMap &m, long long a, int guess)
{
    int f = guess;
    if(f<0) f = 0;
    if(f>=m.n_frames) f = m.n_frames-1;
    while((f>0)&&((long long)m.fa[f].start>a)) f--;
    while((f+1<m.n_frames)&&((long long)m.fa[f+1].start<=a)) f++;
    return f;
}

SDV_HD AsmLine stitch_line(const StitchMap &m, long long a, int *frame_hint)
{
    AsmLine o; o.rec = 0; o.frame = 0; o.line = 0;
    if(a<m.n_carry) { o.rec = m.carry+a; o.frame = m.carry_meta[2*a]; o.line = m.carry_meta[2*a+1]; if(o.line<0) { o.rec = 0; o.line = -o.line-1; } return o; }
    a -= m.n_carry;
    if(a<m.lead) { o.frame = m.frame_base; o.line = m.lead_line0+2*(int)a; return o; }
    const long long end = (m.n_frames>0) ? ((long long)m.fa[m.n_frames-1].start+m.fa[m.n_frames-1].total) : (long long)m.lead;
    if(a>=end) { o.frame = m.frame_base+m.n_frames+1; o.line = 1+2*(int)(a-end); return o; }
    const int f = stitch_find_frame(m, a, *frame_hint);
    *frame_hint = f;
    o = frame_asm_line(m.fa[f], f, (int)(a-m.fa[f].start), m.recs, m.H);
    o.frame += m.frame_base;
    return o;
}

// ------------------------------------------------------------------------------------------------ seam queue (tryPadding)
// STC007DataStitcher::tryPadding (stc007datastitcher.cpp:1417-1740): the queue = the last 120-padding lines of field 1,
// [padding] empty lines, the first 120 lines of field 2; one data block per start line, then burst statistics.
enum { SEAM_LINES = 112+8, SEAM_MAX_BURST_SILENCE = 8, SEAM_MAX_BURST_BROKEN = 1 };
// A field vector as the seam sweep sees it: [size] lines from record [first] on, one record skipped at position [hole].
struct SeamField { u32 first; u16 size, hole; };
struct SeamTask { SeamField f1, f2; u16 pad0, n_pad; u32 out; u8 res1, res2, pad_[2]; };   // paddings pad0 .. pad0+n_pad-1 -> out[0..n_pad); res1 / res2: resolution
                                                                                            // modes of the two fields (RES_ANY = the caller's cfg.res_mode)
enum { RES_ANY = 0xFF };
// STC007DataStitcher::getResolutionModeForSeam (stc007datastitcher.cpp:1214-1253): the deinterleaver mode for a block that starts
// in a field of mode a and ends in a field of mode b.
SDV_HD u8 seam_res_mode(u8 a, u8 b)
{
    if(a==b) return (a==SDV_RES_MODE_14BIT_AUTO) ? (u8)SDV_RES_MODE_14BIT : ((a==SDV_RES_MODE_16BIT_AUTO) ? (u8)SDV_RES_MODE_16BIT : a);
    if((a==SDV_RES_MODE_14BIT)&&(b==SDV_RES_MODE_14BIT_AUTO)) return SDV_RES_MODE_14BIT_AUTO;
    if((a==SDV_RES_MODE_14BIT_AUTO)&&(b==SDV_RES_MODE_14BIT)) return SDV_RES_MODE_14BIT_AUTO;
    if((a==SDV_RES_MODE_16BIT)&&(b==SDV_RES_MODE_14BIT)) return SDV_RES_MODE_14BIT_AUTO;
    return SDV_RES_MODE_16BIT_AUTO;
}
SDV_HD const sdv_line_rec *seam_field_rec(const sdv_line_rec *recs, const SeamField &f, int k) { return recs+f.first+k+((k>=(int)f.hole) ? 1 : 0); }

struct SeamGeom { int start1, t1, pad, t2, n, nblk; };
SDV_HD SeamGeom seam_geom(int n1, int n2, int pad)
{
    SeamGeom g;
    const int keep = SEAM_LINES-pad;                // lines of field 1 that stay in front of the padding (negative: none)
    g.start1 = (n1>keep) ? (n1-keep) : 0;
    if(g.start1>n1) g.start1 = n1;
    g.t1 = n1-g.start1;
    g.pad = pad;
    g.t2 = (n2>SEAM_LINES) ? SEAM_LINES : n2;
    g.n = g.t1+pad+g.t2;
    g.nblk = (g.n>112) ? (g.n-112) : 0;
    return g;
}
// tryPadding sets the deinterleaver once per queue: getDataBlockResolution(&padding_queue, 0) (stc007datastitcher.cpp:1549,
// 1272-1414) = the fields queue lines 0 and 112 belong to (padding lines carry the frame number and the parity of field 1).
SDV_HD u8 seam_queue_res_mode(const SeamTask &t, const SeamGeom &g, u8 fallback)
{
    if((t.res1==RES_ANY)||(t.res2==RES_ANY)) return fallback;
    const u8 first = ((g.t1>0)||(g.pad>0)) ? t.res1 : t.res2;
    const u8 last = (112<g.t1+g.pad) ? t.res1 : t.res2;
    return seam_res_mode(first, last);
}
// Flags of queue block s: bit 0 valid and checkable and not silent, 1 silent, 2 unchecked, 3 BROKEN.
SDV_HD u8 seam_block_flags(const sdv_line_rec *recs, const SeamTask &t, const SeamGeom &g, int s, DeintCfg cfg)
{
    BlockIn in; in.ok = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<8;k++)
    {
        const int q = s+16*k;
        const sdv_line_rec *r = 0;
        if(q<g.t1) r = seam_field_rec(recs, t.f1, g.start1+q);
        else if(q>=g.t1+g.pad) r = seam_field_rec(recs, t.f2, q-g.t1-g.pad);
        u16 w = 0, sw = 0; bool ok = false;
        if(r) { w = r->words[k]; sw = r->words[7]; ok = line_rec_ok(r, cfg.ignore_crc!=0); }
        in.w[k] = w; in.sw[k] = sw;
        if(ok) in.ok |= (u8)(1u<<k);
    }
    Block blk;
    deint_dispatch(&blk, &in, cfg);
    const bool broken = blk.audio_state==SDV_AUD_BROKEN;
    const bool silent = blk_silent(&blk);
    const int errs = popc8((u32)(~blk.line_crc)&blk_word_limit_mask(&blk));
    const bool can_force = (!broken)&&((blk.resolution==RES_14BIT) ? (errs<=1) : (errs==0));
    const bool unch = cfg.q_corr ? ((!can_force)||(blk.audio_state==SDV_AUD_FIX_Q)) : (blk.audio_state==SDV_AUD_FIX_P);
    return (u8)((blk_block_valid(&blk)&&(!silent)&&can_force ? 1 : 0)|(silent ? 2 : 0)|(unch ? 4 : 0)|(broken ? 8 : 0));
}
struct SeamCount { int valid_cnt, silence_cnt, uncheck_cnt, broken_cnt, valid_max, silence_max, uncheck_max; };
SDV_HD void seam_count_init(SeamCount *c) { c->valid_cnt = c->silence_cnt = c->uncheck_cnt = c->broken_cnt = c->valid_max = c->silence_max = c->uncheck_max = 0; }
SDV_HD void seam_count_step(SeamCount *c, u8 f, int lim)
{
    if(f&1) c->valid_cnt++; else if(c->valid_cnt>c->valid_max) c->valid_max = c->valid_cnt;
    if(f&2) { c->silence_cnt++; if(c->silence_cnt>=SEAM_MAX_BURST_SILENCE) c->valid_cnt = 0; }
    else { if(c->silence_cnt>c->silence_max) c->silence_max = c->silence_cnt; c->silence_cnt = 0; }
    if(f&4) { c->uncheck_cnt++; if(c->uncheck_cnt>=lim) c->valid_cnt = 0; }
    else { if(c->uncheck_cnt>c->uncheck_max) c->uncheck_max = c->uncheck_cnt; c->uncheck_cnt = 0; }
    if(f&8) { c->broken_cnt++; if(c->broken_cnt>=SEAM_MAX_BURST_BROKEN) c->valid_cnt = 0; }
}
SDV_HD sdv_stitch_stats seam_count_finish(SeamCount *c, const SeamGeom &g, int lim)
{
    sdv_stitch_stats o; memset(&o, 0, sizeof(o));
    if(g.n<112) { o.silent = o.unchecked = o.broken = 0xFF; o.result = SDV_DS_RET_NO_DATA; return o; }    // FieldStitchStats::clear() values: the reference leaves the caller's object alone
    // n == 112: no block fits, all counters zero -> NO_PAD; the reference writes the statistics here only by grace of an
    // uninitialised flag (run_lock, stc007datastitcher.cpp:1424/1563) -- its compiled behaviour is followed
    if(c->valid_cnt>c->valid_max) c->valid_max = c->valid_cnt;
    if(c->silence_cnt>c->silence_max) c->silence_max = c->silence_cnt;
    if(c->uncheck_cnt>c->uncheck_max) c->uncheck_max = c->uncheck_cnt;
    o.index = (u16)g.pad; o.valid = (u16)c->valid_max; o.silent = (u16)c->silence_max; o.unchecked = (u16)c->uncheck_max; o.broken = (u16)c->broken_cnt;
    if(c->broken_cnt>=SEAM_MAX_BURST_BROKEN) o.result = SDV_DS_RET_BROKE;
    else if(c->silence_max>SEAM_MAX_BURST_SILENCE) o.result = SDV_DS_RET_SILENCE;
    else if(c->uncheck_max>lim) o.result = SDV_DS_RET_NO_PAD;
    else if(c->valid_max==0) o.result = SDV_DS_RET_NO_PAD;
    else o.result = SDV_DS_RET_OK;
    return o;
}

// ------------------------------------------------------------------------------------------------ audio resolution of a field
// STC007DataStitcher::getFieldResolution (stc007datastitcher.cpp:996-1195): every block that lies inside the trimmed field
// is deinterleaved twice -- as 14-bit and as 16-bit data, P correction only, parity check forced -- and two counters follow the
// blocks in order: +1 for a valid, checkable, non-silent block, -1 (not below 0) for a BROKEN one.
enum { ST_RES_UNKNOWN = 0, ST_RES_14BIT = 1, ST_RES_16BIT = 2 };        // STC007DataStitcher::SAMPLE_RES_*
// Code of block [index] of the field: bits 0-1 for the 14-bit try, bits 2-3 for the 16-bit try (1 = counts, 2 = BROKEN).
SDV_HD u8 field_res_flags(const sdv_line_rec *recs, const SeamField &f, int index, bool m2)
{
    BlockIn in; in.ok = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<8;k++)
    {
        const sdv_line_rec *r = seam_field_rec(recs, f, index+16*k);
        in.w[k] = r->words[k]; in.sw[k] = r->words[7];
        if(line_rec_ok(r, false)) in.ok |= (u8)(1u<<k);
    }
    u8 out = 0;
    for(int pass=0;pass<2;pass++)
    {
        DeintCfg cfg; cfg.res_mode = pass ? SDV_RES_MODE_16BIT : SDV_RES_MODE_14BIT; cfg.ignore_crc = 0; cfg.force_check = 1; cfg.p_corr = 1; cfg.q_corr = 0; cfg.m2 = m2 ? 1 : 0;
        Block blk;
        deint_dispatch(&blk, &in, cfg);
        const bool broken = blk.audio_state==SDV_AUD_BROKEN;
        const int errs = popc8((u32)(~blk.line_crc)&blk_word_limit_mask(&blk));
        const bool can_force = (!broken)&&((blk.resolution==RES_14BIT) ? (errs<=1) : (errs==0));
        const u8 code = (blk_block_valid(&blk)&&can_force&&!blk_silent(&blk)) ? 1 : (broken ? 2 : 0);
        out |= (u8)(code<<(2*pass));
    }
    return out;
}
SDV_HD void field_res_step(int *c14, int *c16, u8 flags)
{
    if((flags&3)==1) (*c14)++; else if(((flags&3)==2)&&(*c14>0)) (*c14)--;
    if(((flags>>2)&3)==1) (*c16)++; else if((((flags>>2)&3)==2)&&(*c16>0)) (*c16)--;
}
SDV_HD u8 field_res_decide(int c14, int c16)
{
    if(c14<=32) return ST_RES_UNKNOWN;                  // INTERLEAVE_OFS*2
    const u16 t = (u16)((u16)(c16*128)/(u16)c14);       // uint16_t arithmetic of the reference
    return (t>32) ? ST_RES_16BIT : ST_RES_14BIT;
}

// ------------------------------------------------------------------------------------------------ blocks of the assembled stream
// Block b of the stream of a StitchMap: its eight lines, and whether performDeinterleave's seam masking applies
// (stc007datastitcher.cpp:6738-6771): the block runs across the inner seam of a frame whose inner padding is not trusted
// (start line number above the stop line number, both in that frame), or across the seam between two frames whose
// outer padding is not trusted.
SDV_HD bool stitch_block_in(const StitchMap &m, long long b, bool ignore_crc, BlockIn *in, int *hint, u8 *res_mode)
{
    in->ok = 0;
    AsmLine first, last;
    first.frame = last.frame = 0; first.line = last.line = 0; first.rec = last.rec = 0;
    for(int k=0;k<8;k++)
    {
        const AsmLine l = stitch_line(m, b+16*k, hint);
        u16 w = 0, sw = 0; bool ok = false;
        if(l.rec) { w = l.rec->words[k]; sw = l.rec->words[7]; ok = line_rec_ok(l.rec, ignore_crc); }
        in->w[k] = w; in->sw[k] = sw;
        if(ok) in->ok |= (u8)(1u<<k);
        if(k==0) first = l;
        if(k==7) last = l;
    }
    bool masked = false;
    const int fi = last.frame-m.frame_base-1;           // the frame being assembled when the reference makes this block
    if(m.step_res&&(m.n_frames>0))
    {   // (the closing lines of a file carry the number of the frame behind the last one and are queued with it)
        const int step = (fi<0) ? 0 : ((fi>=m.n_frames) ? (m.n_frames-1) : fi);
        *res_mode = seam_res_mode(stitch_line_res(m, step, first.frame, first.line), stitch_line_res(m, step, last.frame, last.line));
    }
    if((fi>=0)&&(fi<m.n_frames))
    {
        const u8 mk = m.fa[fi].mask;
        if((mk&1)&&(first.frame==last.frame)&&(first.line>last.line)) masked = true;
        if((mk&2)&&(first.frame!=last.frame)&&(first.frame==last.frame-1)) masked = true;
    }
    return masked;
}

// ------------------------------------------------------------------------------------------------ the carried state as a blob
// sdv_stc007_stitch_state_save / _load: everything a call with file_start = 0 reads from the handle, in one canonical byte
// layout, so that two states with the same future compare equal with memcmp.  The header (host part of the state: frame state,
// histories rotated to position 0, countdown, counts) is built on the host; the line part moves on the device.  Frame numbers
// are stored counted from the first frame after the state (that frame = 0); lines past the valid counts are zero.
enum { SB_MAGIC = 0x53535453u /* "STSS" */, SB_VERSION = 1, SB_HDR = 256,
       SB_RECS = SB_HDR,                        // ST_TAIL carried line records (sdv_line_rec, 32 bytes)
       SB_META = SB_RECS+ST_TAIL*32,            // ST_TAIL (frame, line) pairs (i32)
       SB_CWD = SB_META+ST_TAIL*8,              // ST_TAIL CWD-patched lines (CwdLine, 32 bytes, frame number in its last word)
       SB_BYTES = SB_CWD+ST_TAIL*32 };
// Header byte offsets.
enum { SBH_MAGIC = 0, SBH_VERSION = 4, SBH_FLAGS = 6, SBH_SIZE = 8, SBH_CARRY = 12, SBH_CWD_VALID = 16, SBH_COUNTDOWN = 20,
       SBH_F0 = 24 /* FrameSt: 4 x u16, then 13 x u8 */, SBH_LAST_PAD = 56, SBH_ORDER = 64 /* 65 entries */, SBH_RES = 132 /* 65 entries */ };
enum { SB_FLAG_CWD = 1, SB_FLAG_RES_AUTO = 2 };
struct StitchBlobHdr { u32 w[SB_HDR/4]; };

#if defined(__CUDACC__)
// Blob word k <- header | records | (frame - base, line) | CWD lines with frame - base.  n_carry / n_cwd: valid lines.
__global__ void __launch_bounds__(256) stitch_state_pack_kernel(StitchBlobHdr hdr, const u32 *recs, const i32 *meta, const u32 *cwd,
                                                                int n_carry, int n_cwd, i32 base, u32 *blob)
{
    for(int k=blockIdx.x*blockDim.x+threadIdx.x;k<SB_BYTES/4;k+=gridDim.x*blockDim.x)
    {
        u32 v = 0;
        if(k<SB_RECS/4)
        {   // (selected, not indexed: a dynamic index into a kernel parameter would put it on the stack)
#pragma unroll
            for(int j=0;j<SB_HDR/4;j++) if(j==k) v = hdr.w[j];
        }
        else if(k<SB_META/4) { const int i = k-SB_RECS/4; if(i/8<n_carry) v = recs[i]; }
        else if(k<SB_CWD/4) { const int i = k-SB_META/4; if(i/2<n_carry) v = (i&1) ? (u32)meta[i] : (u32)(meta[i]-base); }
        else { const int i = k-SB_CWD/4; if(i/8<n_cwd) v = ((i&7)==7) ? (u32)((i32)cwd[i]-base) : cwd[i]; }
        blob[k] = v;
    }
}
// The line part of a blob back into the handle's carry slot, frame numbers + base.
__global__ void __launch_bounds__(256) stitch_state_unpack_kernel(const u32 *blob, u32 *recs, i32 *meta, u32 *cwd, i32 base)
{
    for(int k=SB_RECS/4+blockIdx.x*blockDim.x+threadIdx.x;k<SB_BYTES/4;k+=gridDim.x*blockDim.x)
    {
        const u32 v = blob[k];
        if(k<SB_META/4) recs[k-SB_RECS/4] = v;
        else if(k<SB_CWD/4) { const int i = k-SB_META/4; meta[i] = (i&1) ? (i32)v : (i32)v+base; }
        else { const int i = k-SB_CWD/4; cwd[i] = ((i&7)==7) ? (u32)((i32)v+base) : v; }
    }
}
#endif

}   // namespace sdv
