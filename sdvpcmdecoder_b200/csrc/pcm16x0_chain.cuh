// pcm16x0_chain.cuh -- the inter-line chain of VideoToDigital::doBinarize (videotodigital.cpp:698-1815) for PCM-16x0:
// three sub-lines per video line, the prescan reads the right part, a line forced bad takes its later parts with it.
#pragma once
#include "pcm16x0_line.cuh"
#include "pcm1_chain.cuh"

namespace sdv {

struct X0ChainCtx
{
    BinState bin;
    u8 field_state, line_dup, prescan_ref, force_bad_line;
    u16 last_words[3][3];                   // per part: words of the previous sub-line with PCM in this field
    Coord last_valid[COORD_HISTORY_DEPTH*3];
    Coord long_valid[COORD_LONG_HISTORY];
    int n_last, n_long;
    Coord frame_avg;
    P1Preset run_g;                         // presets of the file's first frame: the running pair G of the bulk pass
    int n_fv, n_fi;
    int good_in_field, pcm_in_field, line_in_field;
    Coord frame_valid[SDV_MAX_H*3];
    Coord frame_invalid[SDV_MAX_H*3];
};

SDV_HD bool x0_words_almost_silent(const u16 *w)
{   // pcm16x0subline.cpp:294-319
    const i16 a = (i16)w[0], b = (i16)w[2];
    return ((a<4)&&(a>=-4))||((b<4)&&(b>=-4));
}
SDV_HD int x0_words_diff8(const u16 *a, const u16 *b)
{
    int cnt = 0;
    for(int i=0;i<3;i++)
    {
        u32 d = (u32)((a[i]^b[i])&0xFF);
#if defined(__CUDA_ARCH__)
        cnt += __popc(d);
#else
        cnt += __builtin_popcount(d);
#endif
    }
    return cnt;
}
SDV_HD void x0_bin_set_good(BinState *b, const X0Line *l)
{
    if(x0_crc_ok_ign(l)) { b->def_ref = l->ref; bin_set_coords(b, l->coords); bin_set_bw(b, l->black, l->white); }
}
SDV_HD Coord median_hist(const Coord *v, int n)
{   // medianCoordinates over up to 27 entries (median_small works on any small n)
    return median_small(v, n);
}

SDV_HD void x0_chain_reset(X0ChainCtx *x, int mode, int line_dup)
{
    bin_set_mode(&x->bin, mode);
    x->bin.def_coord = coord_none();
    bin_reset_good(&x->bin);
    x->field_state = FIELD_NEW; x->line_dup = (u8)(line_dup ? 1 : 0); x->prescan_ref = 128; x->force_bad_line = 0;
    for(int p=0;p<3;p++) for(int i=0;i<3;i++) x->last_words[p][i] = 0;
    x->n_last = x->n_long = 0; x->n_fv = x->n_fi = 0;
    x->frame_avg = coord_none();
    x->good_in_field = x->pcm_in_field = x->line_in_field = 0;
}
SDV_HD void x0_chain_frame_start(X0ChainCtx *x, bool prescan_ran, P1Preset ps)
{
    x->frame_avg = coord_none();
    if(prescan_ran)
    {
        bin_reset_good(&x->bin);
        if(ps.valid) { x->frame_avg = ps.coords; x->prescan_ref = ps.ref; }
    }
    if(!coord_valid(x->frame_avg)) x->frame_avg = median_small(x->long_valid, x->n_long);
    else x->bin.def_ref = x->prescan_ref;
    if(coord_valid(x->frame_avg)) bin_set_coords2(&x->bin, x->frame_avg.start, x->frame_avg.stop);
    x->field_state = FIELD_NEW;
    x->good_in_field = x->pcm_in_field = 0;
}
SDV_HD void x0_chain_field_end(X0ChainCtx *x)
{
    x->field_state = FIELD_NEW;
    x->good_in_field = x->pcm_in_field = x->line_in_field = 0;
    for(int p=0;p<3;p++) for(int i=0;i<3;i++) x->last_words[p][i] = 0;
}
SDV_HD void x0_chain_frame_end(X0ChainCtx *x, Coord med_valid, Coord med_invalid)
{
    x->frame_avg = med_valid;
    if(coord_valid(x->frame_avg))
    {
        if(x->n_long==COORD_LONG_HISTORY) { for(int i=1;i<COORD_LONG_HISTORY;i++) x->long_valid[i-1] = x->long_valid[i]; x->n_long--; }
        x->long_valid[x->n_long++] = x->frame_avg;
    }
    else
    {
        x->frame_avg = med_invalid;
        if(!coord_valid(x->frame_avg)) x->frame_avg = median_small(x->long_valid, x->n_long);
    }
    x->n_fv = x->n_fi = 0;
}
// setCoordinatesSearch() before each sub-line (videotodigital.cpp:915-937).
SDV_HD bool x0_chain_coord_search(const X0ChainCtx *x)
{
    if((x->bin.mode==SDV_MODE_DRAFT)||(x->bin.mode==SDV_MODE_FAST)) return !((x->good_in_field>9)||(x->pcm_in_field>15));
    return true;
}

// What doBinarize does with one decoded sub-line (videotodigital.cpp:1006-1657), thread 0 only.  [scan_done]: the
// coordinate search has run on this video line (VideoLine::scan_done).  Call x0_chain_line_start() before the left part.
SDV_HD void x0_chain_line_start(X0ChainCtx *x) { x->force_bad_line = 0; }
SDV_HD void x0_chain_subline(X0ChainCtx *x, X0Line *line, bool scan_done)
{
    const int part = line->line_part;
    bool has_data = line->bw_set!=0;
    bool has_pcm = x0_crc_ok(line)||has_data;
    line->queue_order = (u16)x->line_in_field;
    if(has_pcm&&(x->field_state==FIELD_NEW)) x->field_state = FIELD_UNSAFE;
    if(x0_crc_ok(line)&&x->force_bad_line) line->forced_bad = 1;
    if(x0_crc_ok(line))
    {
        x->good_in_field++;
        if(x->line_dup)
        {
            if(x->field_state==FIELD_UNSAFE)
            {
                x0_bin_set_good(&x->bin, line);
                if(FINE_FIRST_LINE_DUP) { line->forced_bad = 1; x->force_bad_line = 1; }
            }
            else
            {
                bool same = x0_words_diff8(line->words, x->last_words[part])<=(X0L_PART_BITS/32);
                if((!x0_words_almost_silent(line->words))&&same) line->forced_bad = 1;
            }
        }
        if(x0_crc_ok_ign(line))
        {
            const int depth = COORD_HISTORY_DEPTH*3;
            if(x->n_last==depth) { for(int i=1;i<depth;i++) x->last_valid[i-1] = x->last_valid[i]; x->n_last--; }
            x->last_valid[x->n_last++] = line->coords;
            if(x->n_fv<SDV_MAX_H*3) x->frame_valid[x->n_fv++] = line->coords;
            if(x->n_last>(COORD_HISTORY_DEPTH/2))
            {
                Coord target = median_small(x->last_valid, x->n_last);
                if(!coord_valid(target)) target = x->frame_avg;
                if(coord_valid(target))
                {
                    i16 ds = (i16)(line->coords.start-target.start), de = (i16)(line->coords.stop-target.stop);
                    if(delta_warning(ds, de, (int)(u8)(x0_get_ppb(line)*3))) { line->forced_bad = 1; x->force_bad_line = 1; }
                }
            }
        }
        if(x0_crc_ok(line)) x0_bin_set_good(&x->bin, line);
        if(part==X0L_RIGHT) x->field_state = FIELD_INIT;
    }
    else
    {
        if(coord_valid(line->coords)) { if(x->n_fi<SDV_MAX_H*3) x->frame_invalid[x->n_fi++] = line->coords; }
        if(has_data)
        {
            Coord preset = median_small(x->last_valid, x->n_last);
            if(!coord_valid(preset)) preset = x->frame_avg;
            if(part==X0L_RIGHT)
            {
                x->field_state = FIELD_INIT;
                bin_set_coords(&x->bin, preset);
                bin_set_bw(&x->bin, 0, 0);
            }
            else
            {   // keep what this part found for the next part of the same line
                x->bin.def_ref = line->ref;
                bin_set_bw(&x->bin, line->black, line->white);
                if(scan_done) bin_set_coords(&x->bin, line->coords);
                else bin_set_coords(&x->bin, preset);
            }
        }
        else bin_set_bw(&x->bin, 0, 0);
    }
    if(has_pcm) { x->pcm_in_field++; for(int i=0;i<3;i++) x->last_words[part][i] = line->words[i]; }
    x->line_in_field++;
}

// Sub-line record: words[0..3], words[4] = queue_order, reserved = line_part, flag bit 11 = control bit.
SDV_HD void x0_export_line(const X0Line *l, sdv_line_rec *r, sdv_line_aux *a)
{
    sdv_line_rec t;
    for(int i=0;i<X0L_WORDS;i++) t.words[i] = l->words[i];
    t.words[4] = l->queue_order; t.words[5] = t.words[6] = t.words[7] = t.words[8] = 0;
    u16 f = 0;
    if(x0_crc_ok(l)) f |= SDV_LF_CRC_OK;
    if(x0_crc_ok_ign(l)) f |= SDV_LF_CRC_OK_IGN;
    if(l->forced_bad) f |= SDV_LF_FORCED_BAD;
    if(l->bw_set) f |= SDV_LF_BW_SET;
    if(l->coords_set) f |= SDV_LF_COORDS_SET;
    if(l->sweeped) f |= SDV_LF_REF_SWEEP;
    if(l->by_ext) f |= SDV_LF_BY_EXT;
    if(l->coord_sweeped) f |= SDV_LF_COORD_SWEEP;
    if(l->control_bit) f |= SDV_LF_CONTROL_BIT;
    if(x0_words_almost_silent(l->words)) f |= SDV_LF_ALMOST_SILENT;
    t.flags = f;
    t.ref = l->ref; t.black = l->black; t.white = l->white; t.hyst = l->hyst;
    t.data_start = l->coords.start; t.data_stop = l->coords.stop;
    t.shift = l->shift; t.service_type = l->service;
    t.mark_stages = (u8)(l->picked_left|(l->picked_right<<4));
    t.reserved = l->line_part;
#if defined(__CUDA_ARCH__)
    {
        uint4 v[2];
        memcpy(v, &t, sizeof(t));
        ((uint4 *)r)[0] = v[0]; ((uint4 *)r)[1] = v[1];
    }
#else
    *r = t;
#endif
    if(a)
    {
        sdv_line_aux u;
        u.ref_low = l->ref_low; u.ref_high = l->ref_high;
        u.marker_start_bg = u.marker_start_ed = u.marker_stop_ed = 0;
        u.word_crc_mask = u.word_valid_mask = 0;
        u.pad[0] = u.pad[1] = u.pad[2] = u.pad[3] = 0;
        *a = u;
    }
}

}   // namespace sdv
