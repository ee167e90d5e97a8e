// stc007_deint.cuh -- STC-007 deinterleave + P/Q error correction for one data block.
//
// Restructuring of STC007Deinterleaver::processBlock (stc007deinterleaver.cpp:286-1123) with its helpers
// (setWordData 1126-1294, calcPcode/calcQcode 1297-1317, fixByP 1376-1464, fixByQ 1468-2048, matrices 4-75) and the
// STC007DataBlock flag logic (stc007datablock.cpp:79-201, 305-312, 465-477, 507-562) as one thread per data block:
// the block lives in registers (8 words + two 8-bit flag masks) and the b-adjacent code is evaluated with
// shift/feedback steps of T and parity-of-AND against the (T^k+I)^-1 bit matrices.  CWD is out of scope.
#pragma once
#include "sdv_common.cuh"

namespace sdv {

enum { W_L0 = 0, W_R0, W_L1, W_R1, W_L2, W_R2, W_P0, W_Q0, W_CNT };
enum { RES_14BIT = 0, RES_16BIT = 1 };
enum { NO_ERR_INDEX = 64, DI_MAX_PASSES = 3 };
enum { DSTG_DATA_FILL = 0, DSTG_ERROR_CHECK, DSTG_TASK_SELECTION, DSTG_CWD_CORR, DSTG_P_CORR, DSTG_Q_CORR, DSTG_BAD_BLOCK, DSTG_NO_CHECK, DSTG_DATA_OK, DSTG_CONVERT_MAX };
enum { FIX_NOT_NEED = 0, FIX_SWITCH_P, FIX_BROKEN, FIX_NA, FIX_DONE };
enum { SDV_BF_VALID = 1, SDV_BF_BROKEN = 2, SDV_BF_FIX_P = 4, SDV_BF_FIX_Q = 8, SDV_BF_SILENT = 16, SDV_BF_UNSAFE = 32 };

struct Block
{
    u16 words[W_CNT];
    u8 line_crc, word_valid;        // bit masks over the 8 words
    u8 resolution, audio_state;
    u8 m2;                          // STC007DataBlock::m2_format: M2 range/sign expansion of the samples
};

// T = multiplication by x modulo x^14 + x^8 + 1 (rows of TP1_MATRIX, stc007deinterleaver.cpp:8-11) and its inverse.
SDV_HD u32 t_fwd(u32 v) { u32 fb = (v>>13)&1u; return ((v<<1)&0x3FFFu)^fb^(fb<<8); }
// Q = sum T^(6-k) w[k] over the six audio words: T is 'times x' modulo x^14+x^8+1, so the sum is the 20-bit polynomial
// sum w[k] x^(6-k) folded once (its top six bits land on bits 0..5 and 8..13: no second carry).
SDV_HD u32 q_of_words(const u32 *w)
{
    const u32 u = ((w[0]&0x3FFFu)<<6)^((w[1]&0x3FFFu)<<5)^((w[2]&0x3FFFu)<<4)^((w[3]&0x3FFFu)<<3)^((w[4]&0x3FFFu)<<2)^((w[5]&0x3FFFu)<<1);
    const u32 hi = u>>14;
    return (u&0x3FFFu)^hi^(hi<<8);
}
SDV_HD u32 t_inv(u32 v) { u32 lb = v&1u; return ((v>>1)^(lb<<13)^(lb<<7))&0x3FFFu; }
SDV_HD u32 t_pow(u32 v, int k) { v &= 0x3FFFu; for(;k>0;k--) v = t_fwd(v); for(;k<0;k++) v = t_inv(v); return v; }

// (T^k + I)^-1, k = 1..5, as bit matrices: row r = mask of the input bits XOR-ed into output bit r
// (TP1IN1_MATRIX .. TP5IN1_MATRIX, stc007deinterleaver.cpp:56-75).
#define SDV_TPIN1_ROWS \
    { 0x3FFE, 0x3FFC, 0x3FF8, 0x3FF0, 0x3FE0, 0x3FC0, 0x3F80, 0x3F00, 0x01FF, 0x03FF, 0x07FF, 0x0FFF, 0x1FFF, 0x3FFF }, \
    { 0x1554, 0x2AA8, 0x1550, 0x2AA0, 0x1540, 0x2A80, 0x1500, 0x2A00, 0x0155, 0x02AA, 0x0555, 0x0AAA, 0x1555, 0x2AAA }, \
    { 0x1248, 0x2490, 0x0920, 0x1240, 0x2480, 0x0900, 0x1200, 0x2400, 0x1A49, 0x3492, 0x2924, 0x1249, 0x2492, 0x0924 }, \
    { 0x0445, 0x088A, 0x1115, 0x222A, 0x0455, 0x08AA, 0x1155, 0x22AA, 0x0111, 0x0222, 0x0444, 0x0888, 0x1111, 0x2222 }, \
    { 0x1AD7, 0x35AF, 0x2B5E, 0x16BD, 0x2D7B, 0x1AF7, 0x35EF, 0x2BDE, 0x0D6B, 0x1AD6, 0x35AD, 0x2B5A, 0x16B5, 0x2D6B }
#if defined(__CUDACC__)
__constant__ u16 c_tpin1[5][14] = { SDV_TPIN1_ROWS };
#endif
static const u16 h_tpin1[5][14] = { SDV_TPIN1_ROWS };
#if defined(__CUDA_ARCH__)
#define SDV_TPIN1 c_tpin1
#else
#define SDV_TPIN1 h_tpin1
#endif
SDV_HD u32 parity32(u32 v)
{
#if defined(__CUDA_ARCH__)
    return (u32)__popc(v)&1u;
#else
    return (u32)__builtin_parity(v);
#endif
}
SDV_HD u32 mult_tpin1(int k /*1..5*/, u32 v)
{
    u32 r = 0;
    for(int bit=0;bit<14;bit++) r |= parity32((u32)SDV_TPIN1[k-1][bit]&v&0x3FFFu)<<bit;
    return r;
}

SDV_HD u16 blk_calc_p(const Block *b) { return (u16)(b->words[0]^b->words[1]^b->words[2]^b->words[3]^b->words[4]^b->words[5]); }
SDV_HD u16 blk_calc_q(const Block *b)
{   // Q = sum T^(6-i) w_i, Horner form
    u32 q = 0;
    for(int i=0;i<6;i++) q = t_fwd(q^(b->words[i]&0x3FFFu));
    return (u16)q;
}
SDV_HD u16 blk_synd_p(const Block *b) { return (u16)(blk_calc_p(b)^b->words[W_P0]); }
SDV_HD u16 blk_synd_q(const Block *b) { return (u16)(blk_calc_q(b)^b->words[W_Q0]); }
SDV_HD bool blk_crc(const Block *b, int i) { return (b->line_crc>>i)&1; }
SDV_HD bool blk_valid(const Block *b, int i) { return (b->word_valid>>i)&1; }
SDV_HD void blk_set_valid(Block *b, int i) { b->word_valid |= (u8)(1u<<i); }
// Word access by a run-time index is written as an unrolled select so that the block stays in registers.
SDV_HD u16 blk_get_word(const Block *b, int i)
{
    u16 r = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<W_CNT;k++) r = (k==i) ? b->words[k] : r;
    return r;
}
SDV_HD void blk_set_word(Block *b, int i, u16 w, bool ok)
{
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<W_CNT;k++) b->words[k] = (k==i) ? w : b->words[k];
    u8 m = (u8)(1u<<i);
    if(ok) { b->line_crc |= m; b->word_valid |= m; } else { b->line_crc &= (u8)~m; b->word_valid &= (u8)~m; }
}
SDV_HD u8 blk_word_limit_mask(const Block *b) { return (b->resolution==RES_16BIT) ? 0x7F : 0xFF; }
SDV_HD void blk_mark_broken(Block *b)
{
    u8 m = blk_word_limit_mask(b);
    b->word_valid &= (u8)~m; b->line_crc &= (u8)~m;
    b->audio_state = SDV_AUD_BROKEN;
}
// STC007DataBlock::markAsUnsafe (stc007datablock.cpp:168-201)
SDV_HD void blk_mark_unsafe(Block *b)
{
    if(b->audio_state==SDV_AUD_BROKEN) return;
    u8 m = blk_word_limit_mask(b);
    b->word_valid = (u8)((b->word_valid&~m)|(b->line_crc&m));
    b->line_crc &= (u8)~m;
    b->audio_state = SDV_AUD_ORIG;
}
SDV_HD int lowest_bit(u32 v)
{
#if defined(__CUDA_ARCH__)
    return __ffs((int)v)-1;
#else
    return __builtin_ctz(v);
#endif
}
SDV_HD int popc8(u32 v)
{
#if defined(__CUDA_ARCH__)
    return __popc(v&0xFFu);
#else
    return __builtin_popcount(v&0xFFu);
#endif
}

SDV_HD void blk_recalc_p(Block *b)
{
    u16 p = blk_calc_p(b);
    if(b->words[W_P0]!=p) blk_set_word(b, W_P0, p, blk_crc(b, W_P0));
    blk_set_valid(b, W_P0);
}

SDV_HD u8 blk_fix_by_p(Block *b, u8 first_bad)
{
    b->audio_state = SDV_AUD_ORIG;
    u16 check = blk_synd_p(b);
    if(check==0) { if(first_bad!=NO_ERR_INDEX) blk_set_valid(b, first_bad); return FIX_NOT_NEED; }
    else if(first_bad==NO_ERR_INDEX) return FIX_BROKEN;
    blk_set_word(b, first_bad, (u16)(check^blk_get_word(b, first_bad)), false);
    blk_set_valid(b, first_bad);
    return FIX_DONE;
}

SDV_HD u8 blk_fix_by_q(Block *b, u8 first_bad, u8 second_bad)
{
    bool fix_found = false;
    u16 sp = 0, sq, e1 = 0, e2 = 0;
    b->audio_state = SDV_AUD_ORIG;
    if(second_bad==NO_ERR_INDEX) if(!blk_valid(b, W_P0)) second_bad = W_P0;
    sq = blk_synd_q(b);
    if(second_bad==W_P0)
    {
        if(sq==0)
        {
            if(first_bad!=NO_ERR_INDEX) blk_set_valid(b, first_bad);
            blk_recalc_p(b);
            return FIX_NOT_NEED;
        }
    }
    else
    {
        sp = blk_synd_p(b);
        if((sp==0)&&(sq==0))
        {
            if(first_bad<W_CNT) blk_set_valid(b, first_bad);
            if(second_bad<W_CNT) blk_set_valid(b, second_bad);
            return FIX_NOT_NEED;
        }
    }
    if((second_bad!=W_P0)&&(!blk_valid(b, W_P0))) return FIX_NA;
    if(first_bad==NO_ERR_INDEX) return FIX_BROKEN;
    else if(second_bad==NO_ERR_INDEX) return FIX_SWITCH_P;
    if(first_bad<=W_R2)
    {
        if(second_bad==W_P0)
        {   // one audio word + P: e1 = T^-(6-i) Sq
            e1 = (u16)t_pow(sq, -(6-(int)first_bad));
            fix_found = true;
        }
        else if((second_bad<=W_R2)&&(second_bad>first_bad))
        {   // two audio words i<j: e1 = (T^(j-i)+I)^-1 (T^-(6-j) Sq + Sp), e2 = e1 + Sp
            e1 = (u16)(t_pow(sq, -(6-(int)second_bad))^sp);
            e1 = (u16)mult_tpin1((int)second_bad-(int)first_bad, e1);
            e2 = (u16)(e1^sp);
            fix_found = true;
        }
    }
    if(fix_found)
    {
        u16 old1 = blk_get_word(b, first_bad), old2;
        if(e1!=0) blk_set_word(b, first_bad, (u16)(old1^e1), false);
        blk_set_valid(b, first_bad);
        old2 = blk_get_word(b, second_bad);
        if(second_bad==W_P0) e2 = (u16)(old2^blk_calc_p(b));
        if(e2!=0) blk_set_word(b, second_bad, (u16)(old2^e2), false);
        blk_set_valid(b, second_bad);
        if((e1==0)&&(e2==0)) return FIX_NOT_NEED;
        return FIX_DONE;
    }
    return FIX_BROKEN;
}

struct DeintCfg { u8 res_mode, ignore_crc, force_check, p_corr, q_corr, m2; };

// The 8 (word, line-valid) inputs of a block: in_w[k] = all 8 data words of line s+16k are not needed, only word k and
// (16-bit mode) the S word (word 7) of the same line.
struct BlockIn { u16 w[8]; u16 sw[8]; u8 ok; };     // ok: bit k = line s+16k has a valid CRC (per cfg.ignore_crc)

// Does this line give the block a trusted word?  Normally the line's CRC state (STC007Line::isWordCRCOk); with CRC
// ignored, any line that carried data: valid coordinates and black/white levels (stc007deinterleaver.cpp:1139-1163).
SDV_HD bool line_rec_ok(const sdv_line_rec *r, bool ignore_crc)
{
    if(r->service_type!=SDV_SRV_NO) return false;
    if(!ignore_crc) return (r->flags&SDV_LF_CRC_OK)!=0;
    Coord c; c.start = r->data_start; c.stop = r->data_stop;
    return coord_valid(c)&&((r->flags&SDV_LF_BW_SET)!=0);
}

SDV_HD void blk_fill(Block *b, const BlockIn *in, u8 res)
{
    b->line_crc = b->word_valid = 0; b->audio_state = SDV_AUD_ORIG; b->resolution = res;
    if(res==RES_14BIT)
    {
        for(int k=0;k<8;k++) blk_set_word(b, k, in->w[k], (in->ok>>k)&1);
    }
    else
    {
        for(int k=0;k<7;k++)
        {
            u16 f1 = (u16)(in->w[k]<<2);
            u16 s = (u16)((in->sw[k]>>(12-2*k))&0x3);
            blk_set_word(b, k, (u16)(f1+s), (in->ok>>k)&1);
        }
        blk_set_word(b, W_Q0, 0, true);
    }
}

SDV_HD void deint_block(Block *blk, const BlockIn *in, DeintCfg cfg)
{
    u8 run_res, stage_count = 0, fill_passes, all_errs = 0, aud_errs = 0, first_bad = NO_ERR_INDEX, second_bad = NO_ERR_INDEX, fix_result, st;
    if(cfg.res_mode==SDV_RES_MODE_14BIT) { run_res = RES_14BIT; fill_passes = DI_MAX_PASSES; }
    else if(cfg.res_mode==SDV_RES_MODE_14BIT_AUTO) { run_res = RES_14BIT; fill_passes = 0; }
    else if(cfg.res_mode==SDV_RES_MODE_16BIT_AUTO) { run_res = RES_16BIT; fill_passes = 0; }
    else { run_res = RES_16BIT; fill_passes = DI_MAX_PASSES; }
    st = DSTG_DATA_FILL;
    for(;;)
    {
        stage_count++;
        if(st==DSTG_DATA_FILL)
        {
            blk_fill(blk, in, run_res);
            fill_passes++;
            st = DSTG_ERROR_CHECK;
        }
        else if(st==DSTG_ERROR_CHECK)
        {
            first_bad = second_bad = NO_ERR_INDEX;
            {   // the first two audio words without a valid line CRC
                u32 bad = (u32)(~blk->line_crc)&0x3Fu;
                if(bad) { first_bad = (u8)lowest_bit(bad); bad &= bad-1; if(bad) second_bad = (u8)lowest_bit(bad); }
            }
            aud_errs = (u8)popc8((u32)(~blk->line_crc)&0x3Fu);
            all_errs = (u8)popc8((u32)(~blk->line_crc)&blk_word_limit_mask(blk));
            st = DSTG_TASK_SELECTION;
        }
        else if(st==DSTG_TASK_SELECTION)
        {
            st = DSTG_BAD_BLOCK;
            if(all_errs<=2)
            {
                if(aud_errs==0)
                {
                    if(!cfg.force_check) st = DSTG_DATA_OK;
                    else if(cfg.p_corr) st = DSTG_P_CORR;
                    else st = DSTG_NO_CHECK;
                }
                else if(aud_errs==1) { if(cfg.p_corr) st = DSTG_P_CORR; }
                else if(aud_errs==2) { if(run_res==RES_14BIT) { if(cfg.q_corr) st = DSTG_Q_CORR; } }
            }
        }
        else if(st==DSTG_P_CORR)
        {
            st = DSTG_BAD_BLOCK;
            if(blk_valid(blk, W_P0))
            {
                fix_result = blk_fix_by_p(blk, first_bad);
                if(fix_result==FIX_BROKEN) blk_mark_broken(blk);
                else
                {
                    st = DSTG_DATA_OK;
                    if(fix_result==FIX_DONE) blk->audio_state = SDV_AUD_FIX_P;
                    else if(fix_result==FIX_NOT_NEED) { if(first_bad<W_P0) blk->audio_state = SDV_AUD_FIX_P; }
                    if((run_res==RES_14BIT)&&cfg.q_corr)
                    {
                        if(blk_valid(blk, W_Q0))
                        {
                            if(cfg.force_check) { if(blk_synd_q(blk)!=0) { st = DSTG_BAD_BLOCK; blk_mark_broken(blk); } }
                        }
                        else
                        {
                            u16 q = blk_calc_q(blk);
                            if(blk->words[W_Q0]!=q) blk_set_word(blk, W_Q0, q, blk_crc(blk, W_Q0));
                            blk_set_valid(blk, W_Q0);
                        }
                    }
                }
            }
            else
            {
                if(run_res==RES_14BIT)
                {
                    if(cfg.q_corr) st = DSTG_Q_CORR;
                    else if(aud_errs==0) st = DSTG_NO_CHECK;
                }
                else if(aud_errs==0) st = DSTG_NO_CHECK;
            }
        }
        else if(st==DSTG_Q_CORR)
        {
            st = DSTG_BAD_BLOCK;
            if(blk_valid(blk, W_Q0))
            {
                fix_result = blk_fix_by_q(blk, first_bad, second_bad);
                if(!blk_crc(blk, W_P0)) second_bad = W_P0;
                if(fix_result==FIX_DONE) { st = DSTG_DATA_OK; blk->audio_state = SDV_AUD_FIX_Q; }
                else if(fix_result==FIX_NOT_NEED) { st = DSTG_DATA_OK; if(first_bad<W_P0) blk->audio_state = SDV_AUD_FIX_Q; }
                else if(fix_result==FIX_SWITCH_P) st = DSTG_P_CORR;
                else if(fix_result==FIX_BROKEN) blk_mark_broken(blk);
            }
            else if(first_bad==NO_ERR_INDEX)
            {
                st = DSTG_NO_CHECK;
                blk_set_word(blk, W_P0, blk_calc_p(blk), false); blk_set_valid(blk, W_P0);
                blk_set_word(blk, W_Q0, blk_calc_q(blk), false); blk_set_valid(blk, W_Q0);
            }
        }
        else if(st==DSTG_BAD_BLOCK)
        {
            if(fill_passes>=DI_MAX_PASSES) break;
            run_res = (run_res==RES_16BIT) ? RES_14BIT : RES_16BIT;
            st = DSTG_DATA_FILL;
        }
        else break;
        if(stage_count>(DSTG_CONVERT_MAX*DI_MAX_PASSES)) break;
    }
}

// processBlock for the stitcher's standard setting -- fixed 14-bit resolution, forced parity check, P and Q correction
// on (STC007DataStitcher::performDeinterleave with a resolution preset, stc007datastitcher.cpp:6684-6720) -- written
// out as straight-line code over the number of erased words; same results as deint_block(), far fewer instructions.
SDV_HD void deint_block_std14(Block *blk, const BlockIn *in)
{
    u32 w[8];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<8;k++) w[k] = in->w[k];
    const u32 ok = in->ok;
    u32 crc = ok, valid = ok, state = SDV_AUD_ORIG;
    const u32 bad_all = (~ok)&0xFFu, bad_aud = bad_all&0x3Fu;
    const int n_all = popc8(bad_all), n_aud = popc8(bad_aud);
    const bool pv = (ok>>W_P0)&1u, qv = (ok>>W_Q0)&1u;
    bool broken = false;
    if(n_all<=2)
    {
        const u32 cp = w[0]^w[1]^w[2]^w[3]^w[4]^w[5];
        const u32 cq = q_of_words(w);
        const u32 sp = cp^w[W_P0], sq = cq^w[W_Q0];
        if(n_aud==0)
        {
            if(pv)
            {   // parity check of an undamaged block; Q checked too, or regenerated when its line was bad
                if(sp!=0) broken = true;
                else if(qv) { if(sq!=0) broken = true; }
                else { w[W_Q0] = cq; valid |= 1u<<W_Q0; }
            }
            else if(qv)
            {   // P line bad: check by Q, regenerate P
                if(sq==0) { w[W_P0] = cp; valid |= 1u<<W_P0; } else broken = true;
            }
            else { w[W_P0] = cp; w[W_Q0] = cq; valid |= (1u<<W_P0)|(1u<<W_Q0); }     // nothing to check with
        }
        else if(n_aud==1)
        {
            const int i = lowest_bit(bad_aud);
            if(pv)
            {   // single erasure by P, then the Q check on the corrected words
                state = SDV_AUD_FIX_P;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
                for(int k=0;k<6;k++) w[k] ^= (k==i) ? sp : 0u;
                valid |= 1u<<i;
                const u32 cq2 = q_of_words(w);
                if(qv) { if((cq2^w[W_Q0])!=0) broken = true; }
                else { w[W_Q0] = cq2; valid |= 1u<<W_Q0; }
            }
            else
            {   // audio word + P erased: e = T^-(6-i) Sq, P regenerated
                state = SDV_AUD_FIX_Q;
                const u32 e1 = (sq==0) ? 0u : t_pow(sq, -(6-i));
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
                for(int k=0;k<6;k++) w[k] ^= (k==i) ? e1 : 0u;
                valid |= (1u<<i)|(1u<<W_P0);
                w[W_P0] = w[0]^w[1]^w[2]^w[3]^w[4]^w[5];
            }
        }
        else
        {   // two audio words erased (P and Q both good): e1 = (T^(j-i)+I)^-1 (T^-(6-j) Sq + Sp), e2 = e1 + Sp
            const int i = lowest_bit(bad_aud), j = lowest_bit(bad_aud&(bad_aud-1));
            state = SDV_AUD_FIX_Q;
            u32 e1 = 0, e2 = 0;
            if((sp!=0)||(sq!=0)) { e1 = mult_tpin1(j-i, t_pow(sq, -(6-j))^sp); e2 = e1^sp; }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for(int k=0;k<6;k++) w[k] ^= ((k==i) ? e1 : 0u)^((k==j) ? e2 : 0u);
            valid |= (1u<<i)|(1u<<j);
        }
    }
    if(broken) { crc = 0; valid = 0; state = SDV_AUD_BROKEN; }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<8;k++) blk->words[k] = (u16)w[k];
    blk->line_crc = (u8)crc; blk->word_valid = (u8)valid; blk->resolution = RES_14BIT; blk->audio_state = (u8)state;
}

// ---- Two adjacent blocks of the standard setting in one instruction stream.  Block s sits in the low 16-bit half of every
// word, block s+1 in the high half ("packed").  A pair in which each block has at most one untrusted line -- the clean tape:
// the uncaptured lines of a field are 16 lines apart from nothing else in a block -- is finished here with masks, without a
// branch; any other pair goes to deint_block_std14() block by block (deint_pair_std14() returns false).

// __byte_perm(x, y, s) without the sign modes: byte i of the result = byte (s>>4i)&7 of the 8-byte value y:x.
SDV_HD u32 prmt(u32 x, u32 y, u32 s)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, s);
#else
    const u64 v = ((u64)y<<32)|x;
    u32 r = 0;
    for(int i=0;i<4;i++) r |= (u32)((v>>(8*((s>>(4*i))&7u)))&0xFFu)<<(8*i);
    return r;
#endif
}
#if defined(__CUDA_ARCH__)
// PTX prmt in its default mode: a selector nibble with bit 3 set replicates the sign of the selected byte over the result byte
// (__byte_perm() drops that bit).
__device__ __forceinline__ u32 prmt_sign(u32 x, u32 s)
{
    u32 r;
    asm("prmt.b32 %0, %1, 0, %2;" : "=r"(r) : "r"(x), "r"(s));
    return r;
}
#endif
// Bit 15 / bit 31 -> 0xFFFF in the low / high half.
SDV_HD u32 msb_to_halves(u32 h)
{
#if defined(__CUDA_ARCH__)
    return prmt_sign(h, 0xBB99);                // every byte the sign of byte 1 / byte 3
#else
    return ((h>>15)&0x10001u)*0xFFFFu;
#endif
}
// 0xFFFF in each half that is not zero.
SDV_HD u32 nz_halves(u32 v) { return msb_to_halves((((v&0x7FFF7FFFu)+0x7FFF7FFFu)|v)&0x80008000u); }
// The line-trusted masks of words 2m (hi = 0) and 2m+1 (hi = 1) from the 2-bit fields of okf: bits 0 / 1 = word 2m of block
// s / s+1, bits 16 / 17 = word 2m+1.  One multiplication puts the four bits on the sign bits of the four bytes.
SDV_HD u32 pair_okmask(u32 okf, int hi)
{
    const u32 y = (okf&0x00030003u)*0x4080u;
#if defined(__CUDA_ARCH__)
    return prmt_sign(y, hi ? 0xBBAA : 0x9988);
#else
    const u32 a = (y>>(7+16*hi))&1u, b = (y>>(15+16*hi))&1u;
    return (a ? 0x0000FFFFu : 0u)|(b ? 0xFFFF0000u : 0u);
#endif
}
// q_of_words() on both halves.  The low 14 bits of every shifted word stay in their half once the bits pushed past bit 13
// (and, in the high half, the low half's carried-over bits) are masked off; those top bits -- six at most -- are gathered
// shifted down by 14, and the sum is folded once as in q_of_words().
SDV_HD u32 q_of_word_pairs(const u32 *w)
{
    u32 lo = 0, top = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<6;k++)
    {
        const int s = 6-k;
        const u32 low_s = (1u<<s)-1u;
        lo ^= (w[k]<<s)&(0x3FFF3FFFu&~(low_s<<16));
        top ^= (w[k]>>(14-s))&(low_s*0x10001u);
    }
    return lo^top^(top<<8);
}

struct BlockPair
{
    u32 words[8];       // packed block words after correction / regeneration
    u32 okm[8];         // 0xFFFF per half: the line of word k is trusted (line_crc of a block that is not BROKEN)
    u32 broken;         // 0xFFFF per half: BROKEN
    u32 fixed;          // 0xFFFF per half: an audio word was put right by P (SDV_AUD_FIX_P)
};

// deint_block_std14() for blocks s and s+1: w = packed words 0..7, okf[m] = the 2-bit fields of words 2m and 2m+1 (see
// pair_okmask; other bits are ignored).  With at most one untrusted word per block the cases of deint_block_std14() are
//   audio word i untrusted: w_i ^= Sp, then the Q check on the corrected words;
//   P untrusted: the Q check, P regenerated;  Q untrusted: the P check, Q regenerated;  none: the P and Q checks,
// which is: correct by Sp wherever an audio word is untrusted, then BROKEN = (Q trusted and Sq of the corrected words != 0)
// or (P and all audio words trusted and Sp != 0).  Returns false when a block has two or more untrusted words.
SDV_HD bool deint_pair_std14(const u32 *w, const u32 *okf, BlockPair *r)
{
    u32 o[8];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int m=0;m<4;m++) { o[2*m] = pair_okmask(okf[m], 0); o[2*m+1] = pair_okmask(okf[m], 1); }
    u32 any = 0, two = 0;           // per half: some / a second untrusted word
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<8;k++) { two |= any&~o[k]; any |= ~o[k]; }
    const u32 sp = w[0]^w[1]^w[2]^w[3]^w[4]^w[5]^w[W_P0];
    u32 c[6];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<6;k++) c[k] = w[k]^(sp&~o[k]);
    const u32 cq = q_of_word_pairs(c);
    const u32 sq = cq^w[W_Q0];
    const u32 aud_ok = o[0]&o[1]&o[2]&o[3]&o[4]&o[5];
    const u32 broken = nz_halves((sq&o[W_Q0])|(sp&aud_ok&o[W_P0]));
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<6;k++) r->words[k] = c[k];
    // a regenerated word only where the block is not BROKEN; an untrusted P means no audio word was corrected
    const u32 reg_p = ~o[W_P0]&~broken, reg_q = ~o[W_Q0]&~broken;
    r->words[W_P0] = (w[W_P0]&~reg_p)|((sp^w[W_P0])&reg_p);
    r->words[W_Q0] = (w[W_Q0]&~reg_q)|(cq&reg_q);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<8;k++) r->okm[k] = o[k];
    r->broken = broken;
    r->fixed = ~aud_ok;
    return two==0;          // (decided last: nothing above waits for it)
}

// The six samples of each block (words << 2 in 14-bit mode), as the 24 bytes they take in the sample stream.
SDV_HD void pair_samples(const BlockPair *r, u32 *d /*[6]*/)
{
    u32 s[6];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<6;k++) s[k] = (r->words[k]<<2)&0xFFFCFFFCu;
    d[0] = prmt(s[0], s[1], 0x5410); d[1] = prmt(s[2], s[3], 0x5410); d[2] = prmt(s[4], s[5], 0x5410);
    d[3] = prmt(s[0], s[1], 0x7632); d[4] = prmt(s[2], s[3], 0x7632); d[5] = prmt(s[4], s[5], 0x7632);
}
// blk_output_flags() of both blocks as the 12 flag bytes: a block that is not BROKEN has all words valid here, so a sample's
// flags are BLOCK_OK | WORD_VALID, and WORD_FIXED where its line was trusted; a BROKEN block's are 0.
SDV_HD void pair_flags(const BlockPair *r, u32 *f /*[3]*/)
{
    u32 g[6];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for(int k=0;k<6;k++) g[k] = ~r->broken&((r->okm[k]&(SDV_SF_WORD_FIXED*0x10001u))|((SDV_SF_BLOCK_OK|SDV_SF_WORD_VALID)*0x10001u));
    const u32 g01 = prmt(g[0], g[1], 0x6240), g23 = prmt(g[2], g[3], 0x6240), g45 = prmt(g[4], g[5], 0x6240);     // [A_k A_k+1 B_k B_k+1]
    f[0] = prmt(g01, g23, 0x5410); f[1] = prmt(g45, g01, 0x7610); f[2] = prmt(g23, g45, 0x7632);
}
// Bit 0 / 1: block s / s+1 is BROKEN and not silent (may open a countdown window).
SDV_HD u32 pair_broken_ns(const BlockPair *r)
{
    const u32 loud = nz_halves((r->words[0]|r->words[1]|r->words[2]|r->words[3]|r->words[4]|r->words[5])&0x3FFF3FFFu);
    const u32 b = r->broken&loud;
    return (b&1u)|((b>>15)&2u);
}
// The two Blocks deint_block_std14() would give (what the pair carries in packed form).
SDV_HD void pair_unpack(const BlockPair *r, Block *a, Block *b)
{
    Block *blk[2] = { a, b };
    for(int h=0;h<2;h++)
    {
        const int sh = 16*h;
        u32 ok = 0;
        for(int k=0;k<8;k++) { blk[h]->words[k] = (u16)(r->words[k]>>sh); ok |= ((r->okm[k]>>sh)&1u)<<k; }
        const bool broken = (r->broken>>sh)&1u;
        blk[h]->line_crc = broken ? 0 : (u8)ok;
        blk[h]->word_valid = broken ? 0 : 0xFF;
        blk[h]->resolution = RES_14BIT;
        blk[h]->audio_state = broken ? SDV_AUD_BROKEN : (((r->fixed>>sh)&1u) ? SDV_AUD_FIX_P : SDV_AUD_ORIG);
    }
}

SDV_HD bool deint_cfg_is_std14(DeintCfg cfg) { return (cfg.res_mode==SDV_RES_MODE_14BIT)&&cfg.force_check&&cfg.p_corr&&cfg.q_corr; }
SDV_HD void deint_dispatch(Block *blk, const BlockIn *in, DeintCfg cfg)
{
    if(deint_cfg_is_std14(cfg)) deint_block_std14(blk, in);
    else deint_block(blk, in, cfg);
    blk->m2 = cfg.m2;
}

SDV_HD i16 blk_sample(const Block *b, int i)
{   // STC007DataBlock::getSample (stc007datablock.cpp:505-557)
    if(b->m2) return stc_sample(b->words[i], true);
    return (b->resolution==RES_16BIT) ? (i16)b->words[i] : (i16)(u16)(b->words[i]<<2);
}
SDV_HD bool blk_silent(const Block *b)
{   // all six samples zero; without the M2 expansion that is: all six words zero in their 14 (16) bits
    if(b->m2) { for(int i=0;i<6;i++) if(blk_sample(b, i)!=0) return false; return true; }
    const u32 o = (u32)b->words[0]|b->words[1]|b->words[2]|b->words[3]|b->words[4]|b->words[5];
    return ((b->resolution==RES_16BIT) ? (o&0xFFFFu) : (o&0x3FFFu))==0;
}
SDV_HD bool blk_block_valid(const Block *b) { return (b->word_valid&0x3F)==0x3F; }

// STC007DataStitcher::outputSamplePair (stc007datastitcher.cpp:6525-6569): 6 samples + per-sample flags.
// The six flag bytes at once: f03 = samples 0..3 (byte i = sample i), f45 = samples 4, 5.  Bits of a mask are spread to
// bytes by one multiplication (the shifted copies do not overlap).
SDV_HD void blk_output_flags(const Block *b, u32 *f03, u32 *f45)
{
    const bool broken = b->audio_state==SDV_AUD_BROKEN;
    const bool bstate = (!broken)&&blk_block_valid(b);
    const u32 v = broken ? 0u : (u32)(b->word_valid&0x3F);          // word valid
    const u32 c = bstate ? (u32)(b->line_crc&0x3F) : 0u;            // "fixed" = the word's line had a valid CRC
    const u32 ok = bstate ? 1u : 0u;
    *f03 = (ok*0x01010101u*SDV_SF_BLOCK_OK)|((((v&0xFu)*0x00204081u)&0x01010101u)*SDV_SF_WORD_VALID)|((((c&0xFu)*0x00204081u)&0x01010101u)*SDV_SF_WORD_FIXED);
    *f45 = (ok*0x0101u*SDV_SF_BLOCK_OK)|((((v>>4)*0x81u)&0x0101u)*SDV_SF_WORD_VALID)|((((c>>4)*0x81u)&0x0101u)*SDV_SF_WORD_FIXED);
}
SDV_HD void blk_output(const Block *b, i16 *smp /*[6]*/, u8 *fl /*[6]*/)
{
    u32 f03, f45;
    blk_output_flags(b, &f03, &f45);
    for(int i=0;i<4;i++) fl[i] = (u8)(f03>>(8*i));
    fl[4] = (u8)f45; fl[5] = (u8)(f45>>8);
    if(b->m2) { for(int i=0;i<6;i++) smp[i] = stc_sample(b->words[i], true); }
    else if(b->resolution==RES_16BIT) { for(int i=0;i<6;i++) smp[i] = (i16)b->words[i]; }
    else { for(int i=0;i<6;i++) smp[i] = (i16)(u16)(b->words[i]<<2); }
}
SDV_HD void blk_export(const Block *b, bool unsafe, sdv_block_rec *r)
{
    sdv_block_rec t;
    for(int i=0;i<8;i++) t.words[i] = b->words[i];
    t.line_crc = b->line_crc; t.word_valid = b->word_valid;
    t.audio_state = b->audio_state; t.resolution = b->resolution;
    u8 f = 0;
    if(blk_block_valid(b)) f |= SDV_BF_VALID;
    if(b->audio_state==SDV_AUD_BROKEN) f |= SDV_BF_BROKEN;
    if(b->audio_state==SDV_AUD_FIX_P) f |= SDV_BF_FIX_P;
    if(b->audio_state==SDV_AUD_FIX_Q) f |= SDV_BF_FIX_Q;
    if(blk_silent(b)) f |= SDV_BF_SILENT;
    if(unsafe) f |= SDV_BF_UNSAFE;
    t.flags = f;
    for(int i=0;i<11;i++) t.reserved[i] = 0;
    *r = t;
}

}   // namespace sdv
