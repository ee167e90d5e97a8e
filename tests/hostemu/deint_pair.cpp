// tests/hostemu/deint_pair.cpp -- TEST INFRASTRUCTURE ONLY.
//
// The two-blocks-at-once deinterleave of the standard setting (stc007_deint.cuh: deint_pair_std14, pair_samples, pair_flags,
// pair_broken_ns, pair_unpack) built as host code beside the one-block path it stands in for (deint_block_std14 +
// blk_output + the BROKEN candidate rule of stc007_deint_kernel), so that tests/test_stc007_deint_pair.py can compare them
// on any words and trusted-line masks.  Built into tests/hostemu/_build/ on first use; never part of the product library.
#include <cstring>
#include "../../sdvpcmdecoder_b200/csrc/stc007_deint.cuh"

using namespace sdv;

// One record per block: words[8], line_crc, word_valid, resolution, audio_state, samples[6], flags[6], broken_ns.
struct EmuBlock { u16 words[8]; u8 line_crc, word_valid, resolution, audio_state; i16 samples[6]; u8 flags[6]; u8 broken_ns; u8 pad; };

static void put(const Block *b, EmuBlock *o)
{
    memset(o, 0, sizeof(*o));
    for(int k=0;k<8;k++) o->words[k] = b->words[k];
    o->line_crc = b->line_crc; o->word_valid = b->word_valid; o->resolution = b->resolution; o->audio_state = b->audio_state;
}

// words [n][2][8] (block s, block s+1), ok [n][2]; out [n][2].  The one-block path.
extern "C" void emu_pair_scalar(int n, const u16 *words, const u8 *ok, EmuBlock *out)
{
    for(int i=0;i<2*n;i++)
    {
        BlockIn in; in.ok = ok[i];
        for(int k=0;k<8;k++) { in.w[k] = words[8*i+k]; in.sw[k] = 0; }
        Block b;
        deint_block_std14(&b, &in);
        b.m2 = 0;
        put(&b, out+i);
        blk_output(&b, out[i].samples, out[i].flags);
        out[i].broken_ns = (b.audio_state==SDV_AUD_BROKEN)&&!blk_silent(&b);
    }
}

// The pair path on the same inputs; covered[i] = 0 where it hands the pair back (out[2i], out[2i+1] are then left zero).
extern "C" void emu_pair_packed(int n, const u16 *words, const u8 *ok, EmuBlock *out, u8 *covered)
{
    for(int i=0;i<n;i++)
    {
        u32 w[8], okf[4] = { 0, 0, 0, 0 };
        for(int k=0;k<8;k++) w[k] = (u32)words[16*i+k]|((u32)words[16*i+8+k]<<16);
        for(int k=0;k<8;k++)
            for(int h=0;h<2;h++) okf[k>>1] |= (u32)((ok[2*i+h]>>k)&1u)<<(16*(k&1)+h);
        okf[1] |= 0xFFFCFFFCu;          // bits outside the fields are ignored
        memset(out+2*i, 0, 2*sizeof(EmuBlock));
        BlockPair bp;
        covered[i] = deint_pair_std14(w, okf, &bp) ? 1 : 0;
        if(!covered[i]) continue;
        Block a, b;
        pair_unpack(&bp, &a, &b);
        put(&a, out+2*i); put(&b, out+2*i+1);
        u32 d[6], f[3];
        pair_samples(&bp, d);
        pair_flags(&bp, f);
        memcpy(out[2*i].samples, d, 12); memcpy(out[2*i+1].samples, d+3, 12);
        u8 fb[12]; memcpy(fb, f, 12);
        memcpy(out[2*i].flags, fb, 6); memcpy(out[2*i+1].flags, fb+6, 6);
        const u32 bns = pair_broken_ns(&bp);
        out[2*i].broken_ns = bns&1u; out[2*i+1].broken_ns = (bns>>1)&1u;
    }
}
