// tests/hostemu/chain_state_cont.cpp -- TEST INFRASTRUCTURE ONLY.
//
// The line-decode chains of every format on the host build of the device code, with the chain context owned by the caller
// (PCM-1 / PCM-16x0: pcm_chain_cont.cpp; STC-007 / M2: the chain of hostemu.cpp's emu_v2d_chain), plus the pack / unpack of
// the chain-state blob (chain_state.cuh) that sdv_bin_chain_state_save / _load run on the device.  So a tape can be decoded in
// pieces with pack -> unpack into a fresh context between them, the way a decode is handed from one handle to another.
// Built by tests/test_chain_state.py into tests/hostemu/_build/; never linked into, or loaded by, the product library.
#include "pcm_chain_cont.cpp"
#include "../../sdvpcmdecoder_b200/csrc/chain_state.cuh"

static Work g_stc_w;

// STC-007 / M2 (line_dup: bit 0 duplicate-line check, bit 1 M2 samples).  cont = 0: the call opens the file; 1: it goes on from *ctx.
extern "C" int emu_stc_v2d_chain_cont(int mode, int line_dup, const u8 *luma, int n_frames, int H, int W, sdv_line_rec *recs, sdv_line_aux *aux,
                                      ChainCtx *ctx, int cont)
{
    ChainCtx &x = *ctx;
    Cta c = { 0, 1 };
    Geom g = make_geom(W);
    if(!cont) chain_reset(&x, mode, line_dup);
    int hf = H/2;
    for(int f=0;f<n_frames;f++)
    {
        chain_frame_start(&x, (f==0)&&!cont);
        for(int fld=0;fld<2;fld++)
        {
            for(int k=0;k<hf;k++)
            {
                BinState b = x.bin;
                process_line_cta(c, &g_stc_w, &b, luma+((size_t)f*H+2*k+fld)*W, g);
                chain_line(&x, &g_stc_w.o);
                size_t ridx = (size_t)f*H+(size_t)fld*hf+k;
                export_line(&g_stc_w.o, recs+ridx, aux ? aux+ridx : 0);
            }
            chain_field_end(&x);
        }
        Coord mv, mi;
        { int scr = 0; median_cta(c, x.frame_valid, x.n_fv, &mv, &scr); }
        { int scr = 0; median_cta(c, x.frame_invalid, x.n_fi, &mi, &scr); }
        chain_frame_end(&x, mv, mi);
    }
    return 0;
}

// kind: CS_KIND_STC / CS_KIND_P1 / CS_KIND_X0
extern "C" int emu_chain_ctx_size(int kind)
{
    return (kind==CS_KIND_STC) ? (int)sizeof(ChainCtx) : ((kind==CS_KIND_P1) ? (int)sizeof(P1ChainCtx) : (int)sizeof(X0ChainCtx));
}
extern "C" int emu_chain_blob_bytes(void) { return CS_BYTES; }
// The chain-state part of a blob (what chain_state_pack_kernel writes behind the header); the header is left zero.
extern "C" int emu_chain_pack(int kind, const void *ctx, u8 *blob)
{
    memset(blob, 0, CS_BYTES);
    if(kind==CS_KIND_STC) cs_pack_stc((const ChainCtx *)ctx, blob);
    else if(kind==CS_KIND_P1) cs_pack_p1((const P1ChainCtx *)ctx, blob);
    else cs_pack_x0((const X0ChainCtx *)ctx, blob);
    return 0;
}
extern "C" int emu_chain_unpack(int kind, const u8 *blob, void *ctx)
{
    if(kind==CS_KIND_STC) cs_unpack_stc(blob, (ChainCtx *)ctx);
    else if(kind==CS_KIND_P1) cs_unpack_p1(blob, (P1ChainCtx *)ctx);
    else cs_unpack_x0(blob, (X0ChainCtx *)ctx);
    return 0;
}
