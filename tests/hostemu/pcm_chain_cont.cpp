// tests/hostemu/pcm_chain_cont.cpp -- TEST INFRASTRUCTURE ONLY.
//
// The PCM-1 / PCM-16x0 line decode + chain of hostemu.cpp (emu_p1_v2d_chain / emu_x0_v2d_chain: prescan, frame presets, every
// (sub-)line through *_process_line_cta() + the chain rules, one-thread "blocks"), with the chain context owned by the caller, so
// that a tape can be run batch by batch the way sdv_bin_decode_frames continues a file (sdv_bin_config.reserved[3]):
//   cont = 0: the call opens the file (chain reset, frame 0 carries the NEW_FILE line);
//   cont = 1: it goes on from the chain state in *ctx.
// *ctx holds the chain state at the end of the call either way (what the chain kernels leave in the handle's context).
// Built by tests/test_pcm_batches.py into tests/hostemu/_build/; never linked into, or loaded by, the product library.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../../sdvpcmdecoder_b200/csrc/pcm1_chain.cuh"
#include "../../sdvpcmdecoder_b200/csrc/pcm16x0_chain.cuh"

using namespace sdv;

static P1Work g_p1w;
static X0Work g_x0w;

extern "C" int emu_pcm_ctx_sizes(int *out) { out[0] = (int)sizeof(P1ChainCtx); out[1] = (int)sizeof(X0ChainCtx); return 0; }

extern "C" int emu_p1_v2d_chain_cont(int mode, int line_dup, const u8 *luma, int n_frames, int H, int W, sdv_line_rec *recs, sdv_line_aux *aux,
                                     P1Preset *presets /*[n_frames], may be NULL*/, P1ChainCtx *ctx, int cont)
{
    P1ChainCtx &x = *ctx;
    Cta c = { 0, 1 };
    Geom g = make_geom(W);
    if(!cont) p1_chain_reset(&x, mode, line_dup);
    int hf = H/2;
    for(int f=0;f<n_frames;f++)
    {
        const bool first = (f==0)&&!cont;
        const bool ran = p1_prescan_runs(H, first, mode);
        P1Preset ps; ps.valid = 0; ps.ref = 0; ps.coords = coord_none(); ps.pad[0] = ps.pad[1] = 0;
        if(ran)
        {
            P1Preset r[P1_COORD_CHECK_LINES];
            for(int idx=0;idx<P1_COORD_CHECK_LINES;idx++)
            {
                r[idx] = ps;
                int row = p1_prescan_row(H, first, idx);
                if(row<0) continue;
                BinState b = x.bin; bin_reset_good(&b);
                p1_process_line_cta(c, &g_p1w, &b, true, luma+((size_t)f*H+row)*W, g);
                if(p1_crc_ok(&g_p1w.o)) { r[idx].valid = 1; r[idx].coords = g_p1w.o.coords; r[idx].ref = g_p1w.o.ref; }
            }
            ps = p1_prescan_reduce(r);
        }
        if(presets) presets[f] = ps;
        p1_chain_frame_start(&x, ran, ps);
        for(int fld=0;fld<2;fld++)
        {
            for(int k=0;k<hf;k++)
            {
                BinState b = x.bin;
                p1_process_line_cta(c, &g_p1w, &b, p1_chain_coord_search(&x), luma+((size_t)f*H+2*k+fld)*W, g);
                p1_chain_line(&x, &g_p1w.o);
                size_t ridx = (size_t)f*H+(size_t)fld*hf+k;
                p1_export_line(&g_p1w.o, recs+ridx, aux ? aux+ridx : 0);
            }
            p1_chain_field_end(&x);
        }
        p1_chain_frame_end(&x, median_small(x.frame_valid, x.n_fv), median_small(x.frame_invalid, x.n_fi));
    }
    return 0;
}

extern "C" int emu_x0_v2d_chain_cont(int mode, int line_dup, const u8 *luma, int n_frames, int H, int W, sdv_line_rec *recs, sdv_line_aux *aux,
                                     P1Preset *presets /*[n_frames], may be NULL*/, X0ChainCtx *ctx, int cont)
{
    X0ChainCtx &x = *ctx;
    Cta c = { 0, 1 };
    Geom g = make_geom(W);
    if(!cont) x0_chain_reset(&x, mode, line_dup);
    int hf = H/2;
    std::vector<u8> scanned(H);
    for(int f=0;f<n_frames;f++)
    {
        const bool first = (f==0)&&!cont;
        const bool ran = p1_prescan_runs(H, first, mode);
        P1Preset ps; ps.valid = 0; ps.ref = 0; ps.coords = coord_none(); ps.pad[0] = ps.pad[1] = 0;
        std::fill(scanned.begin(), scanned.end(), 0);
        if(ran)
        {
            P1Preset r[P1_COORD_CHECK_LINES];
            for(int idx=0;idx<P1_COORD_CHECK_LINES;idx++)
            {
                r[idx] = ps;
                int row = p1_prescan_row(H, first, idx);
                if(row<0) continue;
                BinState b = x.bin; bin_reset_good(&b);
                g_x0w.scan_done = 0;
                x0_process_line_cta(c, &g_x0w, &b, X0L_RIGHT, true, luma+((size_t)f*H+row)*W, g);
                scanned[row] = g_x0w.scan_done;
                if(x0_crc_ok(&g_x0w.o)) { r[idx].valid = 1; r[idx].coords = g_x0w.o.coords; r[idx].ref = g_x0w.o.ref; }
            }
            ps = p1_prescan_reduce(r);
        }
        if(presets) presets[f] = ps;
        x0_chain_frame_start(&x, ran, ps);
        for(int fld=0;fld<2;fld++)
        {
            for(int k=0;k<hf;k++)
            {
                const int row = 2*k+fld;
                g_x0w.scan_done = scanned[row];
                x0_chain_line_start(&x);
                for(int part=0;part<3;part++)
                {
                    BinState b = x.bin;
                    x0_process_line_cta(c, &g_x0w, &b, part, x0_chain_coord_search(&x), luma+((size_t)f*H+row)*W, g);
                    x0_chain_subline(&x, &g_x0w.o, g_x0w.scan_done!=0);
                    size_t ridx = ((size_t)f*H+(size_t)fld*hf+k)*3+part;
                    x0_export_line(&g_x0w.o, recs+ridx, aux ? aux+ridx : 0);
                }
            }
            x0_chain_field_end(&x);
        }
        x0_chain_frame_end(&x, median_small(x.frame_valid, x.n_fv), median_small(x.frame_invalid, x.n_fi));
    }
    return 0;
}
